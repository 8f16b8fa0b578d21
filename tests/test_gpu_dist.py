"""GPU tests of the sharded path: the CUDA stage kernels behind debwt_b200.dist (include/debwt_b200_dev.h).
World size 1 in-process, and world size 2 / 3 as separate processes sharing cuda:0 over a gloo group
(collectives staged through host memory), against the oracle and the reference's golden vectors."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from debwt_b200 import api, dist as D, synth
from oracle import coracle, stages as st
from tests.util import as_bytes_records, golden, seeded_records, sha

pytestmark = pytest.mark.gpu
G = golden()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _check(recs, w, s, d):
    sym, _ = st.text_from_records(as_bytes_records(recs))
    ow, os_, od = coracle.bwt(sym)
    return bool((w == ow).all() and (s == os_).all() and (d == od).all())


def _case(name):
    if name in G["small"]:
        return G["small"][name]["records"]
    if name == "big_segments":
        rng = np.random.default_rng(5)
        master = synth.random_bases(77, 2000)
        recs = []
        for _ in range(3):
            parts = []
            for _ in range(300):
                el = master.copy()
                idx = rng.integers(0, el.size, size=20)
                el[idx] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=20)]
                parts.append(el)
            recs.append(np.concatenate(parts))
        return recs
    return seeded_records(name)


CASES = ["survey_golden", "pathological", "haplotypes_6x1500", "planted_repeats", "c4_like_5x100k", "c3_like_600k_3rec",
         "c2_like_1m", "big_segments"]


@pytest.mark.parametrize("name", CASES)
def test_sharded_world1_cuda(name):
    recs = _case(name)
    text, seps = api.join_records(recs)
    stats = {}
    w, s, d = D.build_sharded(text, seps, D.Comm(), D.CudaOps(0), stats)
    assert _check(recs, w, s, d)
    assert stats["launches"] > 20


def _worker(rank, world, port, names, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.cuda.set_device(0)
        comm = D.Comm(staged=True)
        for name in names:
            recs = _case(name)
            text, seps = api.join_records(recs)
            stats = {}
            w, s, d = D.build_sharded(text, seps, comm, D.CudaOps(0), stats)
            if rank == 0:
                out.put((name, _check(recs, w, s, d), stats["keys_local"]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_multi_rank_one_gpu(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, CASES, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0
    got = {}
    while not q.empty():
        name, ok, kl = q.get()
        got[name] = (ok, kl)
    assert set(got) == set(CASES)
    for name, (ok, kl) in got.items():
        assert ok, name
        assert len(kl) == world and min(kl) >= 0


# ---- the production exchange path: one process per GPU, NCCL + CUDA-IPC peer stores (needs >= 2 real GPUs) -----------
def _worker_nccl(rank, world, port, names, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        comm = D.Comm()
        assert not comm.staged and comm.coll_device.type == "cuda"
        ops = D.CudaOps(rank)
        for name in names:
            recs = _case(name)
            text, seps = api.join_records(recs)
            stats = {}
            w, s, d = D.build_sharded(text, seps, comm, ops, stats)
            if rank == 0:
                out.put((name, _check(recs, w, s, d), stats["keys_local"], D.PeerExchange._cache != {}))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_nccl_p2p_real_gpus(world):
    """partition_scatter_p2p*_kernel (peer stores over NVLink) + NCCL collectives on K9/K10-heavy inputs, against the oracle"""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    names = ["c4_like_5x100k", "big_segments", "c3_like_600k_3rec", "c2_like_1m", "pathological", "survey_golden"]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_nccl, args=(r, world, port, names, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=900)
        assert p.exitcode == 0
    got = {}
    while not q.empty():
        name, ok, kl, p2p = q.get()
        got[name] = (ok, kl, p2p)
    assert set(got) == set(names)
    for name, (ok, kl, p2p) in got.items():
        assert ok, name
        assert p2p, "the peer-store exchange did not run"
        assert len(kl) == world
