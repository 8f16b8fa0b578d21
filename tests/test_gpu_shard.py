"""The sharded build behind the C ABI (csrc/shard.cu: debwt_shard_*, debwt_build_multi) against the oracle and the
reference's golden vectors: one rank, several ranks as PROCESSES sharing cuda:0 (CUDA IPC peer buffers, the torchrun
arrangement), several ranks as THREADS of one process (debwt_build_multi, what `deBWT -g 0,1,..` runs), and -- when the
box has them -- one rank per real GPU over NVLink."""
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from debwt_b200 import api
from oracle import coracle, stages as st
from tests.test_gpu_dist import CASES, _case
from tests.util import as_bytes_records

pytestmark = pytest.mark.gpu


def _check(recs, w, s, d):
    sym, _ = st.text_from_records(as_bytes_records(recs))
    ow, os_, od = coracle.bwt(sym)
    return bool((w == ow).all() and (s == os_).all() and (d == od).all())


@pytest.mark.parametrize("name", CASES)
def test_shard_world1(name):
    recs = _case(name)
    text, seps = api.join_records(recs)
    with api.Shard(0, 0, 1, f"t1_{os.getpid()}") as sh:
        sh.build_host(text, seps)
        w, s, d = sh.result()
        stats = sh.stats()
        sh.build_host(text, seps)                           # a second build on the same shard reuses its buffers
        w2, s2, d2 = sh.result()
    assert _check(recs, w, s, d)
    assert (w == w2).all() and (s == s2).all() and (d == d2).all()
    assert stats["n_keys_local"] == stats["n_keys"]


def _worker(rank, world, tag, names, devices, out):
    try:
        dev = devices[rank]
        torch.cuda.set_device(dev)
        with api.Shard(dev, rank, world, tag) as sh:
            for name in names:
                recs = _case(name)
                text, seps = api.join_records(recs)
                sh.build_host(text, seps)
                res = sh.result()
                if rank == 0:
                    out.put((name, _check(recs, *res), sh.stats()["n_keys_local"]))
    except Exception as e:  # noqa: BLE001
        out.put(("error", f"rank {rank}: {e}", 0))
        raise


def _run_processes(world, devices, names):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    tag = f"tp_{os.getpid()}_{world}_{len(set(devices))}"
    procs = [ctx.Process(target=_worker, args=(r, world, tag, names, devices, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=900)
    got = {}
    while not q.empty():
        name, ok, kl = q.get()
        got[name] = (ok, kl)
    assert "error" not in got, got.get("error")
    for p in procs:
        assert p.exitcode == 0
    assert set(got) == set(names)
    for name, (ok, _) in got.items():
        assert ok, name


@pytest.mark.parametrize("world", [2, 3])
def test_shard_processes_one_gpu(world):
    _run_processes(world, [0] * world, CASES)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_shard_processes_real_gpus(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    _run_processes(world, list(range(world)), ["c4_like_5x100k", "big_segments", "c3_like_600k_3rec", "c2_like_1m", "pathological"])


@pytest.mark.parametrize("n_threads", [1, 2, 3])
def test_build_multi_threads_one_gpu(n_threads):
    for name in ["survey_golden", "haplotypes_6x1500", "c4_like_5x100k", "big_segments"]:
        recs = _case(name)
        text, seps = api.join_records(recs)
        w, s, d, stats = api.build_multi(text, seps, [0] * n_threads)
        assert _check(recs, w, s, d), name
        assert stats["n_symbols"] == text.size


def test_build_multi_threads_real_gpus():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    for name in ["c4_like_5x100k", "big_segments", "c2_like_1m"]:
        recs = _case(name)
        text, seps = api.join_records(recs)
        w, s, d, _ = api.build_multi(text, seps, list(range(min(n, 8))))
        assert _check(recs, w, s, d), name
