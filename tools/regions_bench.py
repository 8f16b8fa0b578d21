"""BWA-MEM seed extension at scale: python tools/regions_bench.py [--n 1.5e9] [--reads 1000000] [--json out.json]

The workload of tools/chain_bench.py: both strands of a C3-generator text (synth_gpu.genome_like, 1.5 Gbp in 12 records,
and their reverse complements: T = 3.0 G symbols) in HBM, 1 M seeded 150-bp reads, half of them from the reverse copies
and 25 % with 1-3 substitutions, the suffix array sampled at rate 32, bwa's default seed, chain and extension options.
It times the first debwt_index_regions after sampling (it derives the pac), then debwt_index_chains (size query + fill)
against debwt_index_regions (a one-pass fill into a buffer large enough, and a size query + fill), with a host clock
around the synchronous C call, calls alternating, median of --reps.  The first --check reads are checked against
tests/ext_ref.py over the chains() of the same reads, which also counts the DP cells; the tool exits non-zero if anything
differs.  Prints one JSON object (and writes it with --json), with the GPU's name and power limit read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from debwt_b200 import api, synth_gpu  # noqa: E402
from debwt_b200.binding import c_p, c_u64, check, lib  # noqa: E402
from locate_bench import gpu_info, make_reads, timed  # noqa: E402
from tests import chain_ref as cr  # noqa: E402
from tests import ext_ref as er  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=1.5e9, help="bases of one strand")
    ap.add_argument("--records", type=int, default=12, help="records of one strand")
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--mutated", type=float, default=0.25, help="share of reads with 1-3 substitutions")
    ap.add_argument("--rate", type=int, default=32)
    ap.add_argument("--check", type=int, default=2000, help="reads checked against tests/ext_ref.py")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--json", default="")
    ap.add_argument("--profile", action="store_true", help="after the timed calls, one chains fill and one regions fill under "
                    "torch.profiler: device time per kernel (the timed numbers are taken before, without the profiler)")
    a = ap.parse_args()
    import torch

    info = gpu_info(a.device)
    torch.cuda.set_device(a.device)
    F = int(a.n)
    seq = synth_gpu.genome_like(F, 5, device=a.device)
    per = -(-F // a.records)
    recs = [seq[i:i + per] for i in range(0, F, per)]
    text_d, seps = synth_gpu.join_records_device(recs + [synth_gpu.reverse_complement(r) for r in recs])
    del seq, recs
    n, R = int(text_d.numel()), seps.size // 2
    b = api.BwtBuilder(device=a.device)
    b.set_text_device(text_d.data_ptr(), n, seps)
    b.build()
    text = text_d.cpu().numpy()
    del text_d
    torch.cuda.empty_cache()
    sample_ms = b.sample_sa(a.rate)

    m, L = a.reads, a.read_len
    half = int(seps[R - 1]) + 1
    fr, _, fm = make_reads(text[:half], seps[:R], m - m // 2, L, a.mutated, seed=7)
    rr, _, rm = make_reads(text[half:], seps[R:] - np.uint64(half), m // 2, L, a.mutated, seed=8)
    reads = np.empty((m, L), dtype=np.uint8)
    reads[0::2], reads[1::2] = fr, rr
    mutated = int(fm.sum() + rm.sum())
    blob = np.ascontiguousarray(np.concatenate([reads.reshape(-1), np.zeros(1, np.uint8)]))
    offs = np.arange(m + 1, dtype=np.uint64) * np.uint64(L)
    sopts = api.SeedOpts(19, 10, 20, 500, 1.5)
    copts = api.ChainOpts(100, 10000, 0, 1 << 30, 0.5, 0.5)
    eopts = api.ExtOpts(1, 4, 6, 1, 6, 1, 5, 5, 100)
    P = lambda x: x.ctypes.data_as(c_p)  # noqa: E731
    lb = lib()
    co, ns = np.zeros(m + 1, dtype=np.uint64), c_u64()
    ro = np.zeros(m + 1, dtype=np.uint64)
    c_head = (b._h, P(blob), P(offs), m, ctypes.addressof(sopts), ctypes.addressof(copts), P(co), ctypes.addressof(ns))
    r_head = (b._h, P(blob), P(offs), m, ctypes.addressof(sopts), ctypes.addressof(copts), ctypes.addressof(eopts), P(ro))

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    check(lb.debwt_index_regions(*r_head, c_p(0), 0))                  # the first call after sampling derives the pac
    first_ms = (time.perf_counter() - t0) * 1e3
    check(lb.debwt_index_chains(*c_head, c_p(0), 0, c_p(0), 0))
    chains = np.zeros(int(co[-1]), dtype=api.CHAIN_DTYPE)
    cseeds = np.zeros(int(ns.value), dtype=api.CHAIN_SEED_DTYPE)
    regions = np.zeros(int(ro[-1]), dtype=api.REGION_DTYPE)
    calls = {
        "chains_query": lambda: check(lb.debwt_index_chains(*c_head, c_p(0), 0, c_p(0), 0)),
        "chains_fill": lambda: check(lb.debwt_index_chains(*c_head, P(chains), chains.size, P(cseeds), cseeds.size)),
        "regions_fill": lambda: check(lb.debwt_index_regions(*r_head, P(regions), regions.size)),
        "regions_query": lambda: check(lb.debwt_index_regions(*r_head, c_p(0), 0)),
    }
    for f in calls.values():                                           # warm-up
        f()
    ms = {k: [] for k in calls}
    for _ in range(a.reps):                                            # alternate, so that drift hits all alike
        for k, f in calls.items():
            ms[k] += timed(f, 1)[1]
    med = {k: float(np.median(v)) for k, v in ms.items()}

    kernel_ms = "not measured"
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        kernel_ms = {}
        for name in ("chains_fill", "regions_fill"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                calls[name]()
                torch.cuda.synchronize()
            kernel_ms[name] = {e.key: {"ms": e.device_time_total / 1e3, "calls": e.count} for e in prof.key_averages()
                               if e.device_time_total > 0}
    k = min(a.check, m)
    rd = [reads[i].tobytes() for i in range(k)]
    c0 = int(co[k])
    s_end = int(chains[c0 - 1]["seed_begin"] + chains[c0 - 1]["n_seeds"]) if c0 else 0
    ch, cs = cr.as_tuples(chains[:c0], cseeds[:s_end])
    cells0 = er.cells()
    want = er.reference(co[:k + 1].tolist(), ch, cs, rd, text, seps)
    cells = er.cells() - cells0
    ok = ro[:k + 1].tolist() == want[0] and er.as_tuples(regions[:int(ro[k])]) == want[1]
    del text
    b.close()
    res = {"gpu": info,
           "workload": {"n_symbols": n, "records": 2 * R, "bases_per_strand": F, "generator": "synth_gpu.genome_like(seed 5) + reverse complements"},
           "sa_sample": {"rate": a.rate, "ms": sample_ms},
           "reads": {"n": m, "length": L, "reverse_strand": m // 2, "mutated": mutated, "seeds": [7, 8]},
           "options": {"min_seed_len": 19, "split_factor": 1.5, "split_width": 10, "max_mem_intv": 20, "max_occ": 500, "w": 100,
                       "max_chain_gap": 10000, "min_chain_weight": 0, "mask_level": 0.5, "drop_ratio": 0.5, "max_chain_extend": 1 << 30,
                       "a": 1, "b": 4, "o_del": 6, "e_del": 1, "o_ins": 6, "e_ins": 1, "pen_clip5": 5, "pen_clip3": 5, "zdrop": 100},
           "timing": "host clock around the synchronous C call, calls alternating, median of reps",
           "first_regions_call_ms": first_ms,
           "pac_build_ms_estimate": first_ms - med["regions_query"],
           "pac_bytes": (n - 2 * R) // 2 // 4,
           "ms": med, "ms_all": ms,
           "chains_ms": med["chains_query"] + med["chains_fill"],
           "regions_one_pass_ms": med["regions_fill"],
           "regions_query_plus_fill_ms": med["regions_query"] + med["regions_fill"],
           "regions_fill_minus_chains_fill_ms": med["regions_fill"] - med["chains_fill"],
           "chains": int(chains.size), "chain_seeds": int(cseeds.size), "regions": int(regions.size),
           "regions_per_read": regions.size / m, "reads_with_regions": int((np.diff(ro.astype(np.int64)) > 0).sum()),
           "region_bytes": int(regions.nbytes),
           "kernel_ms": kernel_ms,
           "dp_cells_checked_reads": {"reads": k, "cells": cells, "per_read": cells / max(k, 1),
                                      "method": "tests/ext_dp.c: band cells of every extension row and the full matrix of seed SW"},
           "check": {"reads": k, "method": "regions() = tests/ext_ref.py over chains() of the same reads", "ok": bool(ok)}}
    print(json.dumps(res))
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
