"""BWA-MEM seed chaining at scale: python tools/chain_bench.py [--n 1.5e9] [--reads 1000000] [--json out.json]

The workload of tools/seed_bench.py: both strands of a C3-generator text (synth_gpu.genome_like, 1.5 Gbp in 12 records,
and their reverse complements: T = 3.0 G symbols) in HBM, 1 M seeded 150-bp reads, half of them from the reverse copies
and 25 % with 1-3 substitutions, the suffix array sampled at rate 32, bwa's default seed and chain options.  In the same
run it times debwt_index_seeds and debwt_index_chains, each as a size query and a fill, with a host clock around the
synchronous C call (a warm-up call each, then the two calls alternating, median of --reps).  chains runs the seeding
inside it, so chains minus seeds is what chaining adds end to end; the chains download no hits.  The first --check reads
are checked against tests/chain_ref.py over the seeds() of the same reads; the tool exits non-zero if anything differs.
Prints one JSON object (and writes it with --json), with the GPU's name and power limit read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from debwt_b200 import api, synth_gpu  # noqa: E402
from debwt_b200.binding import c_p, c_u64, check, lib  # noqa: E402
from locate_bench import gpu_info, make_reads, timed  # noqa: E402
from tests import chain_ref as cr  # noqa: E402
from tests import seed_ref as sr  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=1.5e9, help="bases of one strand")
    ap.add_argument("--records", type=int, default=12, help="records of one strand")
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--mutated", type=float, default=0.25, help="share of reads with 1-3 substitutions")
    ap.add_argument("--rate", type=int, default=32)
    ap.add_argument("--check", type=int, default=2000, help="reads checked against tests/chain_ref.py")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--json", default="")
    ap.add_argument("--profile", action="store_true", help="after the timed calls, one fill of each under torch.profiler: "
                    "device time per kernel (the timed numbers are taken before, without the profiler)")
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
    del text
    reads = np.empty((m, L), dtype=np.uint8)
    reads[0::2], reads[1::2] = fr, rr
    mutated = int(fm.sum() + rm.sum())
    blob = np.ascontiguousarray(np.concatenate([reads.reshape(-1), np.zeros(1, np.uint8)]))
    offs = np.arange(m + 1, dtype=np.uint64) * np.uint64(L)
    sopts = api.SeedOpts(19, 10, 20, 500, 1.5)
    copts = api.ChainOpts(100, 10000, 0, 1 << 30, 0.5, 0.5)
    P = lambda x: x.ctypes.data_as(c_p)  # noqa: E731
    lb = lib()
    so, nh = np.zeros(m + 1, dtype=np.uint64), c_u64()
    co, ns = np.zeros(m + 1, dtype=np.uint64), c_u64()
    s_head = (b._h, P(blob), P(offs), m, ctypes.addressof(sopts), P(so), ctypes.addressof(nh))
    c_head = (b._h, P(blob), P(offs), m, ctypes.addressof(sopts), ctypes.addressof(copts), P(co), ctypes.addressof(ns))

    check(lb.debwt_index_seeds(*s_head, c_p(0), 0, c_p(0), 0))
    check(lb.debwt_index_chains(*c_head, c_p(0), 0, c_p(0), 0))
    seeds = np.zeros(int(so[-1]), dtype=api.SEED_DTYPE)
    hits = np.zeros(int(nh.value), dtype=api.HIT_DTYPE)
    chains = np.zeros(int(co[-1]), dtype=api.CHAIN_DTYPE)
    cseeds = np.zeros(int(ns.value), dtype=api.CHAIN_SEED_DTYPE)
    calls = {
        "seeds_query": lambda: check(lb.debwt_index_seeds(*s_head, c_p(0), 0, c_p(0), 0)),
        "seeds_fill": lambda: check(lb.debwt_index_seeds(*s_head, P(seeds), seeds.size, P(hits), hits.size)),
        "chains_query": lambda: check(lb.debwt_index_chains(*c_head, c_p(0), 0, c_p(0), 0)),
        "chains_fill": lambda: check(lb.debwt_index_chains(*c_head, P(chains), chains.size, P(cseeds), cseeds.size)),
    }
    for f in calls.values():                                           # warm-up
        f()
    ms = {k: [] for k in calls}
    for _ in range(a.reps):                                            # alternate, so that drift hits all four alike
        for k, f in calls.items():
            ms[k] += timed(f, 1)[1]
    med = {k: float(np.median(v)) for k, v in ms.items()}

    kernel_ms = "not measured"
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        kernel_ms = {}
        for name in ("seeds_fill", "chains_fill"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                calls[name]()
                torch.cuda.synchronize()
            kernel_ms[name] = {e.key: {"ms": e.device_time_total / 1e3, "calls": e.count} for e in prof.key_averages()
                               if e.device_time_total > 0}
    k = min(a.check, m)
    rd = [reads[i].tobytes() for i in range(k)]
    h_end = int(seeds[int(so[k])]["hit_begin"]) if int(so[k]) < seeds.size else hits.size
    want = cr.reference(so[:k + 1].tolist(), *cr.tuples(seeds[:int(so[k])], hits[:h_end]), seps, [L] * k, **sr.DEFAULTS)
    c0 = int(co[k])
    got_c = chains[:c0]
    got_s = cseeds[:int(got_c[-1]["seed_begin"] + got_c[-1]["n_seeds"])] if c0 else cseeds[:0]
    ok = co[:k + 1].tolist() == want[0] and cr.as_tuples(got_c, got_s) == (want[1], want[2])
    b.close()
    kept = {str(v): int((chains["kept"] == v).sum()) for v in (1, 2, 3)}
    res = {"gpu": info,
           "workload": {"n_symbols": n, "records": 2 * R, "bases_per_strand": F, "generator": "synth_gpu.genome_like(seed 5) + reverse complements"},
           "sa_sample": {"rate": a.rate, "ms": sample_ms},
           "reads": {"n": m, "length": L, "reverse_strand": m // 2, "mutated": mutated, "seeds": [7, 8]},
           "options": {"min_seed_len": 19, "split_factor": 1.5, "split_width": 10, "max_mem_intv": 20, "max_occ": 500, "w": 100,
                       "max_chain_gap": 10000, "min_chain_weight": 0, "mask_level": 0.5, "drop_ratio": 0.5, "max_chain_extend": 1 << 30},
           "timing": "host clock around the synchronous C call, calls alternating, median of reps",
           "ms": med, "ms_all": ms,
           "seeds_ms": med["seeds_query"] + med["seeds_fill"], "chains_ms": med["chains_query"] + med["chains_fill"],
           "chains_fill_minus_seeds_fill_ms": med["chains_fill"] - med["seeds_fill"],
           "seeds": int(seeds.size), "hits": int(hits.size), "hit_bytes": int(hits.nbytes),
           "chains": int(chains.size), "chain_seeds": int(cseeds.size), "chain_bytes": int(chains.nbytes + cseeds.nbytes),
           "chains_per_read": chains.size / m, "kept": kept, "seeds_per_chain": cseeds.size / max(chains.size, 1),
           "reads_with_chains": int((np.diff(co.astype(np.int64)) > 0).sum()),
           "chains_with_frac_rep": int((chains["frac_rep"] > 0).sum()),
           "kernel_ms": kernel_ms,
           "check": {"reads": k, "method": "chains() = tests/chain_ref.py over seeds() of the same reads", "ok": bool(ok)}}
    print(json.dumps(res))
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
