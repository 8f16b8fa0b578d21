"""Sampled suffix array + locate at scale: python tools/locate_bench.py [--n 3.1e9] [--reads 1000000] [--json out.json]

Builds the default bench workload (C3: 3.1 Gbp, 24 records, synth_gpu.config3) in HBM, then for each SA sampling rate
(16, 32, 64) times debwt_index_sample_sa (CUDA events inside the library) and debwt_index_locate on seeded 100-bp reads
taken from T, a share of them with substitutions (host clock around the synchronous C call: pattern upload, search,
offset scan, SA lookups and the download of the positions; a warm-up call first), with debwt_index_count on the same reads
beside it.  Every hit of a subset of the reads is checked against T.  Prints one JSON object (and writes it with --json),
with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from debwt_b200 import api, synth_gpu  # noqa: E402
from debwt_b200.binding import c_p, check, lib  # noqa: E402


def gpu_info(device):
    out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    if out.returncode:
        raise RuntimeError("nvidia-smi query failed: " + out.stderr)
    name, power, clock = [x.strip() for x in out.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def make_reads(text, seps, m, length, mut_frac, seed):
    """m reads of `length` bases from positions inside records; a share `mut_frac` with 1-3 substitutions"""
    rng = np.random.default_rng(seed)
    n = text.size
    starts = np.empty(0, dtype=np.int64)
    while starts.size < m:
        s = rng.integers(0, n - length - 1, 2 * m)
        rec = np.searchsorted(seps, s, side="left")                  # first separator at or after s must lie beyond the read
        s = s[seps[rec].astype(np.int64) >= s + length]
        starts = np.concatenate([starts, s])[:m]
    reads = text[starts[:, None] + np.arange(length)[None, :]]
    origin = reads.copy()
    mutated = rng.random(m) < mut_frac
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    for k in range(3):
        rows = np.flatnonzero(mutated & (rng.random(m) < (1.0 if k == 0 else 0.5)))
        cols = rng.integers(0, length, rows.size)
        old = reads[rows, cols]
        new = acgt[(np.searchsorted(acgt, old) + rng.integers(1, 4, rows.size)) % 4]
        reads[rows, cols] = new
    mutated = (reads != origin).any(axis=1)                           # a later substitution may restore an earlier one
    return np.ascontiguousarray(reads), starts, mutated


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=3.1e9)
    ap.add_argument("--records", type=int, default=24)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--read-len", type=int, default=100)
    ap.add_argument("--mutated", type=float, default=0.25, help="share of reads with 1-3 substitutions")
    ap.add_argument("--rates", default="16,32,64")
    ap.add_argument("--check", type=int, default=10_000, help="reads whose every hit is checked against T")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--json", default="")
    a = ap.parse_args()
    import torch

    n = int(a.n)
    info = gpu_info(a.device)
    torch.cuda.set_device(a.device)
    text_d, seps = synth_gpu.config3(n, a.records, device=a.device)
    n = int(text_d.numel())
    b = api.BwtBuilder(device=a.device)
    b.set_text_device(text_d.data_ptr(), n, seps)
    b.build()
    build_ms = b.stats()["ms_total"]
    text = text_d.cpu().numpy()
    del text_d
    torch.cuda.empty_cache()

    L, m = a.read_len, a.reads
    reads, starts, mutated = make_reads(text, seps, m, L, a.mutated, seed=7)
    blob = np.ascontiguousarray(np.concatenate([reads.reshape(-1), np.zeros(1, np.uint8)]))
    offs = np.arange(m + 1, dtype=np.uint64) * np.uint64(L)
    hits = np.zeros(m + 1, dtype=np.uint64)
    counts = np.zeros(m, dtype=np.uint64)
    P = lambda x: x.ctypes.data_as(c_p)  # noqa: E731
    lb = lib()

    def count():
        check(lb.debwt_index_count(b._h, P(blob), P(offs), m, P(counts)))

    res = {"gpu": info, "workload": {"n_symbols": n, "records": a.records, "generator": "synth_gpu.config3"},
           "build_ms": build_ms, "reads": {"n": m, "length": L, "mutated": int(mutated.sum()), "seed": 7}, "rates": []}
    check(lb.debwt_index_build(b._h))
    count()                                                            # warm-up
    res["count"] = {"ms": timed(count, a.reps)[0]}
    res["count"]["reads_per_s"] = m / (res["count"]["ms"] / 1e3)
    positions = None
    for rate in [int(x) for x in a.rates.split(",")]:
        ms_sample = b.sample_sa(rate)
        sample_bytes = ((n + 31) // 32) * 8 + ((n + rate - 1) // rate) * 4

        def query():
            check(lb.debwt_index_locate(b._h, P(blob), P(offs), m, P(hits), c_p(0), 0))

        query()
        total = int(hits[-1])
        positions = np.empty(total, dtype=np.uint64)

        def fill():
            check(lb.debwt_index_locate(b._h, P(blob), P(offs), m, P(hits), P(positions), total))

        w = min(m, 10_000)                                             # warm-up on a slice of the reads
        wh = np.zeros(w + 1, dtype=np.uint64)
        check(lb.debwt_index_locate(b._h, P(blob), P(offs), w, P(wh), c_p(0), 0))
        wp = np.empty(max(int(wh[-1]), 1), dtype=np.uint64)
        check(lb.debwt_index_locate(b._h, P(blob), P(offs), w, P(wh), P(wp), wp.size))
        fill()
        ms_q, _ = timed(query, a.reps)
        ms_f, all_f = timed(fill, a.reps)
        res["rates"].append({"rate": rate, "sample_sa_ms": ms_sample, "sample_hbm_bytes": sample_bytes,
                             "locate_size_query_ms": ms_q, "locate_fill_ms": ms_f, "locate_fill_ms_all": all_f,
                             "locate_ms": ms_q + ms_f, "hits": total, "hits_per_s": total / ((ms_q + ms_f) / 1e3),
                             "reads_per_s": m / ((ms_q + ms_f) / 1e3)})
        print(json.dumps(res["rates"][-1]), flush=True)

    # checks on the last rate's output
    count()
    assert (np.diff(hits.astype(np.int64)) == counts.astype(np.int64)).all(), "locate hit counts differ from count"
    k = min(a.check, m)
    h = hits[:k + 1].astype(np.int64)
    pos = positions[:h[-1]].astype(np.int64)
    owner = np.repeat(np.arange(k), np.diff(h))
    ok_text = bool(pos.size == 0 or (pos.max() + L <= n and (text[pos[:, None] + np.arange(L)[None, :]] == reads[owner]).all()))
    exact = ~mutated[:k]
    found_origin = np.zeros(k, dtype=bool)
    found_origin[owner[pos == starts[owner]]] = True
    res["check"] = {"reads": k, "hits": int(h[-1]), "every_hit_matches_T": ok_text,
                    "unmutated_reads": int(exact.sum()), "unmutated_reads_found_at_origin": int((found_origin & exact).sum())}
    res["check"]["ok"] = ok_text and res["check"]["unmutated_reads_found_at_origin"] == res["check"]["unmutated_reads"]
    b.close()
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    if not res["check"]["ok"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
