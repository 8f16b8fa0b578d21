"""Extract and whole-text inversion at scale: python tools/extract_bench.py [--n 3.1e9] [--intervals 1000000] [--json out.json]

Builds the default bench workload (C3: 3.1 Gbp, 24 records, synth_gpu.config3) in HBM and runs the list-ranking verifier
once (its device time is the yardstick for a full inversion).  Then for each SA sampling rate (16, 32, 64) it times, with a
host clock around the synchronous C call:
  * the first debwt_index_extract after debwt_index_sample_sa (it derives the inverse samples) on one 150-bp interval,
    and the same call again;
  * 1 M intervals of 150 bp at seeded positions (interval upload, one thread per rate-aligned block, download of the
    150 MB of symbols into pageable memory; a warm-up call first, median of 3);
  * the whole text [0, N), compared byte for byte with T (median of 3).
Every symbol of the first 100 k intervals is checked against T.  Prints one JSON object (and writes it with --json), with
the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from debwt_b200 import api, synth_gpu  # noqa: E402
from debwt_b200.binding import c_p, check, lib  # noqa: E402
from locate_bench import gpu_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=3.1e9)
    ap.add_argument("--records", type=int, default=24)
    ap.add_argument("--intervals", type=int, default=1_000_000)
    ap.add_argument("--length", type=int, default=150)
    ap.add_argument("--rates", default="16,32,64")
    ap.add_argument("--check", type=int, default=100_000, help="intervals whose every symbol is checked against T")
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
    bad, verify_ms = b.verify(device_ptr=text_d.data_ptr(), n_symbols=n)
    assert bad == 0, f"verify: {bad} bad rows"
    text = text_d.cpu().numpy()
    del text_d
    torch.cuda.empty_cache()

    m, L = a.intervals, a.length
    rng = np.random.default_rng(7)
    starts = rng.integers(0, n - L + 1, m).astype(np.uint64)
    ends = starts + np.uint64(L)
    out = np.empty(m * L, dtype=np.uint8)
    whole = np.empty(n, dtype=np.uint8)
    zero, top = np.zeros(1, dtype=np.uint64), np.full(1, n, dtype=np.uint64)
    one_s, one_e = np.array([1000], dtype=np.uint64), np.array([1000 + L], dtype=np.uint64)
    one = np.empty(L, dtype=np.uint8)
    P = lambda x: x.ctypes.data_as(c_p)  # noqa: E731
    lb = lib()

    def short():
        check(lb.debwt_index_extract(b._h, P(one_s), P(one_e), 1, P(one), L))

    def intervals():
        check(lb.debwt_index_extract(b._h, P(starts), P(ends), m, P(out), out.size))

    def invert():
        check(lb.debwt_index_extract(b._h, P(zero), P(top), 1, P(whole), n))

    res = {"gpu": info, "workload": {"n_symbols": n, "records": a.records, "generator": "synth_gpu.config3"},
           "build_ms": build_ms, "verify_ms": verify_ms,
           "intervals": {"n": m, "length": L, "seed": 7}, "rates": []}
    ok = True
    for rate in [int(x) for x in a.rates.split(",")]:
        ms_sample = b.sample_sa(rate)
        t0 = time.perf_counter()
        short()                                                        # builds the inverse samples
        first_ms = (time.perf_counter() - t0) * 1e3
        second_ms, _ = timed(short, 1)
        ok_short = bool((one == text[1000:1000 + L]).all())
        intervals()                                                    # warm-up
        ms_iv, all_iv = timed(intervals, a.reps)
        k = min(a.check, m)
        s = starts[:k].astype(np.int64)
        ok_iv = bool((out[:k * L].reshape(k, L) == text[s[:, None] + np.arange(L)[None, :]]).all())
        ms_inv, all_inv = timed(invert, a.reps)
        ok_inv = bool((whole == text).all())
        ok = ok and ok_short and ok_iv and ok_inv
        res["rates"].append({"rate": rate, "sample_sa_ms": ms_sample, "isa_hbm_bytes": 4 * ((n + rate - 1) // rate),
                             "first_call_ms": first_ms, "second_call_ms": second_ms,
                             "intervals_ms": ms_iv, "intervals_ms_all": all_iv, "intervals_per_s": m / (ms_iv / 1e3),
                             "intervals_gbp_per_s": m * L / (ms_iv / 1e3) / 1e9,
                             "invert_ms": ms_inv, "invert_ms_all": all_inv, "invert_gbp_per_s": n / (ms_inv / 1e3) / 1e9,
                             "checked_intervals": k, "short_ok": ok_short, "intervals_ok": ok_iv, "invert_equals_T": ok_inv})
        print(json.dumps(res["rates"][-1]), flush=True)
    res["ok"] = ok
    b.close()
    print(json.dumps(res))
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
