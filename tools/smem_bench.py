"""SMEM seeding at scale: python tools/smem_bench.py [--n 1.5e9] [--reads 1000000] [--json out.json]

Builds both strands of a C3-generator text (synth_gpu.genome_like, 1.5 Gbp in 12 records, and their reverse complements:
T = 3.0 G symbols; both strands of the full 3.1 Gbp would exceed what one device builds) in HBM, then runs
debwt_index_smem on 1 M seeded 150-bp reads, half of them from the reverse copies and 25 % with 1-3 substitutions, at
min_len = 19.  The size query and the fill are timed separately with a host clock around the synchronous C call (read
upload, count pass, offset scan, and for the fill the write pass and the download; a warm-up call each, median of 3).
The SMEMs of the first 2000 reads are checked against the definition derived through count alone
(tests/smem_ref.smems_by_count); the tool exits non-zero if they differ.  Prints one JSON object (and writes it with
--json), with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from debwt_b200 import api, synth_gpu  # noqa: E402
from debwt_b200.binding import c_p, check, lib  # noqa: E402
from locate_bench import gpu_info, make_reads, timed  # noqa: E402
from tests.smem_ref import smems_by_count  # noqa: E402

SCRATCH_BYTES = 1 << 30          # kSmemScratchBytes of csrc/index.cu


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=1.5e9, help="bases of one strand")
    ap.add_argument("--records", type=int, default=12, help="records of one strand")
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--mutated", type=float, default=0.25, help="share of reads with 1-3 substitutions")
    ap.add_argument("--min-len", type=int, default=19)
    ap.add_argument("--check", type=int, default=2000, help="reads checked against the count-derived definition")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--json", default="")
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
    build_ms = b.stats()["ms_total"]
    t0 = time.perf_counter()
    check(lib().debwt_index_build(b._h))
    index_ms = (time.perf_counter() - t0) * 1e3
    text = text_d.cpu().numpy()
    del text_d
    torch.cuda.empty_cache()

    # half of the reads from the forward records, half from their reverse complements
    m, L = a.reads, a.read_len
    half = int(seps[R - 1]) + 1
    fr, _, fm = make_reads(text[:half], seps[:R], m - m // 2, L, a.mutated, seed=7)
    rr, _, rm = make_reads(text[half:], seps[R:] - np.uint64(half), m // 2, L, a.mutated, seed=8)
    reads = np.empty((m, L), dtype=np.uint8)
    reads[0::2], reads[1::2] = fr, rr
    mutated = int(fm.sum() + rm.sum())
    blob = np.ascontiguousarray(np.concatenate([reads.reshape(-1), np.zeros(1, np.uint8)]))
    offs = np.arange(m + 1, dtype=np.uint64) * np.uint64(L)
    so = np.zeros(m + 1, dtype=np.uint64)
    P = lambda x: x.ctypes.data_as(c_p)  # noqa: E731
    lb = lib()

    def query():
        check(lb.debwt_index_smem(b._h, P(blob), P(offs), m, a.min_len, P(so), c_p(0), 0))

    query()                                                            # warm-up
    ms_q, all_q = timed(query, a.reps)
    total = int(so[-1])
    sm = np.zeros(total, dtype=api.SMEM_DTYPE)

    def fill():
        check(lb.debwt_index_smem(b._h, P(blob), P(offs), m, a.min_len, P(so), P(sm), total))

    fill()                                                             # warm-up
    ms_f, all_f = timed(fill, a.reps)
    props = torch.cuda.get_device_properties(a.device)
    slots = min(props.multi_processor_count * props.max_threads_per_multi_processor, SCRATCH_BYTES // (64 * (L + 1)), m)
    lens = (sm["qend"].astype(np.int64) - sm["qbeg"].astype(np.int64)) if total else np.zeros(1)

    k = min(a.check, m)
    rd = [reads[i].tobytes() for i in range(k)]
    want = smems_by_count(b.count, rd, a.min_len)
    got = [[(int(x["qbeg"]), int(x["qend"]), int(x["count"])) for x in sm[int(so[i]):int(so[i + 1])]] for i in range(k)]
    bad = [i for i in range(k) if got[i] != want[i]]
    b.close()

    res = {"gpu": info,
           "workload": {"n_symbols": n, "records": 2 * R, "bases_per_strand": F, "generator": "synth_gpu.genome_like(seed 5) + reverse complements"},
           "build_ms": build_ms, "index_tables_ms": index_ms,
           "reads": {"n": m, "length": L, "reverse_strand": m // 2, "mutated": mutated, "seeds": [7, 8], "min_len": a.min_len},
           "size_query_ms": ms_q, "size_query_ms_all": all_q, "fill_ms": ms_f, "fill_ms_all": all_f,
           "smem_ms": ms_q + ms_f, "reads_per_s": m / ((ms_q + ms_f) / 1e3), "reads_per_s_fill_only": m / (ms_f / 1e3),
           "smems": total, "smems_per_read": total / m, "mean_smem_len": float(lens.mean()),
           "scratch_slots": slots, "scratch_bytes": slots * 64 * (L + 1), "kernel_ms": "not measured",
           "check": {"reads": k, "method": "count-derived start(e) for every end e", "reads_differing": len(bad),
                     "first_differing": bad[:5], "ok": not bad}}
    print(json.dumps(res))
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    if bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
