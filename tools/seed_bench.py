"""BWA-MEM seed collection at scale: python tools/seed_bench.py [--n 1.5e9] [--reads 1000000] [--json out.json]

The workload of tools/smem_bench.py: both strands of a C3-generator text (synth_gpu.genome_like, 1.5 Gbp in 12 records,
and their reverse complements: T = 3.0 G symbols) in HBM, 1 M seeded 150-bp reads, half of them from the reverse copies
and 25 % with 1-3 substitutions.  The suffix array is sampled at rate 32 (CUDA events inside the library, on its own
line), then debwt_index_seeds runs with bwa's default options (-k 19 -r 1.5, split_width 10, -y 20, -c 500).  The size
query and the fill are timed separately with a host clock around the synchronous C call (read upload, count pass, the
two offset scans, and for the fill the write pass, the hit lookups and the download; a warm-up call each, median of 3).
The first 2000 reads are checked as the scale test does: round 1 equals debwt_index_smem, every seed's count equals
count() of its piece, every hit's text is its piece; the tool exits non-zero if anything differs.  Prints one JSON
object (and writes it with --json), with the GPU's name and power limit read in the same run.
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


def check_reads(b, reads, so, seeds, hits, text, min_len):
    """[indices of reads whose seeds or hits are wrong] for the reads given (the first k of the run)"""
    k = len(reads)
    sub = seeds[:int(so[k])]
    s_off, sm = b.smem(reads, min_len=min_len)
    owner = np.repeat(np.arange(k), np.diff(so[:k + 1].astype(np.int64)))
    bad = set()
    r1 = sub["round"] == 1
    smem_owner = np.repeat(np.arange(k), np.diff(s_off.astype(np.int64)))
    for i in range(k):
        a = sub[r1 & (owner == i)][["row", "rc_row", "count", "qbeg", "qend"]]
        w = sm[smem_owner == i][["row", "rc_row", "count", "qbeg", "qend"]]
        if a.size != w.size or not (a == w).all():
            bad.add(i)
    pieces = [reads[int(i)][int(x["qbeg"]):int(x["qend"])] for i, x in zip(owner, sub)]
    if pieces:
        cnt = b.count(pieces)
        bad.update(int(i) for i in owner[cnt != sub["count"]])
    for j, x in enumerate(sub):
        p, h = pieces[j], int(x["hit_begin"])
        for pos in hits["pos"][h:h + int(x["n_hits"])].tolist():
            if text[pos:pos + len(p)].tobytes() != p:
                bad.add(int(owner[j]))
                break
    return sorted(bad)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=1.5e9, help="bases of one strand")
    ap.add_argument("--records", type=int, default=12, help="records of one strand")
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--mutated", type=float, default=0.25, help="share of reads with 1-3 substitutions")
    ap.add_argument("--rate", type=int, default=32)
    ap.add_argument("--check", type=int, default=2000, help="reads checked as the scale test checks them")
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
    so = np.zeros(m + 1, dtype=np.uint64)
    nh = c_u64()
    opts = api.SeedOpts(19, 10, 20, 500, 1.5)
    P = lambda x: x.ctypes.data_as(c_p)  # noqa: E731
    lb = lib()
    head = (b._h, P(blob), P(offs), m, ctypes.addressof(opts), P(so), ctypes.addressof(nh))

    def query():
        check(lb.debwt_index_seeds(*head, c_p(0), 0, c_p(0), 0))

    query()                                                            # warm-up
    ms_q, all_q = timed(query, a.reps)
    total, total_hits = int(so[-1]), int(nh.value)
    seeds = np.zeros(total, dtype=api.SEED_DTYPE)
    hits = np.zeros(total_hits, dtype=api.HIT_DTYPE)

    def fill():
        check(lb.debwt_index_seeds(*head, P(seeds), total, P(hits), total_hits))

    fill()                                                             # warm-up
    ms_f, all_f = timed(fill, a.reps)

    k = min(a.check, m)
    bad = check_reads(b, [reads[i].tobytes() for i in range(k)], so, seeds, hits, text, 19)
    b.close()
    by_round = {str(r): int((seeds["round"] == r).sum()) for r in (1, 2, 3)}
    print(json.dumps({"sa_sample": {"rate": a.rate, "ms": sample_ms}}))
    res = {"gpu": info,
           "workload": {"n_symbols": n, "records": 2 * R, "bases_per_strand": F, "generator": "synth_gpu.genome_like(seed 5) + reverse complements"},
           "build_ms": build_ms, "sa_sample": {"rate": a.rate, "ms": sample_ms},
           "reads": {"n": m, "length": L, "reverse_strand": m // 2, "mutated": mutated, "seeds": [7, 8]},
           "options": {"min_seed_len": 19, "split_factor": 1.5, "split_width": 10, "max_mem_intv": 20, "max_occ": 500},
           "size_query_ms": ms_q, "size_query_ms_all": all_q, "fill_ms": ms_f, "fill_ms_all": all_f,
           "seeds_ms": ms_q + ms_f, "reads_per_s": m / ((ms_q + ms_f) / 1e3), "hits_per_s_fill": total_hits / (ms_f / 1e3),
           "seeds": total, "seeds_per_read": total / m, "seeds_per_read_by_round": {r: v / m for r, v in by_round.items()},
           "hits": total_hits, "hits_per_read": total_hits / m, "seeds_with_count_above_max_occ": int((seeds["count"] > 500).sum()),
           "kernel_ms": "not measured",
           "check": {"reads": k, "method": "round 1 = smem(), count = count(piece), hit text = piece", "reads_differing": len(bad),
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
