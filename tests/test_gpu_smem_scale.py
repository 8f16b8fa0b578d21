"""SMEM search at the size limit of one device: both strands of a genome_like text, T = n_max(24) symbols (about 4.29 G,
rows above 2^31).  For about 2000 seeded reads the SMEMs are derived through count alone (tests/smem_ref.smems_by_count:
start(e) by binary search for every end e) and compared with smem(), counts included; reverse-complement symmetry too.
Needs the memory of tests/test_gpu_scale.py's whole-path cases; skips, naming the amount, when it is not free."""
import numpy as np
import pytest
import torch

from debwt_b200 import api
from tests import smem_ref as ref
from tests.test_gpu_scale import _need, n_max

pytestmark = [pytest.mark.gpu, pytest.mark.slow]


def both_strands_text(n: int, R: int, seed: int):
    """(device text, seps): R records of genome_like(F, seed) and their reverse complements, N = 2 F + 2 R"""
    from debwt_b200 import synth_gpu
    F = (n - 2 * R) // 2
    seq = synth_gpu.genome_like(F, seed)
    per = -(-F // R)
    recs = [seq[i:i + per] for i in range(0, F, per)]
    return synth_gpu.join_records_device(recs + [synth_gpu.reverse_complement(r) for r in recs])


def seeded_reads(tnp: np.ndarray, seps: np.ndarray, k: int, length: int, seed: int) -> list:
    """k reads from positions inside records (half of them on the reverse copies), a quarter with 1-3 substitutions, some
    with an 'N'"""
    rng = np.random.default_rng(seed)
    n, R = tnp.size, seps.size // 2
    half = int(seps[R - 1]) + 1
    out = []
    while len(out) < k:
        lo, hi = (0, half) if len(out) % 2 == 0 else (half, n)
        s = int(rng.integers(lo, hi - length - 1))
        q = tnp[s:s + length]
        if (q > ord("T")).any() or (q == ord("#")).any() or (q == ord("$")).any():
            continue
        q = bytearray(q.tobytes())
        if rng.random() < 0.25:
            for p in rng.integers(0, length, int(rng.integers(1, 4))).tolist():
                q[p] = b"ACGT"[(b"ACGT".index(q[p]) + 1) % 4]
        if rng.random() < 0.05:
            q[int(rng.integers(0, length))] = ord("N")
        out.append(bytes(q))
    return out


def test_smem_complete_at_limit():
    _need(116, 25)
    R = 12
    n = n_max(2 * R)
    n -= (n - 2 * R) % 2
    text, seps = both_strands_text(n, R, 13)
    assert text.numel() == n and n > (1 << 32) - (1 << 17)
    with api.BwtBuilder(0) as b:
        b.set_text_device(text.data_ptr(), n, seps)
        b.build()
        tnp = text.cpu().numpy()
        del text
        torch.cuda.empty_cache()
        _, C = b.index()
        cnt = np.diff(C[:5].astype(np.int64))
        assert cnt[0] == cnt[3] and cnt[1] == cnt[2]
        reads = seeded_reads(tnp, seps, 2000, 150, 21)
        offs, sm = b.smem(reads, min_len=1)
        got = [[(int(x["qbeg"]), int(x["qend"]), int(x["count"])) for x in sm[int(offs[i]):int(offs[i + 1])]] for i in range(len(reads))]
        want = ref.smems_by_count(b.count, reads)
        bad = [i for i in range(len(reads)) if got[i] != want[i]]
        assert not bad, f"{len(bad)} reads differ, first {bad[0]}: {got[bad[0]]} != {want[bad[0]]}"
        assert (sm["row"] > (1 << 31)).any() and (sm["rc_row"] > (1 << 31)).any()
        # reverse-complement symmetry, rows included
        ro, rs = b.smem([ref.revcomp(q) for q in reads], min_len=1)
        full = [[(int(x["qbeg"]), int(x["qend"]), int(x["row"]), int(x["rc_row"]), int(x["count"])) for x in sm[int(offs[i]):int(offs[i + 1])]]
                for i in range(len(reads))]
        for i, q in enumerate(reads):
            m = len(q)
            r = [(int(x["qbeg"]), int(x["qend"]), int(x["row"]), int(x["rc_row"]), int(x["count"])) for x in rs[int(ro[i]):int(ro[i + 1])]]
            assert r == sorted((m - e, m - s, l, k, c) for s, e, k, l, c in full[i]), i
