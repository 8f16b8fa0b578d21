"""The seed-extension restatement of tests/ext_ref.py without a GPU: its Python and C DP routines against each other and
against a brute-force Gotoh, the planted outcomes of ksw_extend2, mem_flt_chained_seeds' early return and seed drop, and
each path of mem_chain2aln on hand-built chains."""
import ctypes

import numpy as np
import pytest

from debwt_b200 import api
from tests import ext_ref as er

D = er.DEFAULTS


def _rand(rng, n):
    return rng.integers(0, 4, n).astype(np.uint8)


def test_python_and_c_dp_agree():
    rng = np.random.default_rng(1)
    opt_sets = [D, dict(D, o_del=2, e_del=3, o_ins=5, e_ins=1), dict(D, a=2, b=1, o_del=0, o_ins=0), dict(D, zdrop=1), dict(D, zdrop=0)]
    n = 0
    for k in range(3000):
        o = opt_sets[k % len(opt_sets)]
        qlen = int(rng.integers(1, 12)) if k % 7 else 1
        tlen = int(rng.integers(0, 3)) if k % 5 == 0 else int(rng.integers(0, 14))
        q = _rand(rng, qlen)
        if k % 3 == 0:
            q[rng.integers(0, qlen)] = 4
        t = _rand(rng, tlen)
        if k % 2 and tlen:                                                 # related sequences reach deeper cells
            t[:min(qlen, tlen)] = np.where(q[:min(qlen, tlen)] > 3, 0, q[:min(qlen, tlen)])
        w = int(rng.integers(0, 4))
        h0 = [1, 2, 7, 30, 1000][k % 5]
        eb = int(rng.integers(0, 6))
        assert er.extend_py(q, t, w, eb, h0, o) == er.extend_c(q, t, w, eb, h0, o), (q, t, w, eb, h0, o)
        assert er.seed_sw_py(q, t, o) == er.seed_sw_c(q, t, o)
        n += 1
    assert n == 3000


def _gotoh_brute(q, t, o):
    """local alignment with gaps of every length enumerated: H(i, j) = max(0, H(i-1, j-1) + s, max_k H(i-k, j) - o_del -
    k e_del, max_k H(i, j-k) - o_ins - k e_ins)"""
    n, m = len(t), len(q)
    H = [[0] * (m + 1) for _ in range(n + 1)]
    best = 0
    for i in range(1, n + 1):
        for j in range(1, m + 1):
            h = max(0, H[i - 1][j - 1] + er.score(o, t[i - 1], q[j - 1]))
            for k in range(1, i + 1):
                h = max(h, H[i - k][j] - o["o_del"] - k * o["e_del"])
            for k in range(1, j + 1):
                h = max(h, H[i][j - k] - o["o_ins"] - k * o["e_ins"])
            H[i][j] = h
            best = max(best, h)
    return best


def test_local_score_is_gotoh():
    rng = np.random.default_rng(2)
    for k in range(300):
        o = [D, dict(D, o_del=1, e_del=2, o_ins=3, e_ins=1), dict(D, a=3, b=2, o_del=0, e_del=1, o_ins=0, e_ins=2)][k % 3]
        q, t = _rand(rng, int(rng.integers(1, 10))), _rand(rng, int(rng.integers(0, 10)))
        if k % 2 and t.size > 3:
            t = np.concatenate((t[:2], q, t[2:]))[:12]
        assert er.seed_sw_c(q, t, o) == _gotoh_brute(q, t, o) == er.seed_sw_py(q, t, o)


def test_extend_outcomes():
    rng = np.random.default_rng(3)
    q = _rand(rng, 120)
    t = np.concatenate((q, _rand(rng, 30)))
    x = er.extend_c(q, t, 100, 5, 40, D)                                  # an exact continuation
    assert x[0] == 40 + len(q) and x[1] == len(q) and x[4] == 40 + len(q)
    assert er.extend_py(q, t, 100, 5, 40, D) == x
    # two 16-base deletions at w = 20: after the first the best cell is 16 > 3/4 w off the diagonal, so max_off reaches
    # (20 >> 1) + (20 >> 2) = 15; the second is 32 off, inside only the doubled band
    o = dict(D, o_del=2, e_del=1)
    q = _rand(rng, 200)
    t = np.concatenate((q[:60], _rand(rng, 16), q[60:120], _rand(rng, 16), q[120:]))
    x1, x2 = er.extend_c(q, t, 20, 5, 30, o), er.extend_c(q, t, 40, 5, 30, o)
    assert x1[5] >= (20 >> 1) + (20 >> 2) and x2[0] != x1[0]
    assert er.extend_py(q, t, 40, 5, 30, o) == x2
    # z-drop: a divergent stretch ends the extension at zdrop 10; without z-drop it goes on to the matching bases after it
    a, x, y, b = _rand(rng, 60), _rand(rng, 20), _rand(rng, 20), _rand(rng, 200)
    q, t = np.concatenate((a, x, b)), np.concatenate((a, y, b))
    z = er.extend_c(q, t, 100, 5, 30, dict(D, zdrop=10))
    nz = er.extend_c(q, t, 100, 5, 30, dict(D, zdrop=0))
    assert z[0] < 30 + 80 and z[1] <= 80 and nz[0] > 30 + 200 and nz[1] == len(q)
    assert er.extend_py(q, t, 100, 5, 30, dict(D, zdrop=10)) == z


def _pac(recs):
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    return er.Pac(text, seps), text, seps


def test_flt_chained_seeds():
    rng = np.random.default_rng(4)
    assert 5.5 * np.log(725) < 0.05 * 725 and 5.5 * np.log(700) > 0.05 * 700
    rec = bytes(b"ACGT"[i] for i in rng.integers(0, 4, 5000))
    pac, _, _ = _pac([rec])
    for L, ran in ((700, False), (760, True)):
        read = bytearray(rec[1000:1000 + L])
        q = er.nt4(bytes(read))
        good = (1000 + 100, 100, 60)
        bad = (3000, 300, 20)                                             # a 20-base seed at the wrong place: SW far below min_HSP
        fl, r = er.flt_chained_seeds(D, pac, q, L, [dict(seeds=[good, bad], record=0)])
        assert r == ran
        if not ran:
            assert fl == [[good + (60,), bad + (20,)]]                    # scores are len, without the factor a
        else:
            assert fl[0][0][:3] == good and fl[0][0][3] >= 60 and len(fl[0]) == 1
    long_seed = (1000, 0, 250)
    fl, _ = er.flt_chained_seeds(dict(D, a=2), pac, er.nt4(rec[1000:1760]), 760, [dict(seeds=[long_seed], record=0)])
    assert fl == [[long_seed + (500,)]]                                   # len >= 200: no SW, score len a


def _chain(seeds, record=0, strand=0):
    return dict(seeds=seeds, record=record, strand=strand, frac_rep=0.0)


def test_chain2aln_paths():
    rng = np.random.default_rng(5)
    recs = [bytes(b"ACGT"[i] for i in rng.integers(0, 4, n)) for n in (3000, 2000)]
    pac, _, _ = _pac(recs)
    lp = pac.l_pac
    assert lp == 5000
    read = recs[0][500:650]
    # one chain, two seeds on one diagonal: the second is inside the first's region and skipped
    tr = []
    regs = er.read_regions(D, 100, pac, read, [_chain([(520, 20, 40), (600, 100, 30)])], trace=tr)
    assert len(regs) == 1 and "skip" in tr and regs[0]["qb"] == 0 and regs[0]["qe"] == 150 and regs[0]["score"] == 150
    assert regs[0]["rb"] == 500 and regs[0]["re"] == 650 and regs[0]["seedcov"] == 70 and regs[0]["seedlen0"] == 40
    # the overlap test: a contained seed on another diagonal that overlaps a long enough seed is extended anyway
    tr = []
    regs = er.read_regions(D, 100, pac, read, [_chain([(520, 20, 40), (530, 22, 39)])], trace=tr)
    assert "revived" in tr and len(regs) == 2
    # qbeg = 0 and a seed ending at the read's end
    tr = []
    regs = er.read_regions(D, 100, pac, read, [_chain([(500, 0, 150)])], trace=tr)
    assert "qbeg0" in tr and "qend_L" in tr and regs[0]["score"] == 150 and regs[0]["truesc"] == 150
    # a window clipped at a record edge: a read that starts 10 bases before record 1 (whose bases follow record 0's)
    read2 = b"T" * 10 + recs[1][:140]
    tr = []
    regs = er.read_regions(D, 100, pac, read2, [_chain([(3000, 10, 140)], record=1)], trace=tr)
    assert "clip" in tr and regs[0]["rb"] >= 3000
    # a window crossing l_pac: a reverse-strand seed at the start of the reverse strand
    rc = bytes(recs[1][::-1]).translate(bytes.maketrans(b"ACGT", b"TGCA"))
    read3 = rc[:150]
    tr = []
    regs = er.read_regions(D, 100, pac, read3, [_chain([(lp + 50, 50, 100)], record=1, strand=1)], trace=tr)
    assert "cross" in tr and regs[0]["rb"] == lp and regs[0]["score"] == 150
    # a chain emptied by the seed filter (long read, a seed that does not align)
    long_read = recs[0][:800]
    tr = []
    regs = er.read_regions(D, 100, pac, long_read, [_chain([(2500, 300, 19)]), _chain([(0, 0, 300)])], trace=tr)
    assert "empty" in tr and "dropped" in tr and len(regs) == 1 and regs[0]["chain"] == 1
    # local and to-end outcomes for both clipping penalties: a read whose ends do not match the reference
    tail = bytes(b"ACGT"[i] for i in rng.integers(0, 4, 12))
    read4 = tail + recs[0][1000:1100] + tail
    seen = set()
    for pen in (0, 1000):
        tr = []
        o = dict(D, pen_clip5=pen, pen_clip3=pen)
        er.read_regions(o, 100, pac, read4, [_chain([(1000, 12, 100)])], trace=tr)
        seen.update(x for x in tr if isinstance(x, str))
    assert {"left_local", "left_end", "right_local", "right_end"} <= seen, seen


def test_region_layout():
    assert api.REGION_DTYPE.itemsize == 64 and ctypes.sizeof(api.ExtOpts) == 36
    assert [f for f in api.REGION_DTYPE.names if f != "pad_"] == list(er.FIELDS)
    assert api.REGION_DTYPE.fields["chain"][1] == 44 and api.REGION_DTYPE.fields["frac_rep"][1] == 56


@pytest.mark.parametrize("pen", [0, 5])
def test_reference_over_python_dp(pen):
    """the regions reference gives the same regions with the Python DP as with the C twin"""
    rng = np.random.default_rng(6)
    recs = [bytes(b"ACGT"[i] for i in rng.integers(0, 4, 1500))]
    pac, _, _ = _pac(recs)
    read = bytearray(recs[0][200:330])
    for p in (5, 60, 61, 62, 100):
        read[p] = ord("ACGT"[(b"ACGT".index(read[p]) + 1) % 4])
    chains = [_chain([(200, 0, 5), (206, 6, 54), (263, 63, 37)]), _chain([(700, 10, 20)])]
    o = dict(D, pen_clip5=pen, pen_clip3=pen)
    a = er.read_regions(o, 100, pac, bytes(read), chains)
    b = er.read_regions(o, 100, pac, bytes(read), chains, dp=er.extend_py, sw=er.seed_sw_py)
    assert a == b and len(a) >= 2
