"""SMEM search (debwt_index_smem, BwtBuilder.smem) through the C ABI against the FMD-index model of tests/smem_ref.py, exactly
(qbeg, qend, row, rc_row, count), on both strands of the seeded cases; the rows against the sampled suffix array and the
text; loaded results; and the error paths."""
import functools

import numpy as np
import pytest

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from tests import smem_ref as ref
from tests.util import as_bytes_records, golden, seeded_records

pytestmark = pytest.mark.gpu

CASES = ["c3_like_600k_3rec", "c4_like_5x100k", "c2_like_1m"]

_LUT = np.full(256, 255, dtype=np.uint8)
for _c, _v in ((b"A", 0), (b"C", 1), (b"G", 2), (b"T", 3), (b"#", 4), (b"$", 5)):
    _LUT[_c[0]] = _v


@functools.lru_cache(maxsize=1)
def _case(name):
    both = api.both_strands(as_bytes_records(seeded_records(name)))
    text, seps = api.join_records(both)
    return both, text, seps, ref.FmdModel(_LUT[text])


def _mutate(q, rng, k):
    q = bytearray(q)
    for p in rng.choice(len(q), size=k, replace=False).tolist():
        q[p] = b"ACGT"[(b"ACGT".index(q[p]) + int(rng.integers(1, 4))) % 4]
    return bytes(q)


def _reads(both, rng):
    """exact reads from both strands, reads with 1-3 substitutions, reads across two records, reads with 'N' and lower
    case, a 20-kbp read, a 1-base read and an empty one"""
    R = len(both) // 2
    out = []
    for j in range(480):
        rec = int(rng.integers(0, R)) + (R if j % 2 else 0)
        r = both[rec]
        L = int(rng.integers(100, 151))
        a = int(rng.integers(0, len(r) - L))
        q = r[a:a + L]
        kind = j // 2 % 4
        if kind == 1:
            q = _mutate(q, rng, int(rng.integers(1, 4)))
        elif kind == 2:
            nxt = both[(rec + 1) % len(both)]
            k = int(rng.integers(20, L - 20))
            q = r[len(r) - k:] + nxt[:L - k]
        elif kind == 3:
            q = bytearray(q)
            for p in rng.choice(L, size=int(rng.integers(1, 4)), replace=False).tolist():
                q[p] = ord("N")
            lo = int(rng.integers(0, L))
            q = bytes(q[:lo]) + bytes(q[lo:lo + 40]).lower() + bytes(q[lo + 40:])
        out.append(q)
    r = both[0]
    out.append(_mutate(r[len(r) // 3:len(r) // 3 + 20_000], rng, 12))
    out += [b"C", b"", b"n", b"A" * 60, b"acgt"]
    return out


def _tuples(offs, sm):
    rows = [(int(a["qbeg"]), int(a["qend"]), int(a["row"]), int(a["rc_row"]), int(a["count"])) for a in sm]
    return [rows[int(offs[i]):int(offs[i + 1])] for i in range(offs.size - 1)]


def _check_rows(b, reads, offs, sm, text, k=300):
    """every hit of the first k SMEMs, located through sa(): row -> the match, rc_row -> its reverse complement; the rows
    are the ones locate finds for the same piece"""
    n = text.size
    owner = np.repeat(np.arange(offs.size - 1), np.diff(offs.astype(np.int64)))
    t = text.tobytes()
    sel = sm[:k]
    pats = [reads[int(owner[j])][int(x["qbeg"]):int(x["qend"])].upper() for j, x in enumerate(sel)]
    hits, pos = b.locate(pats)
    for j, (x, p) in enumerate(zip(sel, pats)):
        c = int(x["count"])
        assert c >= 1 and int(hits[j + 1] - hits[j]) == c
        fw = b.sa(np.arange(int(x["row"]), int(x["row"]) + c, dtype=np.uint64)).astype(np.int64)
        rc = b.sa(np.arange(int(x["rc_row"]), int(x["rc_row"]) + c, dtype=np.uint64)).astype(np.int64)
        assert (fw < n).all() and (rc < n).all()
        assert sorted(fw.tolist()) == sorted(pos[int(hits[j]):int(hits[j + 1])].astype(np.int64).tolist())
        assert all(t[q:q + len(p)] == p for q in fw.tolist())
        assert all(t[q:q + len(p)] == ref.revcomp(p) for q in rc.tolist())


@pytest.mark.parametrize("name", CASES)
def test_smem_equals_model(name):
    both, text, seps, model = _case(name)
    rng = np.random.default_rng(31)
    reads = _reads(both, rng)
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        offs, sm = b.smem(reads, min_len=1)
        got = _tuples(offs, sm)
        assert offs.size == len(reads) + 1 and sm.dtype == api.SMEM_DTYPE
        for i, q in enumerate(reads):
            assert got[i] == model.smems(q), (i, len(q))
        assert len(got[-5]) == 1 and got[-4] == [] and got[-3] == []   # 'C' occurs; '' and 'n' hold no base
        assert len(got[-6]) >= 1                                       # the 20-kbp read
        # min_len = the filtered min_len = 1 output
        for k in (19, 40):
            o2, s2 = b.smem(reads, min_len=k)
            assert _tuples(o2, s2) == [[x for x in g if x[1] - x[0] >= k] for g in got]
        # reverse-complement symmetry
        ro, rs = b.smem([ref.revcomp(q) for q in reads], min_len=1)
        for q, g, r in zip(reads, got, _tuples(ro, rs)):
            m = len(q)
            assert r == sorted((m - e, m - s, l, k, c) for s, e, k, l, c in g)
        b.sample_sa(16)
        _check_rows(b, reads, offs, sm, text)


def test_poly_a_against_longer_runs():
    """a 2000-base poly-A read against a text with longer A runs: every forward step loses one occurrence, so the interval
    lists grow as long as the read"""
    rng = np.random.default_rng(4)
    acgt = b"ACGT"
    rnd = lambda k: bytes(acgt[int(x)] for x in rng.integers(0, 4, k))  # noqa: E731
    recs = [rnd(40_000), b"A" * 3000 + rnd(500), rnd(200) + b"A" * 2500 + rnd(300), b"C" + b"A" * 2100]
    both = api.both_strands(recs)
    text, _ = api.join_records(both)
    model = ref.FmdModel(_LUT[text])
    reads = [b"A" * 2000, b"a" * 2000, b"T" * 2000, b"G" + b"A" * 2000 + b"C", b"A" * 3500, b"A" * 1000 + b"N" + b"A" * 999,
             rnd(150), b"C" + b"A" * 2101]
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        offs, sm = b.smem(reads, min_len=1)
        got = _tuples(offs, sm)
    for i, q in enumerate(reads):
        assert got[i] == model.smems(q), i
    assert got[0] == [(0, 2000, *model.interval(b"A" * 2000))]
    runs = [len(r) for r in text.tobytes().translate(bytes.maketrans(b"CGT#$", b"xxxxx")).split(b"x")]
    assert got[0][0][4] == sum(r - 2000 + 1 for r in runs if r >= 2000)              # the windows of the A runs
    top = max(runs)
    assert 3000 <= top < 3500
    assert [x[:2] for x in got[4]] == [(s, s + top) for s in range(3500 - top + 1)]   # every window of the longest run


def test_megabase_read_among_short_reads():
    """a 1-Mbp read sizes the scratch slots (64 MB each, 16 of them), so the short reads queue on the work counter"""
    both, text, seps, model = _case("c2_like_1m")
    rng = np.random.default_rng(12)
    rec = both[0]
    assert len(rec) == 1_000_000
    short = [_mutate(rec[a:a + 150], rng, int(rng.integers(0, 3))) for a in rng.integers(0, len(rec) - 150, 300).tolist()]
    reads = short[:150] + [rec] + short[150:]
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        offs, sm = b.smem(reads, min_len=1)
        got = _tuples(offs, sm)
        cnt = int(b.count([rec])[0])
    k, l, s = model.interval(rec)
    assert got[150] == [(0, len(rec), k, l, s)] and s == cnt >= 1
    for i, q in enumerate(reads):
        if i != 150:
            assert got[i] == model.smems(q), i


def test_loaded_result_same_answers(tmp_path):
    both, text, seps, model = _case("c4_like_5x100k")
    reads = _reads(both, np.random.default_rng(77))
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        words, sharp, dollar = b.result()
        want = b.smem(reads, min_len=5)
    path = str(tmp_path / "c4_both.bwt")
    api.write_outputs(path, words, sharp, dollar)
    with api.BwtBuilder() as c:
        w, s, d = api.read_outputs(path, text.size)
        c.set_result(w, text.size, s, d)
        got = c.smem(reads, min_len=5)
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
    assert _tuples(*got) == [model.smems(q, 5) for q in reads]


def test_errors():
    recs = [r.upper().encode() for r in golden()["small"]["haplotypes_6x1500"]["records"]]
    both = api.both_strands(recs)
    L = binding.lib()
    SENT = 0xA5A5A5A5A5A5A5A5

    def raw(b, reads, min_len, cap, offs=None, null=""):
        blob = np.frombuffer(b"".join(reads) + b"\0", dtype=np.uint8)
        if offs is None:
            offs = np.concatenate(([0], np.cumsum([len(r) for r in reads]))).astype(np.uint64)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        so = np.full(len(reads) + 1, SENT, dtype=np.uint64)
        sm = np.zeros(max(cap, 1) + 4, dtype=api.SMEM_DTYPE)
        sm["row"] = SENT
        rc = L.debwt_index_smem(b._h, None if null == "reads" else api._ptr(blob), None if null == "offsets" else api._ptr(offs),
                                len(reads), min_len, None if null == "smem_offsets" else api._ptr(so),
                                None if null == "smems" else api._ptr(sm), cap)
        return rc, so, sm, L.debwt_last_error().decode()

    reads = [q[100:160] for q in both] + [b"ACGTN" * 9]
    with api.BwtBuilder() as b:
        b.set_records(recs)                                       # one strand only
        b.build()
        rc, so, sm, msg = raw(b, reads, 1, 100)
        assert rc != 0 and "no index" in msg and (so == SENT).all() and (sm["row"] == SENT).all()
        b.index()
        rc, so, sm, msg = raw(b, reads, 1, 100)
        assert rc != 0 and "reverse complement" in msg and (so == SENT).all() and (sm["row"] == SENT).all()
        _, C = b.index()
        for base, v in zip("ACGT", np.diff(C[:5]).tolist()):
            assert f"{base} = {v}" in msg
        with pytest.raises(DebwtError, match="both_strands"):
            b.smem(reads)

    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.index()
        offs, sm0 = b.smem(reads, min_len=1)
        total = int(offs[-1])
        assert total >= len(reads) - 1
        rc, so, sm, msg = raw(b, reads, 1, total - 1)             # too small: names the total
        assert rc != 0 and str(total) in msg and (so == offs).all() and (sm["row"] == SENT).all()
        rc, so, sm, msg = raw(b, reads, 1, total)
        assert rc == 0 and (so == offs).all() and (sm[:total] == sm0).all() and (sm["row"][total:] == SENT).all()
        rc, so, sm, msg = raw(b, reads, 1, 0, null="smems")       # size query
        assert rc == 0 and (so == offs).all()
        rc, so, sm, msg = raw(b, reads, 0, 100)
        assert rc != 0 and "min_len" in msg and (so == SENT).all() and (sm["row"] == SENT).all()
        for null in ("reads", "offsets", "smem_offsets"):
            rc, so, sm, msg = raw(b, reads, 1, 100, null=null)
            assert rc != 0 and "null argument" in msg and (sm["row"] == SENT).all(), null
            if null != "smem_offsets":
                assert (so == SENT).all()
        bad = np.array([0, 60, 50, 120], dtype=np.uint64)
        rc, so, sm, msg = raw(b, [b"A" * 40] * 3, 1, 100, offs=bad)
        assert rc != 0 and "read 1" in msg and (so == SENT).all()
        huge = [b"ACGT" * 10, b"A" * (1 << 24)]                    # 2 (2^24 + 1) entries of 32 bytes > 1 GiB
        rc, so, sm, msg = raw(b, huge, 1, 100)
        assert rc != 0 and "read 1" in msg and str(1 << 24) in msg and (so == SENT).all()
        rc, so, sm, msg = raw(b, [], 1, 0)                          # no reads
        assert rc == 0 and int(so[0]) == 0
        o, s = b.smem([])
        assert o.tolist() == [0] and s.size == 0
