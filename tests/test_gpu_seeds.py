"""BWA-MEM seed collection (debwt_index_seeds, BwtBuilder.seeds) through the C ABI against tests/seed_ref.py, exactly (seeds
and located hits), on both strands of the seeded cases and read mix of tests/test_gpu_smem.py; consistency with smem(),
sa(), the text and api.strand_offsets; a repeat above max_occ; long reads; rate, loaded results and the separator cache;
and the error paths."""
import ctypes
import functools

import numpy as np
import pytest

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from tests import seed_ref as sr
from tests import smem_ref as ref
from tests.locate_ref import suffix_array
from tests.test_gpu_smem import _LUT, CASES, _case, _mutate, _reads
from tests.util import golden

pytestmark = pytest.mark.gpu

OPTS = [dict(sr.DEFAULTS), dict(min_len=15, split_factor=1.2, split_width=20, max_mem_intv=0, max_occ=3)]


@functools.lru_cache(maxsize=1)
def _sa(name):
    return suffix_array(_LUT[_case(name)[1]])


def _tuples(seeds, hits):
    s = [(int(x["qbeg"]), int(x["qend"]), int(x["round"]), int(x["row"]), int(x["rc_row"]), int(x["count"]), int(x["hit_begin"]),
          int(x["n_hits"])) for x in seeds]
    h = [(int(x["pos"]), int(x["offset"]), int(x["record"]), int(x["strand"])) for x in hits]
    return s, h


def _check_consistency(b, reads, o, offs, seeds, hits, text, seps):
    """round 1 = smem(); every hit's text is its piece; pos = sa(row + j step); (record, strand, offset) = strand_offsets"""
    so, sm = b.smem(reads, min_len=o["min_len"])
    owner = np.repeat(np.arange(len(reads)), np.diff(offs.astype(np.int64)))
    r1 = seeds[seeds["round"] == 1]
    want = sm[["row", "rc_row", "count", "qbeg", "qend"]]
    assert (r1[["row", "rc_row", "count", "qbeg", "qend"]] == want).all() and r1.size == sm.size
    assert (np.repeat(np.arange(len(reads)), np.diff(so.astype(np.int64))) == owner[seeds["round"] == 1]).all()
    assert (seeds["n_hits"] == np.minimum(seeds["count"], o["max_occ"])).all()
    assert (seeds["hit_begin"] == np.concatenate(([0], np.cumsum(seeds["n_hits"].astype(np.uint64))[:-1]))).all()
    t = text.tobytes()
    rows = []
    for x in seeds:
        rows += sr.hit_rows(int(x["row"]), int(x["count"]), o["max_occ"])
    assert (b.sa(np.array(rows, dtype=np.uint64)) == hits["pos"]).all()
    for j, x in enumerate(seeds):
        q = reads[int(owner[j])][int(x["qbeg"]):int(x["qend"])].upper()
        h = hits[int(x["hit_begin"]):int(x["hit_begin"]) + int(x["n_hits"])]
        assert all(t[p:p + len(q)] == q for p in h["pos"].tolist())
        rec, strand, off = api.strand_offsets(h["pos"], len(q), seps)
        assert (rec == h["record"]).all() and (strand == h["strand"]).all() and (off == h["offset"]).all()


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("opt", range(len(OPTS)))
def test_seeds_equal_reference(name, opt):
    o = OPTS[opt]
    both, text, seps, model = _case(name)
    reads = _reads(both, np.random.default_rng(31))
    want = sr.reference(model, _sa(name), seps, reads, **o)
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(16)
        offs, seeds, hits = b.seeds(reads, **o)
        assert seeds.dtype == api.SEED_DTYPE and hits.dtype == api.HIT_DTYPE
        assert offs.tolist() == want[0]
        got = _tuples(seeds, hits)
        assert got[0] == want[1]
        assert got[1] == want[2]
        for r in (1, 2, 3):                                          # every round fires; round 3 only when switched on
            assert (seeds["round"] == r).any() == (r < 3 or o["max_mem_intv"] > 0), r
        if o["max_occ"] == 3 and name != "c2_like_1m":                 # step > 1 (no piece of c2's reads occurs 6 times)
            assert (seeds["count"] >= 6).any()
        _check_consistency(b, reads, o, offs, seeds, hits, text, seps)


def test_repeat_above_default_max_occ():
    """a 40-base unit in 1100 copies: its seeds have 500 hits, every (count // 500)-th row"""
    rng = np.random.default_rng(9)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    unit = acgt[rng.integers(0, 4, 40)].tobytes()
    recs = [bytearray(acgt[rng.integers(0, 4, 150_000)].tobytes()) for _ in range(2)]
    for j in range(1100):
        r = recs[j % 2]
        p = 100 * (j // 2) + 30
        r[p:p + 40] = unit
    recs = [bytes(r) for r in recs]
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    model = ref.FmdModel(_LUT[text])
    sa = suffix_array(_LUT[text])
    reads = [recs[0][100 * k:100 * k + 150] for k in (3, 40, 200)] + [_mutate(recs[1][100 * k + 10:100 * k + 130], rng, 2) for k in (7, 77)]
    reads += [b"GATTACA" + unit + b"CAT", unit]
    o = dict(sr.DEFAULTS)
    want = sr.reference(model, sa, seps, reads, **o)
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(32)
        offs, seeds, hits = b.seeds(reads)
        assert offs.tolist() == want[0] and _tuples(seeds, hits) == (want[1], want[2])
        big = seeds[seeds["count"] > 1000]
        assert big.size and (big["n_hits"] == 500).all()
        _check_consistency(b, reads, o, offs, seeds, hits, text, seps)


def test_poly_a_and_megabase_reads():
    """a poly-A read against longer A runs (lists as long as the read), and a 1-Mbp read among short reads (the scratch
    slots are sized by it)"""
    rng = np.random.default_rng(4)
    acgt = b"ACGT"
    rnd = lambda k: bytes(acgt[int(x)] for x in rng.integers(0, 4, k))  # noqa: E731
    recs = [rnd(40_000), b"A" * 3000 + rnd(500), rnd(200) + b"A" * 2500 + rnd(300), b"C" + b"A" * 2100]
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    model = ref.FmdModel(_LUT[text])
    sa = suffix_array(_LUT[text])
    reads = [b"A" * 2000, b"G" + b"A" * 2000 + b"C", b"A" * 1000 + b"N" + b"A" * 999, b"C" + b"A" * 2101, b"A" * 2400, rnd(150)]
    want = sr.reference(model, sa, seps, reads, **sr.DEFAULTS)
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(8)
        offs, seeds, hits = b.seeds(reads)
        assert offs.tolist() == want[0] and _tuples(seeds, hits) == (want[1], want[2])
        assert (seeds["qend"] - seeds["qbeg"] >= 2000).any() and (seeds["round"] == 2).any()

    both, text, seps, model = _case("c2_like_1m")
    rec = both[0]
    short = [_mutate(rec[a:a + 150], rng, int(rng.integers(0, 3))) for a in rng.integers(0, len(rec) - 150, 300).tolist()]
    reads = short[:150] + [rec] + short[150:]
    want = sr.reference(model, _sa("c2_like_1m"), seps, reads, **sr.DEFAULTS)
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(16)
        offs, seeds, hits = b.seeds(reads)
        assert offs.tolist() == want[0] and _tuples(seeds, hits) == (want[1], want[2])
        mega = seeds[int(offs[150]):int(offs[151])]
        assert mega.size > 1000 and mega[0]["qbeg"] == 0 and (mega["round"] == 1).sum() == 1


def test_rate_loaded_result_and_separator_cache(tmp_path):
    both, text, seps, model = _case("c4_like_5x100k")
    reads = _reads(both, np.random.default_rng(77))
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        b.sample_sa(1)
        want = b.seeds(reads)
        b.sample_sa(64)
        got = b.seeds(reads)
        assert all((x == y).all() for x, y in zip(got, want))
        words, sharp, dollar = b.result()
    api.write_outputs(str(tmp_path / "c4.bwt"), words, sharp, dollar)

    # another text whose records have other lengths: stale separators would misplace every hit
    both2, text2, seps2, model2 = _case("c3_like_600k_3rec")
    reads2 = _reads(both2, np.random.default_rng(78))
    with api.BwtBuilder() as c:
        w, s, d = api.read_outputs(str(tmp_path / "c4.bwt"), text.size)
        c.set_result(w, text.size, s, d)
        c.sample_sa(32)
        got = c.seeds(reads)
        assert all((x == y).all() for x, y in zip(got, want))
        with api.BwtBuilder() as e:
            e.set_records(both2)
            e.build()
            w2, s2, d2 = e.result()
        c.set_result(w2, text2.size, s2, d2)
        c.sample_sa(32)
        offs, seeds, hits = c.seeds(reads2)
        ref2 = sr.reference(model2, _sa("c3_like_600k_3rec"), seps2, reads2, **sr.DEFAULTS)
        assert offs.tolist() == ref2[0] and _tuples(seeds, hits) == (ref2[1], ref2[2])


def test_errors():
    recs = [r.upper().encode() for r in golden()["small"]["haplotypes_6x1500"]["records"]]
    both = api.both_strands(recs)
    L = binding.lib()
    SENT = 0xA5A5A5A5A5A5A5A5

    def raw(b, reads, cap=100, hcap=1000, offs=None, null="", **kw):
        o = {**dict(min_len=19, split_width=10, max_mem_intv=20, max_occ=500, split_factor=1.5), **kw}
        opts = api.SeedOpts(o["min_len"], o["split_width"], o["max_mem_intv"], o["max_occ"], o["split_factor"])
        blob = np.frombuffer(b"".join(reads) + b"\0", dtype=np.uint8)
        if offs is None:
            offs = np.concatenate(([0], np.cumsum([len(r) for r in reads]))).astype(np.uint64)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        so = np.full(len(reads) + 1, SENT, dtype=np.uint64)
        nh = np.full(1, SENT, dtype=np.uint64)
        sd = np.zeros(max(cap, 1) + 4, dtype=api.SEED_DTYPE)
        sd["row"] = SENT
        ht = np.zeros(max(hcap, 1) + 4, dtype=api.HIT_DTYPE)
        ht["pos"] = SENT
        P = lambda name, a: None if null == name else api._ptr(a)  # noqa: E731
        rc = L.debwt_index_seeds(b._h, P("reads", blob), P("offsets", offs), len(reads), None if null == "opts" else
                                 ctypes.addressof(opts), P("seed_offsets", so), P("n_hits", nh), P("seeds", sd), cap,
                                 P("hits", ht), hcap)
        return rc, so, nh, sd, ht, L.debwt_last_error().decode()

    def untouched(so, nh, sd, ht):
        return (so == SENT).all() and (nh == SENT).all() and (sd["row"] == SENT).all() and (ht["pos"] == SENT).all()

    reads = [q[100:180] for q in both] + [b"ACGTN" * 9]
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.index()
        rc, so, nh, sd, ht, msg = raw(b, reads)                     # no samples
        assert rc != 0 and "debwt_index_sample_sa" in msg and untouched(so, nh, sd, ht)
        with pytest.raises(DebwtError, match="sample_sa"):
            b.seeds(reads)
        b.sample_sa(32)
        offs, seeds, hits = b.seeds(reads)
        total, th = int(offs[-1]), hits.size
        assert total >= len(reads) - 1 and th >= total
        for cap, hcap in ((total - 1, th), (total, th - 1)):        # too small: names both totals, writes no seed or hit
            rc, so, nh, sd, ht, msg = raw(b, reads, cap, hcap)
            assert rc != 0 and str(total) in msg and str(th) in msg and (so == offs).all() and int(nh[0]) == th
            assert (sd["row"] == SENT).all() and (ht["pos"] == SENT).all()
        rc, so, nh, sd, ht, msg = raw(b, reads, total, th)
        assert rc == 0 and (so == offs).all() and (sd[:total] == seeds).all() and (ht[:th] == hits).all()
        assert (sd["row"][total:] == SENT).all() and (ht["pos"][th:] == SENT).all()
        rc, so, nh, sd, ht, msg = raw(b, reads, 0, 0, null="seeds")  # size query
        assert rc == 0 and (so == offs).all() and int(nh[0]) == th and (sd["row"] == SENT).all() and (ht["pos"] == SENT).all()
        for kw, word in ((dict(min_len=0), "min_seed_len"), (dict(max_occ=0), "max_occ"), (dict(split_factor=-1.0), "split_factor"),
                         (dict(split_factor=float("nan")), "split_factor"), (dict(split_factor=float("inf")), "split_factor")):
            rc, so, nh, sd, ht, msg = raw(b, reads, **kw)
            assert rc != 0 and word in msg and untouched(so, nh, sd, ht), kw
        for null in ("reads", "offsets", "seed_offsets", "n_hits", "opts", "hits"):
            rc, so, nh, sd, ht, msg = raw(b, reads, null=null)
            assert rc != 0 and "null argument" in msg and (sd["row"] == SENT).all() and (ht["pos"] == SENT).all(), null
            assert (so == SENT).all() and (nh == SENT).all(), null
        rc, so, nh, sd, ht, msg = raw(b, [b"A" * 40] * 3, offs=np.array([0, 60, 50, 120], dtype=np.uint64))
        assert rc != 0 and "read 1" in msg and untouched(so, nh, sd, ht)
        rc, so, nh, sd, ht, msg = raw(b, [b"ACGT" * 10, b"A" * (1 << 24)])    # 72 * 2^24 + 64 bytes > 1 GiB
        assert rc != 0 and "read 1" in msg and str(1 << 24) in msg and str(((1 << 30) - 64) // 72) in msg and untouched(so, nh, sd, ht)
        rc, so, nh, sd, ht, msg = raw(b, [], 0, 0)                  # no reads
        assert rc == 0 and int(so[0]) == 0 and int(nh[0]) == 0
        o, s, h = b.seeds([])
        assert o.tolist() == [0] and s.size == 0 and h.size == 0

    with api.BwtBuilder() as b:                                       # one strand only: unbalanced
        b.set_records(recs)
        b.build()
        b.sample_sa(32)
        rc, so, nh, sd, ht, msg = raw(b, reads)
        assert rc != 0 and "reverse complement" in msg and untouched(so, nh, sd, ht)
    with api.BwtBuilder() as b:                                       # balanced, but an odd number of records
        b.set_records(both + [b"ACGT" * 16])
        b.build()
        b.sample_sa(32)
        rc, so, nh, sd, ht, msg = raw(b, reads)
        assert rc != 0 and str(len(both) + 1) in msg and untouched(so, nh, sd, ht)
