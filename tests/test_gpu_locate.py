"""Sampled suffix array and locate (debwt_index_sample_sa / _sa / _locate) and loading a finished result into a context
(debwt_set_result), through the C ABI, against the oracle's BWT inverted on the CPU (tests/locate_ref.py) and a plain
scan of the text."""
import numpy as np
import pytest

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from oracle import coracle, stages as st
from tests.locate_ref import suffix_array
from tests.util import as_bytes_records, golden, seeded_records

pytestmark = pytest.mark.gpu

CASES = ["c4_like_5x100k", "c3_like_600k_3rec", "c2_like_1m"]


def _find_all(raw, p):
    out, i = [], raw.find(p)
    while i >= 0:
        out.append(i)
        i = raw.find(p, i + 1)
    return out


def _patterns(raw, n, seed=3):
    """the mix of test_gpu_index.py plus lowercase, a pattern with 'N' and the empty pattern"""
    rng = np.random.default_rng(seed)
    pats = []
    for L in (1, 2, 5, 12, 31, 32, 33, 64, 200):
        for _ in range(6):
            o = int(rng.integers(0, n - L - 1))
            p = raw[o:o + L]
            if b"#" in p or b"$" in p:
                continue
            pats.append(p)
            q = bytearray(p)
            q[int(rng.integers(0, L))] = b"ACGT"[int(rng.integers(0, 4))]
            pats.append(bytes(q))
            pats.append(p.lower())
    pats.append(b"ACGT" * 40)
    o = int(rng.integers(0, n - 40))
    pats.append(raw[o:o + 10] + b"N" + raw[o + 11:o + 20])
    pats.append(b"")
    return pats


def _check_locate(b, raw, sa, pats):
    n = sa.size
    isa = np.empty(n, dtype=np.int64)
    isa[sa.astype(np.int64)] = np.arange(n)
    hits, pos = b.locate(pats)
    counts = b.count(pats)
    assert hits.size == len(pats) + 1 and int(hits[0]) == 0
    assert (np.diff(hits.astype(np.int64)) == counts.astype(np.int64)).all()
    assert pos.size == int(hits[-1])
    for i, p in enumerate(pats):
        got = pos[int(hits[i]):int(hits[i + 1])]
        if p == b"":
            assert (got == sa).all()
            continue
        want = _find_all(raw, p.upper()) if b"N" not in p.upper() else []
        assert sorted(got.tolist()) == want, p
        if got.size:                                            # SA order: the rows [sp, ep) of the pattern, ascending
            rows = isa[got.astype(np.int64)]
            assert (rows == np.arange(rows[0], rows[0] + rows.size)).all(), p
            assert (got == sa[rows[0]:rows[0] + rows.size]).all()
    return hits, pos


def _case(name):
    recs = as_bytes_records(seeded_records(name))
    text, seps = api.join_records(recs)
    sym, _ = st.text_from_records(recs)
    return recs, text, seps, sym


@pytest.mark.parametrize("name", CASES)
def test_sa_exact_every_rate(name):
    _, text, seps, sym = _case(name)
    sa = suffix_array(sym)
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        for rate in (1, 4, 32, 1024):
            ms = b.sample_sa(rate)
            assert ms > 0
            assert (b.sa(np.arange(text.size, dtype=np.uint64)) == sa).all(), rate


@pytest.mark.parametrize("name", CASES)
def test_locate_against_oracle_and_text(name):
    _, text, seps, sym = _case(name)
    sa = suffix_array(sym)
    raw = text.tobytes()
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        for rate in (4, 32):
            b.sample_sa(rate)
            _check_locate(b, raw, sa, _patterns(raw, text.size))


@pytest.mark.parametrize("kind", ["poly_a", "tandem", "two_copies"])
def test_locate_degenerate_repeats(kind):
    rng = np.random.default_rng(3)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    if kind == "poly_a":
        recs = [np.concatenate([np.full(90_000, ord("A"), np.uint8), acgt[rng.integers(0, 4, 3000)]]),
                np.concatenate([acgt[rng.integers(0, 4, 2000)], np.full(70_000, ord("A"), np.uint8), acgt[rng.integers(0, 4, 50)]])]
        pats = [b"A" * 20, b"A" * 1000, b"A" * 12 + b"C"]
    elif kind == "tandem":
        unit = acgt[rng.integers(0, 4, 37)]
        recs = [np.concatenate([np.tile(unit, 4000), acgt[rng.integers(0, 4, 500)]]), np.tile(unit, 1500)]
        pats = [unit[:30].tobytes(), np.tile(unit, 3).tobytes(), unit[:5].tobytes()]
    else:
        a = acgt[rng.integers(0, 4, 120_000)]
        recs = [a, a.copy(), a[:60_000].copy()]
        pats = [a[1000:1100].tobytes(), a[70_000:70_040].tobytes(), a[:3].tobytes()]
    text, seps = api.join_records(recs)
    raw = text.tobytes()
    with api.BwtBuilder() as b:
        b.set_records(recs)
        b.build()
        b.sample_sa(32)
        hits, pos = b.locate(pats)
        for i, p in enumerate(pats):
            got = pos[int(hits[i]):int(hits[i + 1])]
            assert sorted(got.tolist()) == _find_all(raw, p), (kind, i)
    if kind == "poly_a":
        assert int(hits[1] - hits[0]) > 100_000 and int(hits[2] - hits[1]) > 100_000


def _loaded_equals(b_ref, words, sharp, dollar, text, pats, sa):
    n = text.size
    with api.BwtBuilder() as c:
        c.set_result(words, n, sharp, dollar)
        w, s, d = c.result()
        assert (w == words).all() and (s == np.sort(sharp)).all() and int(d[0]) == int(np.asarray(dollar).reshape(-1)[0])
        assert c.verify(text)[0] == 0
        assert (c.count(pats) == b_ref.count(pats)).all()
        c.sample_sa(16)
        assert (c.sa(np.arange(n, dtype=np.uint64)) == sa).all()
        h1, p1 = c.locate(pats)
        h0, p0 = b_ref.locate(pats)
        assert (h1 == h0).all() and (p1 == p0).all()
        with pytest.raises(DebwtError, match="loaded result"):
            c.build()


def test_loaded_results_oracle_files_multi(tmp_path):
    _, text, seps, sym = _case("c4_like_5x100k")
    raw = text.tobytes()
    pats = _patterns(raw, text.size, seed=5)
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        words, sharp, dollar = b.result()
        b.sample_sa(16)
        sa = b.sa(np.arange(text.size, dtype=np.uint64))
        assert (sa == suffix_array(sym)).all()
        # the oracle's own BWT: independent of the CUDA build
        ow, os_, od = coracle.bwt(sym)
        _loaded_equals(b, ow, os_, od, text, pats, sa)
        # the three files written by write_outputs
        path = str(tmp_path / "c4.bwt")
        api.write_outputs(path, words, sharp, dollar)
        _loaded_equals(b, *api.read_outputs(path, text.size), text, pats, sa)
        # the sharded build, two threads on one GPU
        mw, ms, md, _ = api.build_multi(text, seps, [0, 0])
        _loaded_equals(b, mw, ms, md, text, pats, sa)


def _lf_is_one_cycle(codes):
    n = codes.size
    lf = np.empty(n, dtype=np.int64)
    lf[np.argsort(codes, kind="stable")] = np.arange(n)
    r, steps = n - 1, 0
    while True:
        r = int(lf[r])
        steps += 1
        if r == n - 1:
            return steps == n


def test_errors():
    recs = [r.upper().encode() for r in golden()["small"]["haplotypes_6x1500"]["records"]]
    text, seps = api.join_records(recs)
    n = text.size
    L = binding.lib()
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        words, sharp, dollar = b.result()
        assert sharp.size >= 2
        with pytest.raises(DebwtError, match="sample_sa"):
            b.sa([0])
        with pytest.raises(DebwtError, match="sample_sa"):
            b.locate([b"ACG"])
        for rate in (0, 3, 2048):
            with pytest.raises(DebwtError, match="power of two"):
                b.sample_sa(rate)
        b.sample_sa(8)
        with pytest.raises(DebwtError, match="not below N"):
            b.sa([0, n])
        # positions_cap too small: the message names the number of hits
        blob = np.frombuffer(b"A\0", dtype=np.uint8)
        offs = np.array([0, 1], dtype=np.uint64)
        hits = np.zeros(2, dtype=np.uint64)
        assert L.debwt_index_locate(b._h, api._ptr(blob), api._ptr(offs), 1, api._ptr(hits), None, 0) == 0
        total = int(hits[1])
        assert total > 1
        pos = np.zeros(total, dtype=np.uint64)
        assert L.debwt_index_locate(b._h, api._ptr(blob), api._ptr(offs), 1, api._ptr(hits), api._ptr(pos), total - 1) != 0
        assert str(total) in L.debwt_last_error().decode()
        # a new input and build drop the samples
        b.set_text(text, seps)
        b.build()
        with pytest.raises(DebwtError, match="sample_sa"):
            b.sa([0])
        b.sample_sa(8)
        assert b.sa([int(dollar[0])])[0] == 0

    with api.BwtBuilder() as c:
        with pytest.raises(DebwtError, match="'\\$' row"):
            c.set_result(words, n, sharp, [n])
        dup = sharp.copy()
        dup[1] = dup[0]
        with pytest.raises(DebwtError, match="twice"):
            c.set_result(words, n, dup, dollar)
        clash = sharp.copy()
        clash[0] = dollar[0]
        with pytest.raises(DebwtError, match="also listed"):
            c.set_result(words, n, clash, dollar)
        high = sharp.copy()
        high[0] = n
        with pytest.raises(DebwtError, match="not below"):
            c.set_result(words, n, high, dollar)
        with pytest.raises(DebwtError, match="words"):                # a word count that does not fit N
            c.set_result(words, n + 64, sharp, dollar)
        with pytest.raises(DebwtError):                               # nothing loaded after a refused result
            c.result()
        with pytest.raises(DebwtError, match="no input"):
            c.build()

        # not a BWT: two base symbols of a valid one swapped (counts still add up), found by the sampler
        codes = coracle.unpack_bwt(words, n, sharp, dollar)
        rng = np.random.default_rng(1)
        while True:
            i, j = (int(x) for x in rng.integers(0, n, 2))
            if codes[i] < 4 and codes[j] < 4 and codes[i] != codes[j]:
                bad = codes.copy()
                bad[i], bad[j] = codes[j], codes[i]
                if not _lf_is_one_cycle(bad):
                    break
        bw, bs, bd = coracle.pack_bwt(bad)
        c.set_result(bw, n, bs, bd)
        assert int(c.count([b""])[0]) == n                          # counting works on any array
        with pytest.raises(DebwtError, match="not a BWT"):
            c.sample_sa(4)
        with pytest.raises(DebwtError, match="sample_sa"):
            c.sa([0])
        assert c.verify(text)[0] > 0
