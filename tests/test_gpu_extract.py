"""Extract and whole-text inversion (debwt_index_extract, BwtBuilder.extract / text / separators) through the C ABI, against
the text that was built, on loaded results that never saw the text, and on the error paths."""
import numpy as np
import pytest

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from oracle import coracle, stages as st
from tests.util import as_bytes_records, golden, seeded_records

pytestmark = pytest.mark.gpu

CASES = ["c4_like_5x100k", "c3_like_600k_3rec", "c2_like_1m"]


def _intervals(n, seps, rate, rng, k=2000):
    """k seeded intervals of up to 3 rates plus the edges: empty, [N-1, N), [N, N), [0, N), single symbols, across '#',
    inside one block"""
    a = rng.integers(0, n + 1, k)
    b = np.minimum(a + rng.integers(0, 3 * rate + 300, k), n)
    iv = list(zip(a.tolist(), b.tolist()))
    iv += [(0, 0), (n // 2, n // 2), (n - 1, n), (n, n), (0, n), (0, 1), (n - 2, n - 1), (n // 3, n // 3 + 1)]
    for s in np.asarray(seps)[:-1][:5].tolist():
        iv += [(s - 40, s + 41), (s, s + 1)]
    if rate >= 4:
        q = n // rate // 2
        iv += [(q * rate + 1, q * rate + 3), (q * rate, (q + 1) * rate)]
    return [int(x) for x, _ in iv], [int(y) for _, y in iv]


def _check_extract(b, text, starts, ends):
    upper = np.frombuffer(text.tobytes().upper(), dtype=np.uint8)
    offs, out = b.extract(starts, ends)
    assert offs.size == len(starts) + 1 and int(offs[0]) == 0 and out.size == int(offs[-1])
    for i, (a, e) in enumerate(zip(starts, ends)):
        assert int(offs[i + 1] - offs[i]) == e - a
        assert (out[int(offs[i]):int(offs[i + 1])] == upper[a:e]).all(), (i, a, e)


def _case(name):
    recs = as_bytes_records(seeded_records(name))
    text, seps = api.join_records(recs)
    return recs, text, seps


@pytest.mark.parametrize("name", CASES)
def test_extract_against_text(name):
    _, text, seps = _case(name)
    n = text.size
    rng = np.random.default_rng(17)
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        for rate in (1, 4, 32, 1024):
            b.sample_sa(rate)
            starts, ends = _intervals(n, seps, rate, rng)
            _check_extract(b, text, starts, ends)
            assert (b.text() == text).all(), rate
            assert (b.separators() == seps).all(), rate


def test_many_records():
    """1500 records of 33-120 bp: most blocks walk through '#' rows"""
    rng = np.random.default_rng(5)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    recs = [acgt[rng.integers(0, 4, int(rng.integers(33, 121)))] for _ in range(1500)]
    text, seps = api.join_records(recs)
    with api.BwtBuilder() as b:
        b.set_records(recs)
        b.build()
        for rate in (8, 128):
            b.sample_sa(rate)
            assert (b.text() == text).all(), rate
            assert (b.separators() == seps).all()
            starts, ends = _intervals(text.size, seps, rate, rng, k=500)
            _check_extract(b, text, starts, ends)


@pytest.mark.parametrize("kind", ["poly_a", "tandem", "copies"])
def test_degenerate_repeats(kind):
    rng = np.random.default_rng(3)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    if kind == "poly_a":
        recs = [np.full(90_000, ord("A"), np.uint8), np.concatenate([acgt[rng.integers(0, 4, 50)], np.full(70_000, ord("A"), np.uint8)])]
    elif kind == "tandem":
        unit = acgt[rng.integers(0, 4, 37)]
        recs = [np.tile(unit, 4000), np.tile(unit, 1500), np.concatenate([np.tile(unit, 100), unit[:7]])]
    else:
        a = acgt[rng.integers(0, 4, 120_000)]
        recs = [a, a.copy(), a[:60_000].copy(), a.copy()]
    text, seps = api.join_records(recs)
    with api.BwtBuilder() as b:
        b.set_records(recs)
        b.build()
        for rate in (1, 32):
            b.sample_sa(rate)
            assert (b.text() == text).all(), (kind, rate)
            assert (b.separators() == seps).all()


def test_lowercase_comes_back_upper():
    recs = [r.encode() for r in golden()["small"]["lowercase_mixed"]["records"]]
    assert any(c in b"acgt" for r in recs for c in r)
    text, seps = api.join_records(recs)
    with api.BwtBuilder() as b:
        b.set_records(recs)
        b.build()
        b.sample_sa(4)
        got = b.text()
    assert (got == np.frombuffer(text.tobytes().upper(), dtype=np.uint8)).all()
    assert not np.isin(got, np.frombuffer(b"acgt", dtype=np.uint8)).any()


_IUPAC = {"N": "ACGT", "V": "ACG", "D": "ATG", "B": "TCG", "H": "ATC", "W": "AT", "S": "CG", "K": "TG", "M": "AC", "Y": "CT", "R": "AG"}


def test_ambiguity_policy_text():
    rng = np.random.default_rng(9)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    recs = [acgt[rng.integers(0, 4, 50_000)], acgt[rng.integers(0, 4, 30_001)]]
    text, seps = api.join_records(recs)
    codes = np.frombuffer(b"NVDBHWSKMYRnvdbhwskmyr", dtype=np.uint8)
    hits = rng.choice(np.setdiff1d(np.arange(text.size), seps.astype(np.int64)), size=3000, replace=False)
    amb = text.copy()
    amb[hits] = codes[rng.integers(0, codes.size, size=hits.size)]
    got = {}
    for seed in (7, 7, 12345):
        with api.BwtBuilder() as b:
            b.set_ambiguity_policy(True, seed)
            b.set_text(amb, seps)
            b.build()
            b.sample_sa(16)
            t = b.text()
            keep = np.ones(text.size, dtype=bool)
            keep[hits] = False
            assert (t[keep] == text[keep]).all()                  # every A, C, G, T, '#' and '$' as given
            for p in hits.tolist():
                assert chr(t[p]) in _IUPAC[chr(amb[p]).upper()], (p, chr(amb[p]), chr(t[p]))
            assert b.verify(t)[0] == 0
            assert (t == st.resolve_ambiguity(amb, seed)).all()
            if seed in got:
                assert (t == got[seed]).all()                     # the same seed gives the same text
            got[seed] = t
    assert (got[7] != got[12345]).any()


def _loaded_check(words, sharp, dollar, text, seps, pos):
    with api.BwtBuilder() as c:
        c.set_result(words, text.size, sharp, dollar)
        c.sample_sa(16)
        assert (c.text() == text).all()
        s = c.separators()
        assert (s == seps).all()
        assert [x.tolist() for x in api.record_offsets(pos, s)] == [x.tolist() for x in api.record_offsets(pos, seps)]
        starts, ends = _intervals(text.size, seps, 16, np.random.default_rng(8), k=300)
        _check_extract(c, text, starts, ends)


def test_loaded_results(tmp_path):
    recs, text, seps = _case("c4_like_5x100k")
    sym, _ = st.text_from_records(recs)
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        words, sharp, dollar = b.result()
        b.sample_sa(32)
        _, pos = b.locate([text[1000:1012].tobytes(), text[250_000:250_008].tobytes(), b"ACGTA"])
    assert pos.size > 3
    _loaded_check(*coracle.bwt(sym), text, seps, pos)
    path = str(tmp_path / "c4.bwt")
    api.write_outputs(path, words, sharp, dollar)
    _loaded_check(*api.read_outputs(path, text.size), text, seps, pos)
    mw, ms, md, _ = api.build_multi(text, seps, [0, 0])
    _loaded_check(mw, ms, md, text, seps, pos)


def test_state_inverse_samples_follow_the_samples():
    _, text, seps = _case("c3_like_600k_3rec")
    _, other, oseps = _case("c4_like_5x100k")
    rng = np.random.default_rng(2)
    starts, ends = _intervals(text.size, seps, 64, rng, k=300)
    L = binding.lib()
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        b.sample_sa(4)
        _check_extract(b, text, starts, ends)
        b.sample_sa(64)                                           # new samples: stale inverse samples would decode garbage
        c0 = L.debwt_launch_count()
        _check_extract(b, text, starts, ends)
        c1 = L.debwt_launch_count()
        _check_extract(b, text, starts, ends)
        c2 = L.debwt_launch_count()
        assert 0 < c2 - c1 < c1 - c0                              # the second call reuses the inverse samples
        b.set_text(other, oseps)                                  # a new input of another text
        b.build()
        with pytest.raises(DebwtError, match="sample_sa"):
            b.text()
        b.sample_sa(64)
        assert (b.text() == other).all()
        assert (b.separators() == oseps).all()


def test_errors():
    recs = [r.upper().encode() for r in golden()["small"]["haplotypes_6x1500"]["records"]]
    text, seps = api.join_records(recs)
    n = text.size
    L = binding.lib()

    def raw(starts, ends, cap):
        s = np.ascontiguousarray(starts, dtype=np.uint64)
        e = np.ascontiguousarray(ends, dtype=np.uint64)
        out = np.full(max(cap, 1) + 16, 0xA5, dtype=np.uint8)
        rc = L.debwt_index_extract(b._h, api._ptr(s), api._ptr(e), s.size, api._ptr(out), cap)
        return rc, out, L.debwt_last_error().decode()

    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        rc, out, msg = raw([0], [10], 10)
        assert rc != 0 and "sample_sa" in msg and (out == 0xA5).all()
        b.sample_sa(8)
        rc, out, msg = raw([0, 5, 9], [4, 3, 20], 100)           # start > end
        assert rc != 0 and "interval 1" in msg and (out == 0xA5).all()
        rc, out, msg = raw([0, 0, 0, n - 3], [4, 3, 20, n + 1], 100)   # end > N
        assert rc != 0 and "interval 3" in msg and (out == 0xA5).all()
        rc, out, msg = raw([0, 100], [60, 200], 159)             # out too small: names the total
        assert rc != 0 and "160" in msg and (out == 0xA5).all()
        with pytest.raises(DebwtError, match="interval 0"):
            b.extract([n], [n + 1])
        rc, out, msg = raw([], [], 0)                             # no intervals
        assert rc == 0 and (out == 0xA5).all()
        offs, sym = b.extract([], [])
        assert offs.tolist() == [0] and sym.size == 0
        rc, out, msg = raw([0, 100], [60, 200], 160)
        assert rc == 0 and (out[:160] == np.concatenate([text[:60], text[100:200]])).all() and (out[160:] == 0xA5).all()
