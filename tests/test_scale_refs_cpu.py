"""The host references of tests/test_gpu_scale.py (occ recount from the packed words, BWT symbol lookup, LF walks, SA row
checks) against the oracle's BWT and suffix array of a small multi-record text, so that a pass at scale means the library
agrees with a reference that is itself right."""
import numpy as np

from debwt_b200 import api, synth
from oracle import coracle, stages as st
from tests import test_gpu_scale as S
from tests.locate_ref import suffix_array


def _case():
    base = synth.config2(120_000, 3_000, 3, 0.1)[0]
    recs = [base, synth._mutate(base, 7, 0.01), synth.random_bases(5, 30_001)] + [synth.random_bases(9 + i, 1550) for i in range(40)]
    recs = [bytes(r) for r in recs]
    text, seps = api.join_records(recs)
    sym, _ = st.text_from_records(recs)
    words, sharp, dollar = coracle.bwt(sym)
    return text, seps, sym, words, np.sort(sharp.astype(np.int64)), int(dollar[0])


def test_host_references_match_the_oracle():
    text, seps, sym, words, sharp, dollar = _case()
    n, R = sym.size, seps.size
    assert (S._LUT[text] == sym).all()
    codes = coracle.unpack_bwt(words, n, sharp.astype(np.uint64), np.array([dollar], dtype=np.uint64))
    assert (S.bwt_at(words, sharp, dollar, np.arange(n)) == codes).all()

    occ = S.host_occ(words, n, sharp, dollar)
    w = np.minimum(np.arange(occ.shape[0]) * 32, n)
    for c in range(4):
        assert (occ[:, c] == np.concatenate([[0], np.cumsum(codes == c)])[w]).all()
    C = S.c_array(occ, n, R)
    assert C[4] == n - R and C[5] == n - 1

    sa = suffix_array(sym).astype(np.int64)
    lf = S.HostLF(words, occ, C, sharp, dollar)
    assert lf.walk(sym, dollar, 0, n) == (dollar, 0)             # LF is one N-cycle from the '$' row
    for i in range(0, R, 7):
        r, p = lf.walk(sym, n - R + i, int(sa[n - R + i]), 2_000)
        assert sa[r] == p

    class SA:
        def sa(self, rows):
            return sa[np.asarray(rows, dtype=np.int64)].astype(np.uint64)

    rows = S.sa_probe_rows(n, sharp, np.random.default_rng(1))
    q, got = S.check_sa_rows(SA(), words, sharp, dollar, sym, rows)
    assert (got == sa[q]).all()
    # the references catch a wrong SA value: two neighbouring rows swapped
    bad = sa.copy()
    bad[[100, 101]] = bad[[101, 100]]

    class BadSA:
        def sa(self, rows):
            return bad[np.asarray(rows, dtype=np.int64)].astype(np.uint64)

    try:
        S.check_sa_rows(BadSA(), words, sharp, dollar, sym, np.array([100]))
    except AssertionError:
        pass
    else:
        raise AssertionError("check_sa_rows accepted swapped SA values")
