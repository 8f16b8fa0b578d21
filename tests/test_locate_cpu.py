"""CPU side of locate: the reference suffix array of the locate tests (tests/locate_ref.py) against a plain sort under the
reference's suffix order, mapping text positions to record coordinates, and reading the three output files back."""
import functools

import numpy as np
import pytest

from debwt_b200 import api
from debwt_b200.binding import DebwtError
from oracle import coracle, stages as st
from tests.locate_ref import suffix_array
from tests.util import golden


def _plain_sa(sym):
    return np.array(sorted(range(sym.size), key=functools.cmp_to_key(
        lambda a, b: -1 if st.suffix_less(sym, a, b) else (1 if st.suffix_less(sym, b, a) else 0))), dtype=np.uint64)


def _random_texts():
    rng = np.random.default_rng(11)
    acgt = "ACGT"
    out = []
    for n_rec in (1, 2, 4):
        recs = ["".join(acgt[i] for i in rng.integers(0, 4, int(rng.integers(33, 200)))) for _ in range(n_rec)]
        out.append(recs)
    unit = "ACGTTGCA"
    out.append([unit * 9, unit * 9, unit * 5 + "A"])          # equal records: ties compared through the '#'
    out.append(["A" * 60, "A" * 45, "C" + "A" * 40])
    return out


@pytest.mark.parametrize("name", sorted(golden()["small"]))
def test_reference_suffix_array_small_golden(name):
    recs = [r.upper().encode() for r in golden()["small"][name]["records"]]
    sym, _ = st.text_from_records(recs)
    sa = suffix_array(sym)
    assert (sa == _plain_sa(sym)).all()
    # consistent with the oracle's BWT: BWT[r] = T[SA[r] - 1]
    assert (coracle.bwt_symbols(sym) == sym[(sa.astype(np.int64) - 1) % sym.size]).all()


@pytest.mark.parametrize("i", range(len(_random_texts())))
def test_reference_suffix_array_random_multirecord(i):
    sym, _ = st.text_from_records(_random_texts()[i])
    sa = suffix_array(sym)
    assert (sa == _plain_sa(sym)).all()
    assert int(sa[-1]) == sym.size - 1                       # "$" is the largest suffix


def test_record_offsets_hand_made():
    # T = ACGT...(40) # TTTT...(36) # GGG...(50) $ : seps 40, 77, 128
    seps = np.array([40, 77, 128], dtype=np.uint64)
    pos = np.array([0, 39, 40, 41, 76, 77, 78, 127, 128], dtype=np.uint64)
    rec, off = api.record_offsets(pos, seps)
    assert rec.tolist() == [0, 0, 0, 1, 1, 1, 2, 2, 2]
    assert off.tolist() == [0, 39, 40, 0, 35, 36, 0, 49, 50]
    rec, off = api.record_offsets(np.array([], dtype=np.uint64), seps)
    assert rec.size == 0 and off.size == 0
    with pytest.raises(ValueError):
        api.record_offsets([129], seps)
    # against join_records on real records
    recs = ["ACGT" * 10, "T" * 36, "G" * 50]
    text, s2 = api.join_records(recs)
    assert (s2 == seps).all()
    for p in range(text.size):
        r, o = api.record_offsets([p], s2)
        if text[p] not in (ord("#"), ord("$")):
            assert recs[int(r[0])][int(o[0])] == chr(text[p])


@pytest.mark.parametrize("n", [1000, 1024, 33 + 1])
def test_write_read_outputs_round_trip(tmp_path, n):
    rng = np.random.default_rng(n)
    words = rng.integers(0, 2**63, (n + 31) // 32, dtype=np.uint64)
    sharp = np.array(sorted(rng.choice(n - 1, 3, replace=False)), dtype=np.uint64)
    dollar = np.array([n - 1], dtype=np.uint64)
    path = str(tmp_path / "out.bwt")
    api.write_outputs(path, words, sharp, dollar)
    w, s, d = api.read_outputs(path, n)
    assert (w == words).all() and (s == sharp).all() and (d == dollar).all()
    assert w.dtype == np.uint64 and s.dtype == np.uint64
    with pytest.raises(DebwtError):
        api.read_outputs(path, n + 32)
