"""The CPU pieces of the switch-point tests (tests/switch_points.py) against their slow definitions, and the placement of
every switch-point input on its side of its threshold.  No GPU needed."""
import ctypes

import numpy as np
import pytest

from debwt_b200 import binding
from oracle import coracle, stages as st
from tests import switch_points as sw
from tests.util import golden

G = golden()


@pytest.mark.parametrize("kind", ["random", "tie_heavy", "separators", "homopolymer"])
def test_suffix_ranks_match_string_sort(kind):
    rng = np.random.default_rng(len(kind))
    if kind == "random":
        codes = rng.integers(0, 4, size=600)
    elif kind == "tie_heavy":
        codes = np.tile(rng.integers(0, 4, size=13), 50)
        codes[rng.integers(0, codes.size, size=4)] ^= 1
    elif kind == "separators":
        codes = rng.integers(0, 4, size=500)
        codes[rng.integers(0, codes.size, size=40)] = 4
    else:
        codes = np.zeros(400, dtype=np.int64)
    codes = np.concatenate([codes, [5]]).astype(np.uint8)
    b = bytes(codes.tolist())
    want = sorted(range(codes.size), key=lambda i: b[i:])
    assert np.argsort(sw.suffix_ranks(codes)).tolist() == want


def test_doubling_bwt_matches_oracles():
    for recs in (["A" * 300, "AC" * 40], ["ACGTTGCA" * 20, "T" * 90, "ACGTTGCA" * 19 + "A"],
                 G["small"]["haplotypes_6x1500"]["records"][:2]):
        sym, _ = st.text_from_records(recs)
        got = sw.doubling_bwt(sym)
        for want in (coracle.bwt(sym), st.suffix_sort_bwt(recs)):
            assert all((x == y).all() for x, y in zip(got, want))


def test_k10_reference_matches_string_sort():
    rng = np.random.default_rng(3)
    codes = np.tile(rng.integers(0, 4, size=7), 80).astype(np.uint8)
    codes[rng.integers(0, codes.size, size=10)] = 4
    codes = np.concatenate([codes, [5]]).astype(np.uint8)
    sizes = [1, 2, 5, 40, 100]
    offs = np.concatenate(([0], np.cumsum(sizes))).astype(np.uint64)
    spi = np.concatenate([rng.choice(codes.size - 1, size=s, replace=False) for s in sizes]).astype(np.uint64)
    prev = rng.integers(0, 5, size=spi.size).astype(np.uint8)
    got = sw.k10_expected_prev(codes, offs, spi, prev)
    b = bytes(codes.tolist())
    for s in range(len(sizes)):
        lo, hi = int(offs[s]), int(offs[s + 1])
        ent = sorted(zip(spi[lo:hi].tolist(), prev[lo:hi].tolist()), key=lambda e: b[e[0]:])
        assert got[lo:hi].tolist() == [p for _, p in ent]


def test_k10_case_covers_every_bin_edge():
    codes, offs, spi, prev = sw.k10_case()
    sizes = np.diff(offs.astype(np.int64)).tolist()
    assert sizes == sw.K10_SIZES and codes[-1] == 5 and (codes[:-1] != 5).all()
    for edge in (sw.K10_WARP, sw.K10_MID, sw.K10_TINY, sw.K10_SMEM):
        assert {edge - 1, edge, edge + 1} <= set(sizes)
    sep = np.flatnonzero(codes == 4)
    for s, size in enumerate(sizes):
        lo, hi = int(offs[s]), int(offs[s + 1])
        assert np.unique(spi[lo:hi]).size == size
        if size >= 31:                                   # some entries meet a '#' within their first 27 codes
            p = spi[lo:hi].astype(np.int64)
            nxt = sep[np.minimum(np.searchsorted(sep, p), sep.size - 1)]
            assert ((nxt >= p) & (nxt - p < 27)).any(), size


def _slow_counts(records):
    """the build's counts from st.build_bwt's intermediate products, counted per k-mer and per window in plain Python"""
    sym, seps = st.text_from_records(records)
    sk = st.sort_keys(st.extract_keys(sym, seps))
    gmask, _ = st.group_masks(sk, sym, seps)
    specials = st.special_suffixes(sym, seps, sk)
    sp, _ = st.branch_codes(sym, seps, sk, gmask, specials)
    per_kmer = {}
    for key, m in zip(sk.tolist(), gmask.tolist()):
        per_kmer.setdefault(key >> 2, []).append(m)
    n_branch = sum(1 for ms in per_kmer.values() if st.multi_in(ms[0]) or st.multi_out(ms[0]))
    n_blue = sum(len(ms) for ms in per_kmer.values() if st.multi_in(ms[0]))
    emit = {e["pos"] for e in specials if e["emit"]}
    start = 0
    for s in seps.tolist():
        for p in range(start, s - 31):
            if st.multi_out(per_kmer[st._kmer31(sym, p).item()][0]):
                emit.add(p)
        start = s + 1
    assert len(emit) == sp.size
    return {"n_keys": sk.size, "n_branch": n_branch, "n_blue": n_blue, "n_codes": len(emit), "n_special": 32 * seps.size}


@pytest.mark.parametrize("name", ["haplotypes_6x1500", "pathological", "planted_repeats", "survey_golden"])
def test_stats_helper_matches_slow_counts(name):
    recs = G["small"][name]["records"]
    rs = sw.Restated(recs)
    assert rs.stats() == _slow_counts(recs)
    assert rs.stats()["n_blue"] == int(rs.mi.sum())
    assert sw.Restated(recs, specials=False).stats() == {k: v for k, v in rs.stats().items() if k != "n_codes"}


def test_branch_table_helper():
    rs = sw.Restated(G["small"]["planted_repeats"]["records"], specials=False)
    ent, head = rs.branch_table()
    assert ent.size == rs.stats()["n_branch"] and (np.diff(ent.astype(np.float64)) > 0).all()
    for e, h in zip(ent.tolist(), head.tolist()):
        assert rs.ghead[h] and (int(rs.sk[h]) >> 2) == (e >> 2)
        assert (e >> 1) & 1 == int(rs.mi[h]) and e & 1 == int(rs.mo[h])


def test_threshold_mirrors():
    L = binding.lib()
    for n in (1, 2048, 2049, 8191, 8193, 32767, 32769, 3 << 30, 4_000_000_000):
        assert L.debwt_dev_key_index_bits(ctypes.c_uint64(n)) == sw.key_index_bits(n), n
    assert sw.text_hist_applies(2048 * 3, 3) and not sw.text_hist_applies(2048 * 3 - 1, 3)
    rng = np.random.default_rng(1)
    keys = rng.integers(0, 2**56, size=1000, dtype=np.uint64)
    assert sw.sort_sweeps(keys) == 7 and sw.last_pass_skipped(keys)
    assert sw.sort_sweeps(keys | np.uint64(1 << 63)) == 7 and sw.sort_sweeps(np.full(9, 5, dtype=np.uint64)) == 0
    assert sw.k9_one_record_tiles([4094, 9000], 9001).tolist() == [False, True, True]
    assert sw.k9_one_record_tiles([4095, 9000], 9001).tolist() == [True, True, True]
    assert sw.k9_one_record_tiles([4096, 9000], 9001).tolist() == [True, False, True]


def test_edge_runs_definition():
    """edge_runs against a per-source loop on a small input"""
    rs = sw.Restated(G["small"]["planted_repeats"]["records"], specials=False)
    sk = rs.sk
    runs = sw.edge_runs(sk)
    assert sum(e - b for _, _, b, e, _ in runs) == sk.size
    for c, t, b, e, marks in runs:
        for i in range(b, e):
            q = (int(sk[i]) << 2) & ((1 << 64) - 1)
            lb = int(np.searchsorted(sk, np.uint64(q)))
            assert int(sk[i]) >> 62 == c and lb // sw.ME_TILE == t
        assert marks == 0                                   # no run of this input is longer than ME_CAP


@pytest.mark.parametrize("name", [pytest.param(n, marks=pytest.mark.slow) if c.slow else n for n, c in sw.CASES.items()])
def test_case_lies_on_its_side(name):
    case = sw.CASES[name]
    case.place(sw.Restated(case.make(), specials=False))
