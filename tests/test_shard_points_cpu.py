"""The per-rank restatement of the sharded build (tests/shard_points.py) against slow definitions, the host twins in
debwt_b200/dist.py and the library's slice geometry, and the placement of every shard-point input on its side of its edge.
No GPU needed."""
import ctypes
import functools

import numpy as np
import pytest

from debwt_b200 import binding, dist
from oracle import stages as st
from tests import shard_points as sp


@functools.lru_cache(maxsize=None)
def _restated(name):
    c = sp.CASES[name]
    return sp.Restated(c.make(), doubling=c.doubling)


def _case_worlds():
    return [pytest.param(n, G, id=f"{n}-g{G}") for n, c in sp.CASES.items() for G in c.worlds]


def test_windows_before_matches_dist_and_positions():
    for name in ("n417", "sep_edges_g5", "codes_shared", "sample_4097"):
        rs = _restated(name)
        xs = range(rs.n + 40) if rs.n < 6000 else list(range(0, rs.n + 40, 7)) + rs.seps.tolist()
        for x in xs:
            want = int((rs.ppos < x).sum())
            assert sp.windows_before(x, rs.seps) == dist.valid_windows_before(x, rs.seps) == want, (name, x)


def test_slice_geometry_matches_dist_and_library():
    L = binding.lib()
    lo, hi = ctypes.c_uint64(), ctypes.c_uint64()
    for n in (34, 100, 417, 448, 449, 480, 1216, 4066, 60736, 10**6 + 3):
        for G in range(1, sp.MAX_RANKS + 1):
            wp = sp.words_per_slice(n, G)
            assert (wp, wp * G) == dist.slice_geometry(n, G)
            for r in range(G):
                assert L.debwt_shard_slice(r, G, ctypes.c_uint64(n), ctypes.byref(lo), ctypes.byref(hi)) == 0
                a, b = 32 * r * wp, max(min(32 * (r + 1) * wp, n), 32 * r * wp)
                assert (lo.value, hi.value) == (min(a, n), max(min(b, n), min(a, n))), (n, G, r)
            assert 32 * wp * G >= n + 32                       # the slices cover T and its 32 symbols of padding
    assert sp.n_for_wp(2, 128) == 8128 and sp.words_per_slice(8129, 2) == 129


def test_splitters_match_dist():
    rng = np.random.default_rng(5)
    for m in (0, 1, 2, 15, 16, 17, 4096, 12289):
        valid = np.sort(rng.integers(0, 2**63, size=m, dtype=np.uint64) | (rng.integers(0, 2, size=m, dtype=np.uint64) << np.uint64(63)))
        for G in range(1, sp.MAX_RANKS + 1):
            assert (sp.splitters_of(valid, G) == dist.choose_splitters(valid, G)).all(), (m, G)


def test_exchange_stride_is_a_permutation():
    for grid in range(1, 65):
        s = sp.exchange_stride(grid)
        assert sorted((b * s) % grid for b in range(grid)) == list(range(grid)), grid
        assert s % 2 == 1 and (grid >= sp.STRIDE_MIN_GRID or s == 1)
    assert {t: sp.exchange_stride(t) for t in sp.GRID_STRIDES} == sp.GRID_STRIDES
    assert int(15 * sp.GOLDEN) | 1 == 9 and sp.exchange_stride(15) == 7              # the gcd loop lowers 9 to 7


def _slow_emit(rs):
    """code-emitting positions, one position at a time: in-record windows whose k-mer is multi-out, and sentinel windows
    whose flag is set"""
    mask_of = {}
    for key, m in zip(rs.sk.tolist(), rs.gmask.tolist()):
        mask_of.setdefault(key >> 2, m)
    emit = {e["pos"] for e in rs.spec if e["emit"]}
    start = 0
    for s in rs.seps.tolist():
        for p in range(start, s - 31):
            if st.multi_out(mask_of[st._kmer31(rs.sym, p).item()]):
                emit.add(p)
        start = s + 1
    return emit


@pytest.mark.parametrize("name,G", _case_worlds())
def test_rank_restatement_matches_slow_definitions(name, G):
    rs = _restated(name)
    rk = rs.ranks(G)
    assert [lo for lo in rk.pos_lo] == [32 * r * rk.wp for r in range(G)]
    # samples: ns keys of the slice in position order, every stride-th
    for r in range(G):
        keys = [int(k) for p, k in zip(rs.ppos.tolist(), rs.keys.tolist()) if rk.pos_lo[r] <= p < rk.pos_hi[r]]
        assert len(keys) == rk.cnt[r]
        ns = min(len(keys), sp.SAMPLES_PER_RANK)
        stride = max(len(keys) // ns, 1) if ns else 1
        assert rk.samples[r].tolist() == [keys[i * stride] for i in range(ns)]
    # owners by a linear scan over the splitters
    spl = [int(s) for s in rk.splitters]
    assert spl == sorted(spl) and len(spl) == G - 1
    own = [sum(1 for s in spl if s <= (k & sp.KMER_MASK)) for k in rs.keys.tolist()]
    assert np.bincount(own, minlength=G).tolist() == rk.n_keys_local
    assert sum(rk.n_keys_local) == rs.sk.size
    for r in range(G):
        mine = sorted(k for k, o in zip(rs.keys.tolist(), own) if o == r)
        assert rk.owned[r].tolist() == mine
    # row ranges: a key's row goes to its owner, a sentinel suffix's row to the owner of the key before it
    ins = rs.ins
    owner_of_row = np.full(rs.n, -1)
    for i in range(rs.sk.size):
        owner_of_row[i + int(np.searchsorted(ins, i, side="right"))] = rk.rank_of_key(int(rs.sk[i]))
    for t, v in enumerate(ins.tolist()):
        owner_of_row[v + t] = rk.rank_of_key(int(rs.sk[max(v - 1, 0)]))
    assert (owner_of_row >= 0).all()
    for r in range(G):
        rows = np.flatnonzero(owner_of_row == r)
        assert rows.tolist() == list(range(rk.r_lo[r], rk.r_lo[r + 1])), r
    assert rk.r_lo[0] == 0 and rk.r_lo[G] == rs.n
    # code bases by a position-by-position count
    emit = _slow_emit(rs)
    assert len(emit) == rs.sp.size == sum(rk.s_loc)
    for r in range(G):
        assert rk.code_base[r] == sum(1 for p in emit if p < rk.pos_lo[r])
    assert rk.dollar_index == sum(1 for p in emit if p < int(rs.seps[-1]) - 31)
    # exchange grid
    assert rk.grid == [-(-c // 2048) for c in rk.cnt]


@pytest.mark.parametrize("name", sp.CASES)
def test_case_lies_on_its_side(name):
    sp.CASES[name].place(_restated(name))


def test_worlds_cover_1_to_16():
    assert set().union(*(c.worlds for c in sp.CASES.values())) == set(range(1, sp.MAX_RANKS + 1))
