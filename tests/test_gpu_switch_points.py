"""The production K3-K10 path at the thresholds where its kernels switch paths (inputs and placements in
tests/switch_points.py), against the stage restatement of oracle/stages.py.

A BWT comparison alone cannot see a k-mer wrongly marked multi-in or multi-out: such a k-mer only adds a blue segment
whose entries share their previous symbol, or a code to every branch-code string through it, and the BWT stays right.
So every case compares the masks, the branch table, the branch codes and blue entries and the build's counts as well."""
import ctypes

import numpy as np
import pytest

from debwt_b200 import api, binding
from tests import switch_points as sw

pytestmark = pytest.mark.gpu


def _params():
    return [pytest.param(n, marks=pytest.mark.slow) if c.slow else n for n, c in sw.CASES.items()]


@pytest.mark.parametrize("name", _params())
def test_switch_point_matches_restatement(name):
    case = sw.CASES[name]
    recs = case.make()
    rs = sw.Restated(recs, specials=case.codes)
    case.place(rs)
    text, seps = api.join_records(recs)
    if case.bits is not None:
        assert binding.lib().debwt_dev_key_index_bits(ctypes.c_uint64(rs.sk.size)) == case.bits

    # the whole build, with both ways of grouping the blue entries: BWT, counts, sort path
    want = rs.stats()
    sweeps = sw.sort_sweeps(rs.sk)
    hist_launches = 2 if sw.text_hist_applies(rs.n, rs.R) else 1      # text_hist + fix kernels, or the key histogram
    ref = rs.bwt(case.doubling)
    for mode in (1, 2):
        with api.BwtBuilder(blue_grouping=mode) as b:
            b.set_text(text, seps)
            b.build()
            got = b.result()
            s = b.stats()
        assert all((x == y).all() for x, y in zip(ref, got)), mode
        assert {k: s[k] for k in want} == want, mode
        assert s["sort_sweeps"] == sweeps and s["sort_launches"] == hist_launches + 1 + sweeps, mode

    # K5-K7: masks as the build leaves them, and the branch table built from them
    masks = api.k_group_masks(text, seps)
    bad = np.flatnonzero(masks != rs.gmask)
    assert bad.size == 0, (bad[:8], masks[bad[:8]], rs.gmask[bad[:8]])
    ent, head = api.k_branch_kmers(text, seps)
    want_ent, want_head = rs.branch_table()
    assert ent.size == want_ent.size and (ent == want_ent).all() and (head == want_head).all()

    # K9: codes and blue entries
    if case.codes:
        codes, bhead, spi, prev = api.k_codes(text, seps)
        assert codes.size == rs.sp.size and (codes == rs.sp).all()
        assert sorted(zip(bhead.tolist(), spi.tolist(), prev.tolist())) == sorted(rs.blue)


@pytest.mark.parametrize("seed", [41, 42])
def test_k10_bins_match_suffix_ranks(seed):
    """one segment of every size at and around each K10 bin edge, tie-heavy code strings, '#' codes within the first 27
    codes of some entries"""
    codes, offs, spi, prev = sw.k10_case(seed)
    sizes = np.diff(offs.astype(np.int64))
    for edge in (sw.K10_WARP, sw.K10_MID, sw.K10_TINY, sw.K10_SMEM):
        assert {edge - 1, edge, edge + 1} <= set(sizes.tolist())
    got_spi, got_prev = api.k_sort_blue(codes, offs, spi, prev)
    for s in range(sizes.size):
        lo, hi = int(offs[s]), int(offs[s + 1])
        assert sorted(got_spi[lo:hi].tolist()) == sorted(spi[lo:hi].tolist()), sizes[s]
    want = sw.k10_expected_prev(codes, offs, spi, prev)
    for s in range(sizes.size):
        lo, hi = int(offs[s]), int(offs[s + 1])
        assert (got_prev[lo:hi] == want[lo:hi]).all(), sizes[s]
