"""CPU side of BWA-MEM seed chaining: the restatement of tests/chain_ref.py checked against definitions (weights are
set-union lengths, consecutive chain seeds satisfy bwa's merge test, every hit that is no chain seed was contained in
the chain it was tested against), a model of the device's slot bitmap against a linear scan, hand-built hit lists for
every rule, api.bwa_rbeg against bwa's forward-reverse text, and the CHAIN_DTYPE / CHAIN_SEED_DTYPE / ChainOpts
mirrors of include/debwt_b200.h against a C compiler."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from debwt_b200 import api, binding
from tests import chain_ref as cr
from tests import seed_ref as sr
from tests import smem_ref as ref
from tests.locate_ref import suffix_array
from tests.test_seeds_cpu import _setup

OPTS = [dict(cr.DEFAULTS), dict(cr.DEFAULTS, w=5, max_chain_gap=40)]


def _union(iv):
    return len(set().union(*[range(a, b) for a, b in iv]))


@pytest.mark.parametrize("seed", range(3))
@pytest.mark.parametrize("opt", range(len(OPTS)))
def test_chain_set_against_definitions(seed, opt):
    o = OPTS[opt]
    both, text, seps, model, sym, reads = _setup(800 + seed)
    offs, seeds, hits = sr.reference(model, suffix_array(sym), seps, reads, **{**sr.DEFAULTS, "max_occ": 7})
    l_pac = (int(seps[-1]) + 1 - seps.size) // 2
    n_chains = n_sorted = n_contained = 0
    for i in range(len(reads)):
        shits = cr.read_hits(seeds[offs[i]:offs[i + 1]], hits, seps)
        trace = []
        chains = cr.chain_set(shits, l_pac, trace=trace, **o)
        assert [(c["pos"], c["cid"]) for c in chains] == sorted((c["pos"], c["cid"]) for c in chains)
        by_cid = {c["cid"]: c for c in chains}
        placed = sorted((s, c["cid"]) for c in chains for s in c["seeds"])
        assert len(placed) == sum(t[0] != 1 for t in trace)
        for c in chains:
            s = c["seeds"]
            n_chains += 1
            assert c["pos"] == s[0][0]
            for a, b in zip(s, s[1:]):                                # rule 4 between consecutive seeds
                x, y = b[1] - a[1], b[0] - a[0]
                assert y >= 0 and abs(x - y) <= o["w"] and x - a[2] < o["max_chain_gap"] and y - a[2] < o["max_chain_gap"]
                assert not (a[0] < l_pac <= b[0])                     # never across the strand boundary
            wq, wr = _union([(q, q + n) for r, q, n in s]), _union([(r, r + n) for r, q, n in s])
            w = cr.weight(s)
            assert w <= min(wq, wr)
            if all(a[1] <= b[1] and a[0] <= b[0] for a, b in zip(s, s[1:])):
                n_sorted += 1
                assert w == min(wq, wr)
        for (rb, qb, ln, rid), (got, cid, ends) in zip(shits, trace):
            if got == 1:                                              # contained in the chain it was tested against
                n_contained += 1
                first, last = ends
                c = by_cid[cid]
                assert c["rid"] == rid and c["seeds"][0] == first and last in c["seeds"]
                assert qb >= first[1] and qb + ln <= last[1] + last[2] and rb >= first[0] and rb + ln <= last[0] + last[2]
            elif got == 0:                                            # a new chain starts with it
                assert any(c["seeds"][0] == (rb, qb, ln) and c["rid"] == rid for c in chains)
    assert n_chains and n_sorted and n_contained


class SlotModel:
    """the device's chain set: slots = the read's (rbeg, hit) pairs sorted, a bitmap of occupied slots in 64-bit words
    and a summary bit per word"""

    def __init__(self, rbegs):
        self.order = sorted(range(len(rbegs)), key=lambda h: (rbegs[h], h))
        self.key = [rbegs[h] for h in self.order]
        nw = (len(rbegs) + 63) // 64
        self.bits, self.summary = [0] * nw, [0] * ((nw + 63) // 64)

    def before(self, x):
        """slot_before: the greatest occupied slot below x, or -1"""
        if x == 0:
            return -1
        q = x - 1
        w = q >> 6
        m = self.bits[w] & ((1 << ((q & 63) + 1)) - 1)
        if m:
            return w * 64 + m.bit_length() - 1
        sw, below = w >> 6, w & 63
        while sw >= 0:
            s = self.summary[sw] & ((1 << below) - 1)
            if s:
                w2 = sw * 64 + s.bit_length() - 1
                return w2 * 64 + self.bits[w2].bit_length() - 1
            sw, below = sw - 1, 64
        return -1

    def from_(self, x):
        """slot_from: the least occupied slot at or above x"""
        w = x >> 6
        m = self.bits[w] >> (x & 63) << (x & 63)
        if m:
            return w * 64 + (m & -m).bit_length() - 1
        sw, frm = w >> 6, (w & 63) + 1
        while True:
            s = (self.summary[sw] >> frm << frm) & ((1 << 64) - 1) if frm < 64 else 0
            if s:
                w2 = sw * 64 + (s & -s).bit_length() - 1
                return w2 * 64 + (self.bits[w2] & -self.bits[w2]).bit_length() - 1
            sw, frm = sw + 1, 0

    def lower(self, rbeg):
        import bisect
        p = self.before(bisect.bisect_right(self.key, rbeg))
        if p < 0:
            return None
        return self.order[self.from_(bisect.bisect_left(self.key, self.key[p]))]

    def add(self, h, rbeg):
        import bisect
        p = bisect.bisect_left(self.key, rbeg)
        while self.order[p] != h:
            p += 1
        self.bits[p >> 6] |= 1 << (p & 63)
        self.summary[p >> 12] |= 1 << ((p >> 6) & 63)


@pytest.mark.parametrize("seed", range(4))
def test_slot_model_equals_linear_scan(seed):
    rng = np.random.default_rng(seed)
    for H, span, p_new in ((40, 30, 0.5), (700, 200, 0.3), (9000, 5000, 0.02), (20000, 10 ** 9, 0.001)):
        rbegs = rng.integers(0, span, H).tolist()
        m = SlotModel(rbegs)
        created = []                                                  # (pos, hit) in creation order
        for h, rb in enumerate(rbegs):
            cand = [c for c in created if c[0] <= rb]
            want = None
            if cand:
                top = max(c[0] for c in cand)
                want = next(c[1] for c in created if c[0] == top)     # the first created at the greatest pos
            assert m.lower(rb) == want, (H, h)
            if want is None or rng.random() < p_new:
                m.add(h, rb)
                created.append((rb, h))


def _chains(shits, l_pac=10 ** 6, min_seed_len=19, **o):
    return cr.read_chains(shits, l_pac, min_seed_len, **o)


def test_equal_pos_chains_take_the_first_created():
    # two chains at pos 100 (records 0 and 1); a hit of record 1 at 100 is tested against the first (record 0): a third
    # chain, though the second would contain it
    got = cr.chain_set([(100, 0, 30, 0), (100, 0, 30, 1), (100, 5, 20, 1)], 10 ** 6)
    assert [(c["pos"], c["rid"], len(c["seeds"])) for c in got] == [(100, 0, 1), (100, 1, 1), (100, 1, 1)]
    got = cr.chain_set([(100, 0, 30, 0), (100, 0, 30, 1), (100, 5, 20, 0)], 10 ** 6)
    assert [len(c["seeds"]) for c in got] == [1, 1]                   # contained in the first


def test_contained_records_and_strand_boundary():
    got = _chains([(100, 0, 30, 0), (105, 5, 20, 0), (140, 40, 30, 0)])
    assert len(got) == 1 and got[0]["seeds"] == [(100, 0, 30), (140, 40, 30)] and got[0]["w"] == 60
    got = _chains([(100, 0, 30, 0), (140, 40, 30, 1)])                 # another record
    assert len(got) == 2
    got = _chains([(960, 0, 30, 0), (1000, 40, 30, 0)], l_pac=1000)   # colinear, but the second is on the reverse strand
    assert sorted(c["pos"] for c in got) == [960, 1000]
    got = _chains([(1000, 0, 30, 0), (1040, 40, 30, 0)], l_pac=1000)  # both reverse: one chain
    assert len(got) == 1 and got[0]["pos"] == 1000


def _four_on_one_span(extra=()):
    """chains of equal weight on query [0, 50) far apart on the reference: every one overlaps every other"""
    return [(1000 * k, 0, 50, 0) for k in range(1, 5)] + list(extra)


def test_kept_values_and_max_chain_extend():
    got = _chains(_four_on_one_span())
    # a0 kept 3; a1..a3 each 2, then 1 as the first shadowed chain of the one before
    assert [(c["pos"], c["kept"]) for c in got] == [(1000, 3), (2000, 1), (3000, 1), (4000, 1)]
    got = _chains(_four_on_one_span(), max_chain_extend=2)            # the cut falls on the third: it and the fourth go
    assert [(c["pos"], c["kept"]) for c in got] == [(1000, 3), (2000, 1)]
    got = _chains(_four_on_one_span(), max_chain_extend=0)
    assert [(c["pos"], c["kept"]) for c in got] == [(1000, 3)]
    # a 2 that stays: a0 [0, 100) w 100, a1 [0, 60) a0's first shadowed chain, a2 [50, 100) overlaps a0 only (and a1 by
    # less than half)
    got = _chains([(1000, 0, 100, 0), (5000, 0, 60, 0), (9000, 50, 50, 0)])
    assert [(c["pos"], c["kept"]) for c in got] == [(1000, 3), (5000, 1), (9000, 2)]
    # no overlap: all 3
    got = _chains([(1000, 0, 40, 0), (5000, 60, 40, 0)])
    assert [c["kept"] for c in got] == [3, 3]


def test_dropped_chain_revived_and_min_chain_weight():
    # a1 (w 30) is dropped by a0 (w 100: 30 < 50 and 70 >= 38) but is a0's first shadowed chain: kept 1
    got = _chains([(1000, 0, 100, 0), (5000, 10, 30, 0)])
    assert [(c["pos"], c["kept"], c["w"]) for c in got] == [(1000, 3, 100), (5000, 1, 30)]
    # a2 is dropped too and nobody's first: gone
    got = _chains([(1000, 0, 100, 0), (5000, 10, 30, 0), (9000, 20, 30, 0)])
    assert [c["pos"] for c in got] == [1000, 5000]
    assert _chains([(1000, 0, 100, 0), (5000, 10, 30, 0)], min_chain_weight=101) == []
    got = _chains([(1000, 0, 100, 0), (5000, 10, 30, 0)], min_chain_weight=31)
    assert [(c["pos"], c["kept"]) for c in got] == [(1000, 3)]
    got = _chains([(1000, 0, 100, 0), (5000, 10, 30, 0)], mask_level=1.5)     # no overlap is large: both 3
    assert [c["kept"] for c in got] == [3, 3]


def test_frac_rep_sweep():
    assert cr.frac_rep([(0, 30, 600), (10, 40, 501), (50, 60, 900), (55, 58, 10)], 100, 500) == np.float32(0.5)
    assert cr.frac_rep([], 0, 500) == 0


def test_bwa_rbeg_is_bwas_forward_reverse_text():
    rng = np.random.default_rng(3)
    recs = [bytes(b"ACGT"[x] for x in rng.integers(0, 4, k)) for k in (300, 41, 777)]
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    fwd = b"".join(recs)
    bwa_text = fwd + ref.revcomp(fwd)
    t = text.tobytes()
    pos = np.array([p for p in range(text.size - 20) if all(c in b"ACGT" for c in t[p:p + 20])][::7], dtype=np.uint64)
    rec, strand, off = api.strand_offsets(pos, 20, seps)
    rb = api.bwa_rbeg(rec, strand, off, 20, seps)
    for p, r, s, x in zip(pos.tolist(), rb.tolist(), strand.tolist(), rec.tolist()):
        assert bwa_text[r:r + 20] == t[p:p + 20]
        assert (r >= len(fwd)) == bool(s) and (s or r == p - x)
    assert rb.dtype == np.int64


def test_dtypes_match_header_layout(tmp_path):
    structs = {"debwt_chain": api.CHAIN_DTYPE, "debwt_chain_seed": api.CHAIN_SEED_DTYPE}
    body = ""
    for name, dt in structs.items():
        body += f'printf("%zu ", sizeof({name}));' + "".join(f'printf("%zu ", offsetof({name}, {f}));' for f in dt.names)
    opts = [f for f, _ in api.ChainOpts._fields_]
    body += 'printf("%zu ", sizeof(debwt_chain_opts));' + "".join(f'printf("%zu ", offsetof(debwt_chain_opts, {f}));' for f in opts)
    src = tmp_path / "chains.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "debwt_b200.h"\nint main(void){' + body + "return 0;}\n")
    exe = tmp_path / "chains"
    subprocess.check_call(["gcc", "-I", os.path.dirname(binding.HEADER), "-o", str(exe), str(src)])
    out = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert list(api.CHAIN_DTYPE.names) == ["pos", "seed_begin", "n_seeds", "weight", "record", "strand", "kept", "frac_rep"]
    assert list(api.CHAIN_SEED_DTYPE.names) == ["rbeg", "qbeg", "len"]
    for name, dt in structs.items():
        assert out[0] == dt.itemsize and out[1:1 + len(dt.names)] == [dt.fields[f][1] for f in dt.names], name
        out = out[1 + len(dt.names):]
    assert out == [ctypes.sizeof(api.ChainOpts)] + [getattr(api.ChainOpts, f).offset for f in opts]
    assert api.CHAIN_DTYPE.itemsize == 40 and api.CHAIN_SEED_DTYPE.itemsize == 16
