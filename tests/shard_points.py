"""Inputs placed at the slice, splitter and row boundaries of the sharded build (csrc/shard.cu, csrc/dist_kernels.cu), the
per-rank restatement of that build, and the library constants that place the inputs.  tests/test_gpu_shard_points.py runs
every case at each of its world sizes and compares every rank's counts with the restatement; the restatement and the
placement of every case are checked without a GPU in tests/test_shard_points_cpu.py.

A BWT comparison alone cannot see most errors of the sharded orchestration: a splitter chosen from different samples, or
an owner rule that moves the k-mers equal to a splitter to the rank below, still partitions the keys, and the BWT stays
right.  Only each rank's key count sees them.  Every case asserts from the restatement which side of its edge it lies on,
so a retuned constant fails the placement check instead of silently moving the case."""
from __future__ import annotations

import numpy as np

from oracle import stages as st
from tests import switch_points as sw

# ---- library constants -------------------------------------------------------------------------------------------
MAX_RANKS = 16                       # csrc/shard.cu:41 kMaxRanks; csrc/dist_kernels.cu:46 MAX_RANKS
SAMPLES_PER_RANK = 4096              # csrc/shard.cu:42 kSamplesPerRank: at most 4096 sampled keys per slice
KMER_MASK = 0xFFFFFFFFFFFFFFFC       # csrc/shard.cu:43 kKmerMask: splitters and owners compare k-mers (low 2 bits cleared)
PART_TILE = 256 * 8                  # csrc/dist_kernels.cu:44-45: keys per block of the partition / exchange kernels
GOLDEN = 0.6180339887                # csrc/dist_kernels.cu:350: tile stride of the peer-store exchange
STRIDE_MIN_GRID = 8                  # csrc/dist_kernels.cu:352: stride 1 below 8 tiles
GRID_STRIDES = {7: 1, 8: 5, 9: 5, 15: 7}   # the strides at the exchange-grid cases' tile counts; 15 tiles: 9, lowered to 7
SLICE_ALIGN = 32                     # csrc/shard.cu:299-303: slices are whole 32-symbol words


# ---- geometry ----------------------------------------------------------------------------------------------------
def words_per_slice(n, G):
    """wp = ceil(((N + 63) / 32 + 1) / G) (csrc/shard.cu:299-300)"""
    return -(-((n + 63) // 32 + 1) // G)


def n_for_wp(G, wp):
    """the largest N whose slices are wp words long at world G"""
    n = 32 * wp * G
    while words_per_slice(n, G) != wp:
        n -= 1
    return n


def exchange_stride(grid):
    """the tile stride of partition_scatter_p2p_staged_kernel: golden ratio, odd, lowered until coprime with the grid,
    1 below 8 tiles (csrc/dist_kernels.cu:348-352)"""
    stride = int(grid * GOLDEN) | 1
    while stride > 1 and np.gcd(stride, grid) != 1:
        stride -= 2
    return 1 if grid < STRIDE_MIN_GRID else stride


def exchange_grid(n_items):
    return -(-n_items // PART_TILE)


def emit_positions(sym, seps, sorted_keys, gmask, specials):
    """bool per text position: the position emits a branch code.  The emit array of st.branch_codes, which it does not
    return: sentinel windows whose flag is set, and in-record windows whose k-mer is multi-out."""
    emit = np.zeros(sym.size, dtype=bool)
    for e in specials:
        if e["emit"]:
            emit[e["pos"]] = True
    keys = st.extract_keys(sym, seps)
    ppos = window_positions(seps)
    first = np.searchsorted(sorted_keys >> np.uint64(2), keys >> np.uint64(2), side="left")
    emit[ppos[st.multi_out(gmask[first])]] = True
    return emit


def windows_before(x, seps):
    """in-record windows that start at a position < x (csrc/shard.cu:217-227 windows_before)"""
    total, start = 0, 0
    for s in np.asarray(seps).tolist():
        end = min(s - 31, x)                                 # the last window of a record starts at s - 32
        total += max(end - start, 0)
        start = s + 1
        if start >= x:
            break
    return total


def window_positions(seps):
    """text position of every in-record window, in text (= key index) order"""
    out, start = [], 0
    for s in np.asarray(seps).tolist():
        out.append(np.arange(start, s - 31))
        start = s + 1
    return np.concatenate(out)


# ---- the restatement ---------------------------------------------------------------------------------------------
class Restated(sw.Restated):
    """sw.Restated with the sentinel suffixes, the emit positions and the keys in text order kept: what the per-rank
    restatement (ranks()) needs besides the sorted keys and masks."""

    def __init__(self, records, doubling=False):
        super().__init__(records, specials=False)
        self.doubling = doubling
        self.spec = st.special_suffixes(self.sym, self.seps, self.sk)
        self.sp, self.blue = st.branch_codes(self.sym, self.seps, self.sk, self.gmask, self.spec)
        self.keys = st.extract_keys(self.sym, self.seps)
        self.ppos = window_positions(self.seps)
        self.ins = np.array([e["ins"] for e in self.spec], dtype=np.int64)
        self.emit = emit_positions(self.sym, self.seps, self.sk, self.gmask, self.spec)
        self._ref = None
        self._ranks = {}

    def ref(self):
        """(words, sharp rows, dollar row) of T, computed once"""
        if self._ref is None:
            self._ref = self.bwt(self.doubling)
        return self._ref

    def ranks(self, G):
        if G not in self._ranks:
            self._ranks[G] = Ranks(self, G)
        return self._ranks[G]

    def win_branch(self):
        """bool per window (text order): its k-mer is a branch k-mer"""
        first = np.searchsorted(self.sk >> np.uint64(2), self.keys >> np.uint64(2), side="left")
        return self.mi[first] | self.mo[first]


def slice_samples(keys, idx_base, cnt):
    """the sampled keys of one slice, in position order: ns = min(cnt, 4096) keys at stride max(cnt / ns, 1)
    (csrc/shard.cu:358-361)"""
    ns = min(cnt, SAMPLES_PER_RANK)
    if ns == 0:
        return keys[:0]
    stride = max(cnt // ns, 1)
    return keys[idx_base:idx_base + cnt][::stride][:ns]


def splitters_of(valid_sorted, G):
    """valid[i |valid| / G] & ~3 for i = 1 .. G-1, all-ones k-mers when nothing was sampled (csrc/shard.cu:374-376)"""
    m = valid_sorted.size
    return np.array([KMER_MASK if m == 0 else int(valid_sorted[i * m // G]) & KMER_MASK for i in range(1, G)], dtype=np.uint64)


def owners(keys, splitters):
    """owner of a key = number of splitters <= (key & ~3) (OwnerFn, csrc/dist_kernels.cu:55-61)"""
    return np.searchsorted(splitters, np.asarray(keys, dtype=np.uint64) & np.uint64(KMER_MASK), side="right")


class Ranks:
    """What every rank of the sharded build at world G works on, restated from the text.  Lists have one entry per rank."""

    def __init__(self, rs, G):
        assert 1 <= G <= MAX_RANKS
        n, seps = rs.n, rs.seps
        self.G = G
        self.wp = wp = words_per_slice(n, G)
        self.pos_lo = [SLICE_ALIGN * r * wp for r in range(G)]
        self.pos_hi = [max(min(SLICE_ALIGN * (r + 1) * wp, n), lo) for r, lo in enumerate(self.pos_lo)]
        self.n_valid = [hi - lo for lo, hi in zip(self.pos_lo, self.pos_hi)]
        self.idx_base = [windows_before(lo, seps) for lo in self.pos_lo]
        self.cnt = [windows_before(hi, seps) - b if nv else 0 for hi, b, nv in zip(self.pos_hi, self.idx_base, self.n_valid)]
        self.samples = [slice_samples(rs.keys, b, c) for b, c in zip(self.idx_base, self.cnt)]
        self.splitters = splitters_of(np.sort(np.concatenate(self.samples)), G)
        own = owners(rs.sk, self.splitters)
        self.n_keys_local = np.bincount(own, minlength=G).tolist()
        self.key_base = np.concatenate(([0], np.cumsum(self.n_keys_local))).astype(np.int64).tolist()
        self.owned = [rs.sk[self.key_base[r]:self.key_base[r + 1]] for r in range(G)]
        assert (own[1:] >= own[:-1]).all()                   # owners are monotone in the key: every rank owns a key range
        self.sort_sweeps = [sw.sort_sweeps(k) for k in self.owned]
        # rows: a rank's first row is its first key's row (the sentinel suffixes with ins <= key_base go before it)
        self.r_lo = [0 if kb == 0 else kb + int(np.searchsorted(rs.ins, kb, side="right")) for kb in self.key_base[:G]] + [n]
        heads = rs.ghead & (rs.mi | rs.mo)
        self.n_branch_local = [int(heads[self.key_base[r]:self.key_base[r + 1]].sum()) for r in range(G)]
        # branch codes: a rank's codes start at the number of code-emitting positions before its slice
        ce = np.concatenate(([0], np.cumsum(rs.emit)))
        self.code_base = [int(ce[min(lo, n)]) for lo in self.pos_lo]
        self.s_loc = [int(ce[min(hi, n)] - ce[min(lo, n)]) for lo, hi in zip(self.pos_lo, self.pos_hi)]
        self.dollar_index = int(ce[int(seps[-1]) - 31])
        self.grid = [exchange_grid(c) for c in self.cnt]
        self.stride = [exchange_stride(g) if g else 0 for g in self.grid]

    def slice_of(self, p):
        """the rank whose slice holds text position p"""
        return p // (SLICE_ALIGN * self.wp)

    def rank_of_row(self, row):
        """the rank whose row range holds `row` (ranks with empty ranges are skipped)"""
        return int(np.searchsorted(self.r_lo, row, side="right")) - 1

    def rank_of_key(self, key):
        return int(owners([key], self.splitters)[0])

    def kmer_bounds(self, r):
        """first and last k-mer (key >> 2) of rank r, or None when it owns no key"""
        k = self.owned[r]
        return (int(k[0]) >> 2, int(k[-1]) >> 2) if k.size else None


# ---- inputs ------------------------------------------------------------------------------------------------------
def records_at(seps, fill, seed):
    """records whose separators fall at the given text positions (ascending; the last one is N - 1), filled by
    fill(rng, length)"""
    rng = np.random.default_rng(seed)
    recs, start = [], 0
    for s in seps:
        assert s - start > 32, (start, s)
        recs.append(bytes(fill(rng, s - start)))
        start = s + 1
    return recs


def random_fill(rng, n):
    return sw.random_bases(rng, n)


def repeat_fill(rng, n):
    return sw.repeat_rich(rng, n, el_len=60, muts=2)


def alphabet_fill(alpha):
    a = np.frombuffer(alpha, dtype=np.uint8)
    return lambda rng, n: a[rng.integers(0, a.size, size=n)]


def run_fill(head_len, base, run_len, tail_len, alpha=b"ACGT"):
    """head_len random bases, a run of one base, tail_len random bases (one record)"""
    f = alphabet_fill(alpha)
    return lambda rng, n: np.concatenate([f(rng, head_len), np.full(run_len, ord(base), np.uint8), f(rng, tail_len)])[:n]


class Case:
    """make() -> records; place(Restated) asserts the side of its edge the input lies on, at the world sizes it names.
    worlds: the world sizes the GPU test runs it at.  doubling: reference BWT by suffix ranking (long runs)."""

    def __init__(self, make, place, worlds, doubling=False):
        self.make, self.place, self.worlds, self.doubling = make, place, worlds, doubling


# -- empty slices and slices without windows
def _place_tiny(rs):
    assert rs.n == 34 and rs.sk.size == 2
    for G in (4, 8, 16):
        rk = rs.ranks(G)
        assert rk.wp == 1 and [lo >= rs.n for lo in rk.pos_lo].count(True) == G - 2      # ranks 2.. lie past N
        assert rk.n_valid[1] == 2 and rk.cnt[1] == 0                                       # last base and '$', no window
        assert sum(rk.n_keys_local) == 2


def _place_n417(rs):
    assert rs.n == 417 and rs.seps[0] % 32 == 31
    rk = rs.ranks(16)
    assert rk.wp == 1
    assert rk.pos_lo[13] == 416 and rk.n_valid[13] == 1                                   # only the last separator
    assert rk.n_valid[14] == rk.n_valid[15] == 0 and rk.pos_lo[14] >= rs.n
    assert rk.n_valid[2] == 32 and rk.cnt[2] == 0 and rk.pos_hi[2] == int(rs.seps[0]) + 1  # a record's last 32 symbols
    rk8 = rs.ranks(8)
    assert rk8.wp == 2 and rk8.n_valid[7] == 0


# -- separators at slice edges
def _edge_seps(G, wp=8):
    e = 32 * wp
    n = n_for_wp(G, wp)
    seps = [e - 1]                                           # at pos_hi - 1 of rank 0: a record starts at pos_lo of rank 1
    if G >= 3:
        seps.append(2 * e)                                   # at pos_lo of rank 2
    if G >= 4:
        seps += [3 * e - 17, 3 * e + 17]                     # a record of 33 bases across pos_lo of rank 3
    return seps + [n - 1]


def _sep_edges_case(G, seed):
    def place(rs):
        rk = rs.ranks(G)
        seps = rs.seps.tolist()
        assert rk.pos_hi[0] - 1 in seps and rk.pos_lo[1] - 1 in seps
        if G >= 3:
            assert rk.pos_lo[2] in seps
        if G >= 4:
            i = seps.index(rk.pos_lo[3] - 17)
            assert seps[i + 1] - seps[i] - 1 == 33 and seps[i] < rk.pos_lo[3] < seps[i + 1]
        if G >= 4:                                           # a branch k-mer whose window starts in one slice and ends in the next
            wb, p = rs.win_branch(), rs.ppos
            assert ((p >= rk.pos_lo[3] - 31) & (p < rk.pos_lo[3]) & wb).any()
    return Case(lambda: records_at(_edge_seps(G), repeat_fill, seed), place, [G])


# -- code words shared across ranks
def _codes_seps():
    # G = 5, wp = 34: 31 short records in slice 0, one record over all of slice 1, one tail in slice 2, one in slice 3,
    # and the last record's tail in slice 4.  Random bases: the only code positions are the 34 record tails.
    return [34 + 35 * i for i in range(31)] + [2300, 3400, 5299]


def _place_codes(rs):
    rk = rs.ranks(5)
    assert rk.wp == 34 and rs.sp.size == rs.R
    assert rk.code_base == [0, 31, 31, 32, 33]
    assert [c % 32 for c in rk.code_base[1:]] == [31, 31, 0, 1]
    assert rk.s_loc[1] == 0 and rk.s_loc[0] > 0 and rk.s_loc[2] > 0                   # or_range skips rank 1
    assert rk.slice_of(int(rs.seps[-1]) - 31) == 4 and rk.dollar_index == rs.R - 1    # dollar_index on rank 4


# -- sampling stride
def _sampling_case(G, wp, missing, cnt, stride):
    e = 32 * wp

    def make():
        n = n_for_wp(G, wp)
        return records_at([e + 31 - missing, n - 1], repeat_fill, cnt)

    def place(rs):
        rk = rs.ranks(G)
        assert rk.cnt[0] == cnt and max(cnt // min(cnt, SAMPLES_PER_RANK), 1) == stride
        assert rk.samples[0].size == min(cnt, SAMPLES_PER_RANK)
    return Case(make, place, [G])


# -- equal splitters
def _tiny_rank_records(L=9891):
    # random | G run | random, at G = 4: quantile 1 lands on the key just below the G^31 group, quantiles 2 and 3 in it.
    # L is the first run length that places the case; every slice stays below 4096 windows, so every key is sampled.
    return records_at([3000 + L + 3000], run_fill(3000, "G", L, 3000), 61)


def _place_tiny_rank(rs):
    rk = rs.ranks(4)
    g31 = (1 << 62) // 3 * 2                                                            # G^31: 0b1010...10
    assert rk.splitters[1] == rk.splitters[2] == np.uint64(g31 << 2)                  # equal splitters
    assert rk.n_keys_local[2] == 0 and rk.n_keys_local[1] > 0                           # an empty rank in the middle
    assert int((rs.sk >> np.uint64(2) == np.uint64(g31)).sum()) >= 5000                 # a big group exactly at a splitter
    # rank 1 owns one small group just below the G^31 group: a row range inside one output word
    assert rk.n_keys_local[1] < 8 and rk.r_lo[2] - rk.r_lo[1] > 0 and rk.r_lo[1] // 32 == (rk.r_lo[2] - 1) // 32
    assert rk.n_branch_local[2] == 0 and sum(rk.n_branch_local[3:]) > 0                 # repeated branch-table bases


def _below_split_records(L=6264):
    # random | C run | random at G = 6: a splitter is the first k-mer above the C^31 group (L is the first run length
    # that places the case)
    return records_at([2500 + L + 4000], run_fill(2500, "C", L, 4000), 67)


def _place_below_split(rs):
    rk = rs.ranks(6)
    c31 = (1 << 62) // 3
    km = rs.sk >> np.uint64(2)
    assert int((km == np.uint64(c31)).sum()) >= 5000
    nxt = int(km[np.searchsorted(km, np.uint64(c31), side="right")])
    assert nxt << 2 in [int(s) for s in rk.splitters]                                   # the group is just below a splitter
    r = rk.rank_of_key(c31 << 2)
    assert rk.kmer_bounds(r)[1] == c31 and rk.kmer_bounds(r + 1)[0] == nxt


def _place_rank0_empty(rs):
    # C run in a text over C, G, T whose records end in A: C^31 is the smallest k-mer, so the first splitters equal it
    # and ranks 0 and 1 own nothing; the sentinel suffixes "A#" sort below every key (ins == 0)
    rk = rs.ranks(4)
    assert rk.n_keys_local[0] == rk.n_keys_local[1] == 0 and rk.r_lo[:3] == [0, 0, 0]
    assert (rs.ins == 0).sum() == rs.R
    assert rk.n_branch_local[0] == rk.n_branch_local[1] == 0


def _rank0_empty_records():
    cgt = alphabet_fill(b"CGT")
    rng = np.random.default_rng(71)
    recs = [bytes(np.concatenate([cgt(rng, 2000), np.full(9000, ord("C"), np.uint8), cgt(rng, 2000)])) + b"A",
            bytes(cgt(rng, 1500)) + b"A"]
    return recs


def _place_t_alone(rs):
    rk = rs.ranks(4)
    t31 = sw.T31
    assert rk.n_keys_local[2] == 0                                                      # equal splitters at T^31
    last = rk.owned[3]
    assert last.size > 0 and (last >> np.uint64(2) == np.uint64(t31)).all()             # poly-T alone on the last rank
    assert (last == np.uint64(0xFFFFFFFFFFFFFFFF)).any()


# -- in-edges across ranks
def _in_edges_records():
    rng = np.random.default_rng(83)
    recs = [bytes(sw.repeat_rich(rng, 2500, el_len=120, muts=2)) + b"T" * 40 + bytes(sw.random_bases(rng, 500)),
            bytes(sw.repeat_rich(rng, 3000, el_len=120, muts=2))]
    return recs


def _place_in_edges(rs):
    rk = rs.ranks(6)
    dk, cnt = st.rle(rs.sk)
    x = dk & np.uint64((1 << 62) - 1)                                                   # suffix k-mer X of every cX
    rc, rx = owners(dk, rk.splitters), owners(x << np.uint64(2), rk.splitters)
    exists = np.isin(x, rs.sk >> np.uint64(2))
    first = np.array([b[0] if b else -1 for b in map(rk.kmer_bounds, range(6))] + [-1], dtype=object)
    is_first = np.array([int(xi) == first[r] for xi, r in zip(x.tolist(), rx.tolist())])
    assert (exists & (rx == rc + 1) & is_first).any()                                   # cX on rank r, X first of rank r+1
    assert (exists & (rc == rx + 1)).any()                                              # cX on rank r+1, X on rank r
    assert (exists & (cnt >= 2) & (rc != rx)).any()                                     # duplicate (k+1)-mers across ranks
    t = rk.rank_of_key(0xFFFFFFFFFFFFFFFF)                                              # poly-T with other keys
    assert (rk.owned[t] == np.uint64(0xFFFFFFFFFFFFFFFF)).any() and (rk.owned[t] >> np.uint64(2) != np.uint64(sw.T31)).any()


# -- exchange grid
def _grid_case(G, wp, tiles, seps_in_slice0, seed):
    e = 32 * wp

    def make():
        n = n_for_wp(G, wp)
        return records_at([e // 2 + 400 * i for i in range(seps_in_slice0)] + [n - 1], random_fill, seed)

    def place(rs):
        rk = rs.ranks(G)
        assert rk.grid[:len(tiles)] == tiles, rk.grid
        assert [rk.stride[r] for r in range(len(tiles))] == [GRID_STRIDES[t] for t in tiles]
    return Case(make, place, [G])


# -- row ranges
def _rows_records():
    return records_at([1700, 3100, 4400, 6000], repeat_fill, 103)          # the first seed that places the case


def _place_rows(rs):
    rk = rs.ranks(16)
    res = {lo % 32 for lo, hi in zip(rk.r_lo[1:16], rk.r_lo[2:]) if hi > lo}
    assert {0, 1, 31} <= res, res
    assert set(rs.ins.tolist()) & set(rk.key_base[1:16]) - {0}                          # ins == key_base: the rank before


def _boundary_row_records(dollar):
    # rec_a = "GC" + {G,T}*: its first k-mer X is the median key (all keys are sampled at G = 2), so X is rank 1's first
    # k-mer and the suffix at rec_a's start is rank 1's first row.  rec_a first: that row is '$', second: a '#'.
    rng = np.random.default_rng(97 + dollar)
    rec_b = bytes(alphabet_fill(b"AC")(rng, 2031))
    rec_a = b"GC" + bytes(alphabet_fill(b"GT")(rng, 2031))
    return [rec_a, rec_b] if dollar else [rec_b, rec_a]


def _place_boundary_row(dollar):
    def place(rs):
        rk = rs.ranks(2)
        _, sharp, dol = rs.ref()
        row = int(dol[0]) if dollar else int(sharp[0])
        assert row == rk.r_lo[1] and rk.rank_of_row(row) == 1
    return place


# -- case
def _lower_records():
    # the sep_edges layout at G = 6 (wp = 8); the last record holds pos_lo of rank 4 = 1024
    recs = records_at(_edge_seps(6), repeat_fill, 101)
    start = sum(len(r) + 1 for r in recs[:-1])
    e = 4 * 32 * 8 - start
    r = bytearray(recs[-1])
    r[e - 40:e + 40] = r[e - 40:e + 40].lower()
    recs[-1] = bytes(r)
    return recs


def _place_lower(rs):
    rk = rs.ranks(6)
    low = [i for i, c in enumerate(b"".join(r + b"#" for r in rs.records)) if 97 <= c <= 122]
    assert low and low[0] < rk.pos_lo[4] <= low[-1]


CASES = {
    # empty slices, a slice that holds only the last separator, slices with symbols but no windows
    "tiny_33": Case(lambda: [b"ACGT" * 8 + b"A"], _place_tiny, [4, 8, 16]),
    "n417": Case(lambda: records_at([95, 200, 300, 416], repeat_fill, 7), _place_n417, [8, 16]),
    # separators at pos_hi - 1, pos_lo and pos_lo - 1, a 33-base record across an edge, branch windows across edges
    **{f"sep_edges_g{G}": _sep_edges_case(G, 10 + G) for G in (2, 3, 5, 7, 9, 10, 11, 12, 13, 14, 15)},
    # code words shared by ranks, a rank without codes between two with codes, dollar_index off rank 0
    "codes_shared": Case(lambda: records_at(_codes_seps(), random_fill, 19), _place_codes, [1, 5]),
    # sampling: all keys, stride 1 with one key left over, stride 2 with one left over
    "sample_4095": _sampling_case(2, 128, 1, 4095, 1),
    "sample_4096": _sampling_case(2, 128, 0, 4096, 1),
    "sample_4097": _sampling_case(2, 129, 31, 4097, 1),
    "sample_8193": _sampling_case(3, 257, 31, 8193, 2),
    # equal splitters: an empty rank in the middle, at rank 0, and a rank with poly-T alone
    "tiny_rank": Case(_tiny_rank_records, _place_tiny_rank, [4], doubling=True),
    "below_splitter": Case(_below_split_records, _place_below_split, [6],
                           doubling=True),
    "rank0_empty": Case(_rank0_empty_records, _place_rank0_empty, [4], doubling=True),
    "t_alone": Case(lambda: records_at([3000 + 9000], run_fill(3000, "T", 9000, 0), 73), _place_t_alone, [4], doubling=True),
    # in-edges from one rank to the next and back, duplicate (k+1)-mers, poly-T among other keys
    "in_edges": Case(_in_edges_records, _place_in_edges, [6]),
    # key exchange tiles: 7 (stride 1), 8 and 9 (golden-ratio stride), 15 (the gcd loop lowers the stride)
    "grid_7_8": _grid_case(3, 450, [7, 8], 2, 31),
    "grid_9": _grid_case(2, 520, [9], 0, 37),
    "grid_15": _grid_case(2, 950, [15], 0, 43),
    # row ranges: first rows at 0, 1 and 31 mod 32, sentinel suffixes at a rank's first key; '$' / '#' on a first row
    "rows": Case(_rows_records, _place_rows, [16]),
    "dollar_first_row": Case(lambda: _boundary_row_records(True), _place_boundary_row(True), [2]),
    "sharp_first_row": Case(lambda: _boundary_row_records(False), _place_boundary_row(False), [2]),
    # a lowercase run across a slice edge
    "lowercase_edge": Case(_lower_records, _place_lower, [6]),
}
