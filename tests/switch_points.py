"""Inputs placed at the thresholds where the K3-K10 kernels switch paths, the library constants that place them, and the
CPU references the switch-point tests compare with (tests/test_gpu_switch_points.py; the references and the placement of
every input are checked without a GPU in tests/test_switch_points_cpu.py).

Every constant below mirrors one in debwt_b200/csrc.  Each case asserts from the restatement which side of its threshold
it lies on, so a retuned constant fails the placement check instead of silently moving the case off its path."""
from __future__ import annotations

import numpy as np

from oracle import coracle, stages as st

# ---- library constants -------------------------------------------------------------------------------------------
KEYS_PER_BUCKET = 8                  # csrc/stages.cuh:45-49 key_index_bits: about 8 sorted keys per bucket ...
KEY_INDEX_BITS = (8, 28)             # ... in a direct index of 8 to 28 bits
SORT_PASSES = 8                      # csrc/radix_sort.cu:403: eight 8-bit digit passes, a pass skipped when its digit is constant
TEXT_HIST_RATIO = 2048               # csrc/stages.cu:364 text_digit_hist_applies: digit histogram from the text when 2048 R <= N
ME_TILE = 8192                       # csrc/stages.cu:480: target keys per in-edge join tile
ME_CAP = 8 * ME_TILE                 # csrc/stages.cu:481: sources per (first base, tile) run before the rest goes to the over list
K9_TILE_POS = 4096                   # csrc/stages.cu:190 TILE_POS: text positions per K9 block
BLUE_FIX_DIV = 4                     # csrc/api.cu:504: interleaved blue fix when n_blue >= nbw / 4, nbw = ceil(N / 32)
SPECIAL_ALL_PAIRS = 16384            # csrc/special.cuh:69 kSpecialAllPairs: all-pairs ranking up to 16384 sentinel suffixes
K10_WARP, K10_MID, K10_TINY, K10_SMEM = 32, 128, 512, 4096   # csrc/bluesort.cu:134-136 (MID_SEG :37, SMEM_SEG :39), TINY :465
T31 = (1 << 62) - 1                  # the k-mer T^31 as a 62-bit value

BASES = np.frombuffer(b"ACGT", dtype=np.uint8)


# ---- restatement-side quantities ---------------------------------------------------------------------------------
def key_index_bits(n_keys):
    b = KEY_INDEX_BITS[0]
    while b < KEY_INDEX_BITS[1] and (KEYS_PER_BUCKET << b) < n_keys:
        b += 1
    return b


def text_hist_applies(n_symbols, n_records):
    return n_records * TEXT_HIST_RATIO <= n_symbols


def sort_sweeps(keys):
    """digit passes the LSD radix sort runs: one per 8-bit digit that is not the same in every key"""
    keys = np.asarray(keys, dtype=np.uint64)
    if keys.size <= 1:
        return 0
    return sum(int(np.unique((keys >> np.uint64(8 * p)) & np.uint64(255)).size > 1) for p in range(SORT_PASSES))


def last_pass_skipped(keys):
    """the top digit is constant, so the sort's last pass cannot mark the key index (key_index_mark_kernel does)"""
    top = np.asarray(keys, dtype=np.uint64) >> np.uint64(56)
    return bool((top == top[0]).all())


def edge_runs(sk):
    """The in-edge join's runs: source key s (first base c = s >> 62) is served by the tile of its target, i.e. of the
    lower bound of its suffix k-mer among the sorted keys.  Returns (c, tile, begin, end) for every non-empty run
    (sources [begin, end) of the sorted keys) and, per run, the distinct sources at or past begin + ME_CAP whose target
    k-mer exists: the in-edges only the over list marks."""
    sk = np.asarray(sk, dtype=np.uint64)
    q = sk << np.uint64(2)
    lb = np.searchsorted(sk, q, side="left")
    exists = (lb < sk.size) & ((sk[np.minimum(lb, sk.size - 1)] >> np.uint64(2)) == (q >> np.uint64(2)))
    first = np.ones(sk.size, dtype=bool)
    first[1:] = sk[1:] != sk[:-1]
    c = (sk >> np.uint64(62)).astype(np.int64)
    tile = lb // ME_TILE
    runs = []
    brk = np.flatnonzero((c[1:] != c[:-1]) | (tile[1:] != tile[:-1])) + 1
    starts = np.concatenate(([0], brk))
    ends = np.concatenate((brk, [sk.size]))
    for b, e in zip(starts.tolist(), ends.tolist()):
        tail = slice(b + ME_CAP, e) if e - b > ME_CAP else slice(0, 0)
        runs.append((int(c[b]), int(tile[b]), b, e, int((first[tail] & exists[tail]).sum())))
    return runs


def k9_one_record_tiles(seps, n):
    """per K9 tile: the first and the last position of the tile lie in the same record (the one-record fast path)"""
    seps = np.asarray(seps, dtype=np.int64)
    base = np.arange(0, n, K9_TILE_POS)
    last = np.minimum(base + K9_TILE_POS - 1, n - 1)
    return np.searchsorted(seps, base, side="left") == np.searchsorted(seps, last, side="left")


def suffix_ranks(codes):
    """rank[i] = place of the suffix starting at i among all suffixes of `codes` (small non-negative integers; the last
    code must occur nowhere else), by prefix doubling"""
    codes = np.asarray(codes)
    n = codes.size
    rank = codes.astype(np.int64)
    k = 1
    while True:
        nxt = np.full(n, -1, dtype=np.int64)
        nxt[:n - k] = rank[k:]
        order = np.lexsort((nxt, rank))
        a, b = rank[order], nxt[order]
        new_group = np.ones(n, dtype=bool)
        new_group[1:] = (a[1:] != a[:-1]) | (b[1:] != b[:-1])
        rank = np.empty(n, dtype=np.int64)
        rank[order] = np.cumsum(new_group) - 1
        if rank[order[-1]] == n - 1 or k >= n:
            return rank
        k *= 2


def doubling_bwt(sym):
    """(words, sharp, dollar) of T by suffix ranking: for texts with long runs, where the C oracle's comparisons get long"""
    sa = np.argsort(suffix_ranks(sym))
    return st.finish(sym[(sa - 1) % sym.size])


class Restated:
    """The stage restatement (oracle/stages.py) of one input, computed once: sorted keys, group masks and, unless
    `specials` is off (the sentinel sort is plain Python), the branch codes and blue entries."""

    def __init__(self, records, specials=True):
        self.records = records
        self.sym, self.seps = st.text_from_records(records)
        self.sk = st.sort_keys(st.extract_keys(self.sym, self.seps))
        self.gmask, self.ghead = st.group_masks(self.sk, self.sym, self.seps)
        self.mi, self.mo = st.multi_in(self.gmask), st.multi_out(self.gmask)
        self.sp = self.blue = None
        if specials:
            spec = st.special_suffixes(self.sym, self.seps, self.sk)
            self.sp, self.blue = st.branch_codes(self.sym, self.seps, self.sk, self.gmask, spec)

    @property
    def n(self):
        return int(self.sym.size)

    @property
    def R(self):
        return int(self.seps.size)

    def stats(self):
        """the counts BwtBuilder.stats() reports (n_codes only when the branch codes were restated)"""
        out = {"n_keys": int(self.sk.size), "n_branch": int((self.ghead & (self.mi | self.mo)).sum()),
               "n_blue": int(self.mi.sum()) if self.blue is None else len(self.blue), "n_special": 32 * self.R}
        if self.sp is not None:
            out["n_codes"] = int(self.sp.size)
        return out

    def branch_table(self):
        """(k-mer << 2 | multi_in << 1 | multi_out, group head key index) of every branch k-mer, ascending"""
        sel = self.ghead & (self.mi | self.mo)
        ent = (self.sk[sel] & ~np.uint64(3)) | (self.mi[sel].astype(np.uint64) << np.uint64(1)) | self.mo[sel].astype(np.uint64)
        return ent, np.flatnonzero(sel).astype(np.uint64)

    def bwt(self, doubling=False):
        return doubling_bwt(self.sym) if doubling else coracle.bwt(self.sym)


# ---- inputs ------------------------------------------------------------------------------------------------------
def random_bases(rng, n):
    return BASES[rng.integers(0, 4, size=n)]


def repeat_rich(rng, n, el_len=300, copy_rate=0.7, muts=3):
    """n bases: copies of one element with a few point mutations each, between random stretches, so that branch k-mers,
    multi-key groups and blue segments occur all along the text"""
    master = random_bases(rng, el_len)
    parts, total = [], 0
    while total < n:
        if rng.random() < copy_rate:
            el = master.copy()
            el[rng.integers(0, el_len, size=muts)] = BASES[rng.integers(0, 4, size=muts)]
        else:
            el = random_bases(rng, int(rng.integers(50, 400)))
        parts.append(el)
        total += el.size
    return np.concatenate(parts)[:n]


def records_with_keys(n_keys, seed):
    """one repeat-rich record with exactly n_keys in-record windows"""
    return [bytes(repeat_rich(np.random.default_rng(seed), n_keys + 31))]


def straddling_repeat(seed=3):
    """three in-edge tiles and one key, every tile edge inside a k-mer group of several keys"""
    return records_with_keys(3 * ME_TILE + 1, seed)


def t_run_over_tile_edge():
    """a T run longer than one tile at the end of the sorted keys: a tile edge falls inside the T^31 group"""
    rng = np.random.default_rng(5)
    return [bytes(random_bases(rng, 3000)) + b"T" * 9000]


def aaaa_prefix_records(n_rec, length, seed):
    """A^(length - 28) + 28 random bases: every window starts with AAAA, so only the top digit of the keys is constant"""
    rng = np.random.default_rng(seed)
    return [b"A" * (length - 28) + bytes(random_bases(rng, 28)) for _ in range(n_rec)]


def text_hist_edge(minus):
    """four records with N == 2048 R (minus = 0) or one base fewer (minus = 1)"""
    rng = np.random.default_rng(17)
    recs = [repeat_rich(rng, TEXT_HIST_RATIO - 1, el_len=200) for _ in range(4)]
    recs[0] = recs[0][:recs[0].size - minus]
    return [bytes(r) for r in recs]


def over_tail_records(n_tail=ME_CAP + 4, n_x2=8):
    """n_tail records ending in c + X1 (X1 a 31-mer that occurs once inside the text), so one (c, tile) run of the in-edge
    join has more than ME_CAP duplicate sources c.X1, and one record holding c.X2_i for n_x2 31-mers X2_i just above X1
    whose groups exist: distinct sources with existing targets past ME_CAP in that run"""
    rng = np.random.default_rng(23)
    head = bytes(random_bases(rng, 27))
    x1 = head + b"AAAA"
    x2 = [head + bytes(BASES[[(i >> 6) & 3, (i >> 4) & 3, (i >> 2) & 3, i & 3]]) for i in range(1, n_x2 + 1)]
    c = b"G"
    recs = [bytes(random_bases(rng, 2)) + c + x1 for _ in range(n_tail)]
    special = bytes(random_bases(rng, 40)) + x1 + b"C"
    for x in x2:
        special += bytes(random_bases(rng, 40)) + c + x + b"C"
    recs.append(special + bytes(random_bases(rng, 40)))
    return recs


def k9_separator_records(sep_pos):
    """a separator at text position sep_pos (just before, at or after the last position of the first K9 tile), then
    three more records; repeat-rich, so that codes and blue entries occur in every tile"""
    rng = np.random.default_rng(sep_pos)
    return [bytes(repeat_rich(rng, sep_pos, el_len=200))] + [bytes(repeat_rich(rng, 3000, el_len=200)) for _ in range(3)]


def blue_fix_records(delta):
    """two records whose blue-entry count is nbw / 4 + delta (nbw = ceil(N / 32)): an A run of adjustable length inside
    random text makes the A^31 group multi-in with one entry per base of the run"""
    rng = np.random.default_rng(29)
    left, right, other = random_bases(rng, 9000), random_bases(rng, 9000), random_bases(rng, 20000)
    m = 400
    for _ in range(50):
        recs = [bytes(left) + b"A" * m + bytes(right), bytes(other)]
        rs = Restated(recs, specials=False)
        want = ((rs.n + 31) // 32) // BLUE_FIX_DIV + delta
        got = rs.stats()["n_blue"]
        if got == want:
            return recs
        m += want - got
    raise AssertionError("no A run gives the wanted blue-entry count")


def many_short_records(n_rec):
    """n_rec records of 33..80 bases, most of them variants of one sequence: 32 R sentinel suffixes with long ties"""
    rng = np.random.default_rng(n_rec)
    base = random_bases(rng, 80)
    recs = []
    for i in range(n_rec):
        if i % 3 == 0:
            recs.append(bytes(random_bases(rng, int(rng.integers(33, 81)))))
        else:
            r = base[:int(rng.integers(33, 81))].copy()
            r[int(rng.integers(0, r.size))] = BASES[int(rng.integers(0, 4))]
            recs.append(bytes(r))
    return recs


def k10_case(seed=41, unit_len=45, n_units=700):
    """Code strings for K10 alone: a repeated unit with a few flips (deep ties), '#' codes, one of them within the first
    27 codes of some entries of every segment, and '$' last; one segment of every size at and around each bin edge."""
    rng = np.random.default_rng(seed)
    unit = rng.integers(0, 4, size=unit_len).astype(np.uint8)
    codes = np.tile(unit, n_units)
    codes[rng.integers(0, codes.size, size=30)] ^= 1
    seps = rng.choice(codes.size - 40, size=25, replace=False)
    codes[seps] = 4
    codes = np.concatenate([codes, [5]]).astype(np.uint8)
    sizes = np.array(K10_SIZES)
    spi = []
    for s in sizes.tolist():
        pick = rng.choice(codes.size - 1, size=s, replace=False)
        near = np.array([p - d for p in seps[:3].tolist() for d in (0, 5, 26) if p - d >= 0])
        if s >= near.size:                                   # entries that meet a '#' within their first 27 codes
            pick = np.unique(np.concatenate([near, pick]))[:s]
            while pick.size < s:
                pick = np.unique(np.concatenate([pick, rng.choice(codes.size - 1, size=s - pick.size)]))
        spi.append(rng.permutation(pick))
    offs = np.concatenate(([0], np.cumsum(sizes))).astype(np.uint64)
    spi = np.concatenate(spi).astype(np.uint64)
    prev = rng.integers(0, 4, size=spi.size).astype(np.uint8)
    prev[rng.integers(0, spi.size, size=7)] = 4
    return codes, offs, spi, prev


K10_SIZES = [1, 2, 31, 32, 33, 127, 128, 129, 511, 512, 513, 4095, 4096, 4097]


def k10_expected_prev(codes, offs, spi, prev):
    """each segment's previous symbols in the order of its entries' code strings (suffix ranks of the code string)"""
    rank = suffix_ranks(codes)
    out = np.empty_like(prev)
    for s in range(offs.size - 1):
        lo, hi = int(offs[s]), int(offs[s + 1])
        order = np.argsort(rank[spi[lo:hi].astype(np.int64)], kind="stable")
        out[lo:hi] = prev[lo:hi][order]
    return out


# ---- the cases ---------------------------------------------------------------------------------------------------
class Case:
    """make() -> records; place(Restated) asserts the side of the threshold the input lies on.  codes: restate and compare
    the branch codes and blue entries (the sentinel sort of the restatement is plain Python: kept to R <= 64, and to the
    R = 512 / 513 sentinel-sort cases).  doubling: the reference BWT by suffix ranking (long runs).  bits: the key-index
    width the library must choose.  slow: large restatement."""

    def __init__(self, make, place, codes=True, doubling=False, bits=None, slow=False):
        self.make, self.place, self.codes, self.doubling, self.bits, self.slow = make, place, codes, doubling, bits, slow


def _keys_case(n_keys, bits, tiles, seed, straddle=False):
    def place(rs):
        assert rs.sk.size == n_keys and rs.R == 1
        assert key_index_bits(n_keys) == bits, "key-index width moved"
        assert -(-n_keys // ME_TILE) == tiles, "in-edge tile count moved"
        assert k9_one_record_tiles(rs.seps, rs.n).all()           # K9: one record over every tile
        if straddle:                                              # every inner tile edge falls inside a group of several keys
            for a in range(ME_TILE, n_keys - 1, ME_TILE):
                assert not rs.ghead[a] and rs.sk[a - 1] >> np.uint64(2) == rs.sk[a] >> np.uint64(2), a
    make = (lambda: straddling_repeat(seed)) if straddle else (lambda: records_with_keys(n_keys, seed))
    return Case(make, place, bits=bits)


def _place_t_run(rs):
    # a tile edge inside the T^31 group: the join's tile bound takes the (k[a-1] >> 2) + 1 overflow branch
    assert rs.sk.size > ME_TILE
    assert int(rs.sk[ME_TILE - 1] >> np.uint64(2)) == T31 and int(rs.sk[ME_TILE] >> np.uint64(2)) == T31


def _sort_case(sweeps, text_hist):
    def place(rs):
        assert sort_sweeps(rs.sk) == sweeps and last_pass_skipped(rs.sk)
        assert text_hist_applies(rs.n, rs.R) == text_hist
    return place


def _text_hist_case(minus):
    def place(rs):
        assert rs.n == TEXT_HIST_RATIO * rs.R - minus
        assert text_hist_applies(rs.n, rs.R) == (minus == 0)
    return Case(lambda: text_hist_edge(minus), place)


def _over_case(marks_in_tail):
    def place(rs):
        over = [r for r in edge_runs(rs.sk) if r[3] - r[2] > ME_CAP]
        assert over, "no in-edge run longer than ME_CAP"
        marks = sum(r[4] for r in over)
        assert marks >= 8 if marks_in_tail else marks == 0, marks
    return place


def _k9_case(sep_pos, flags):
    def place(rs):
        assert int(rs.seps[0]) == sep_pos
        assert k9_one_record_tiles(rs.seps, rs.n)[:2].tolist() == flags
    return Case(lambda: k9_separator_records(sep_pos), place)


def _blue_fix_case(delta):
    def place(rs):
        nbw = (rs.n + 31) // 32
        assert rs.stats()["n_blue"] == nbw // BLUE_FIX_DIV + delta
        assert (rs.stats()["n_blue"] >= nbw // BLUE_FIX_DIV) == (delta >= 0)
    return Case(lambda: blue_fix_records(delta), place)


def _special_case(n_rec, all_pairs):
    def place(rs):
        assert rs.R == n_rec and (32 * rs.R <= SPECIAL_ALL_PAIRS) == all_pairs
    return Case(lambda: many_short_records(n_rec), place)


CASES = {
    # key-index width (8 keys per bucket) and in-edge tiles (ME_TILE keys)
    "keys_2048": _keys_case(2048, 8, 1, 1),
    "keys_2049": _keys_case(2049, 9, 1, 2),
    "keys_8191": _keys_case(ME_TILE - 1, 10, 1, 3),
    "keys_8192": _keys_case(ME_TILE, 10, 1, 4),
    "keys_8193": _keys_case(ME_TILE + 1, 11, 2, 5),
    "keys_24575": _keys_case(3 * ME_TILE - 1, 12, 3, 6),
    "keys_24576": _keys_case(3 * ME_TILE, 12, 3, 7),
    "keys_24577_straddle": _keys_case(3 * ME_TILE + 1, 12, 4, 3, straddle=True),
    "keys_32767": _keys_case(4 * ME_TILE - 1, 12, 4, 8),
    "keys_32769": _keys_case(4 * ME_TILE + 1, 13, 5, 9),
    "t_run_over_tile_edge": Case(t_run_over_tile_edge, _place_t_run),
    # last sort pass skipped: the key index is built by key_index_mark_kernel; with and without the text histogram
    "aaaa_1x100k": Case(lambda: aaaa_prefix_records(1, 100_000, 11), _sort_case(7, True), doubling=True),
    "aaaa_60x1500": Case(lambda: aaaa_prefix_records(60, 1500, 12), _sort_case(7, False), doubling=True),
    "homopolymer_5000": Case(lambda: [b"A" * 5000], _sort_case(0, True), doubling=True),
    # digit histogram from the text: N == 2048 R and one base fewer
    "text_hist_on": _text_hist_case(0),
    "text_hist_off": _text_hist_case(1),
    # in-edge runs longer than ME_CAP: a tail of duplicates only, and a tail that marks in-edges
    "a_70000": Case(lambda: [b"A" * 70_000], _over_case(False), doubling=True),
    "over_tail_marks": Case(over_tail_records, _over_case(True), codes=False, slow=True),
    # K9: a separator just before, at and just after the last position of the first tile
    "k9_sep_4094": _k9_case(K9_TILE_POS - 2, [False, False]),
    "k9_sep_4095": _k9_case(K9_TILE_POS - 1, [True, False]),
    "k9_sep_4096": _k9_case(K9_TILE_POS, [True, False]),
    # K9 blue fix: plain below nbw / 4 entries, interleaved from there
    "blue_fix_plain": _blue_fix_case(-1),
    "blue_fix_interleaved": _blue_fix_case(0),
    # sentinel suffixes: all-pairs ranking up to 16384 of them, bitonic network beyond
    "special_512": _special_case(512, True),
    "special_513": _special_case(513, False),
}
