"""CPU references for SMEM search (debwt_index_smem), independent of the CUDA path:
  * the definition by brute force over the bytes of T: start(e) = the smallest s for which read[s, e) is made of A/C/G/T
    and occurs in T (e if none), SMEMs = [start(e), e) with start(e) < e and (e = m or start(e + 1) > start(e));
  * Li's definition (2012): the maximal exact matches that no other one contains;
  * a model of the FMD-index search over the oracle's BWT (oracle/bwt_oracle.c): bi-interval extension with '#' and '$'
    sorting after T, and Li's smem1 loop with min_intv = 1, over occ / C counted here from that BWT;
  * the definition again through a count oracle alone (binary search of start(e)), for texts too large for the model."""
import numpy as np

from oracle import coracle

_CODE = np.full(256, 4, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _i
    _CODE[_c | 0x20] = _i
_RC = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")


def codes(read: bytes) -> list:
    """A, C, G, T (either case) -> 0..3, anything else -> 4"""
    return _CODE[np.frombuffer(bytes(read), dtype=np.uint8)].tolist()


def revcomp(read: bytes) -> bytes:
    """reverse complement of a read; case kept, other symbols stay as they are"""
    return bytes(read).translate(_RC)[::-1]


# ---- brute force ------------------------------------------------------------------------------------------------------
def _occurs(read: bytes, s: int, e: int, text: bytes) -> bool:
    piece = bytes(read[s:e]).upper()
    return not piece.translate(None, b"ACGT") and piece in text


def starts(read: bytes, text: bytes) -> list:
    """start(e) for e = 0 .. m; `text` is T in upper case.  A match's pieces match too, so start(e) does not decrease"""
    out, s = [0], 0
    for e in range(1, len(read) + 1):
        while s < e and not _occurs(read, s, e, text):
            s += 1
        out.append(s)
    return out


def smems_from_starts(st: list) -> list:
    m = len(st) - 1
    return [(st[e], e) for e in range(1, m + 1) if st[e] < e and (e == m or st[e + 1] > st[e])]


def brute_smems(read: bytes, text: bytes) -> list:
    """[(qbeg, qend)] ascending, by the start(e) definition"""
    return smems_from_starts(starts(read, text))


def li_smems(read: bytes, text: bytes) -> list:
    """[(qbeg, qend)] ascending: the MEMs (matches that extend neither left nor right) not contained in another MEM"""
    m = len(read)
    mems = []
    for s in range(m):
        e = s
        while e < m and _occurs(read, s, e + 1, text):
            e += 1
        if e > s and (s == 0 or not _occurs(read, s - 1, e, text)):
            mems.append((s, e))
    return sorted(a for a in mems if not any(b != a and b[0] <= a[0] and a[1] <= b[1] for b in mems))


# ---- the FMD-index model ---------------------------------------------------------------------------------------------
class FmdModel:
    """Bi-intervals (k, l, s): rows [k, k + s) start with P, [l, l + s) with rc(P); valid over a text closed under reverse
    complement.  Rows follow the reference's suffix order, A < C < G < T < '#' < '$'."""

    def __init__(self, sym: np.ndarray):
        bwt = coracle.bwt_symbols(np.ascontiguousarray(sym, dtype=np.uint8))
        self.n = int(bwt.size)
        self.occ = np.zeros((self.n + 1, 4), dtype=np.int64)          # occ[r][c] = rows < r holding base c
        for c in range(4):
            np.cumsum(bwt == c, out=self.occ[1:, c])
        tot = self.occ[-1].tolist()
        self.C = [0, tot[0], tot[0] + tot[1], tot[0] + tot[1] + tot[2], sum(tot), self.n - 1]

    def empty(self):
        return (0, 0, self.n)

    def single(self, a):
        return (self.C[a], self.C[3 - a], self.C[a + 1] - self.C[a])

    def backward(self, iv, a):
        """P -> aP"""
        k, l, s = iv
        lo, hi = self.occ[k].tolist(), self.occ[k + s].tolist()
        sz = [hi[c] - lo[c] for c in range(4)]
        l_t = l
        l_g = l_t + sz[3]
        l_c = l_g + sz[2]
        l_a = l_c + sz[1]
        return (self.C[a] + lo[a], (l_a, l_c, l_g, l_t)[a], sz[a])

    def forward(self, iv, a):
        """P -> Pa: backward extension of rc(P) by comp(a), starts swapped back"""
        k, l, s = self.backward((iv[1], iv[0], iv[2]), 3 - a)
        return (l, k, s)

    def smem1(self, q: list, x: int, out: list) -> int:
        """Li's smem1 (BWA's bwt_smem1a with min_intv = 1) from q[x], a base that occurs in T.  Appends (qbeg, qend, k, l, s)
        by descending qbeg; returns the end of the longest match from x."""
        ik, end = self.single(q[x]), x + 1
        curr = []
        i = x + 1
        while i < len(q):
            if q[i] > 3:
                curr.append((ik, end))
                break
            ok = self.forward(ik, q[i])
            if ok[2] != ik[2]:
                curr.append((ik, end))
                if ok[2] == 0:
                    break
            ik, end = ok, i + 1
            i += 1
        if i == len(q):
            curr.append((ik, end))
        prev = curr[::-1]                                             # longest match first
        ret = prev[0][1]
        last_beg = None
        for i in range(x - 1, -2, -1):
            c = q[i] if i >= 0 else 4
            curr = []
            for p, pend in prev:
                ok = self.backward(p, c) if c < 4 else None
                if ok is None or ok[2] == 0:
                    if not curr and (last_beg is None or i + 1 < last_beg):
                        last_beg = i + 1
                        out.append((i + 1, pend) + p)
                elif not curr or ok[2] != curr[-1][0][2]:
                    curr.append((ok, pend))
            if not curr:
                break
            prev = curr
        return ret

    def smems(self, read: bytes, min_len: int = 1) -> list:
        """[(qbeg, qend, row, rc_row, count)] with qend - qbeg >= min_len, ascending"""
        q = codes(read)
        res, x = [], 0
        while x < len(q):
            if q[x] > 3 or self.single(q[x])[2] == 0:                 # no match covers x
                x += 1
                continue
            out = []
            x = self.smem1(q, x, out)
            res += [r for r in reversed(out) if r[1] - r[0] >= min_len]
        return res

    def interval(self, pattern: bytes):
        """the bi-interval of a pattern by backward extension from the empty one"""
        iv = self.empty()
        for a in reversed(codes(pattern)):
            iv = self.backward(iv, a)
        return iv


# ---- the definition through a count oracle ------------------------------------------------------------------------------
def smems_by_count(count, reads: list, min_len: int = 1) -> list:
    """[[(qbeg, qend, count)]] per read from `count(patterns) -> counts` alone: start(e) by binary search (a piece of a
    match matches too, so count(read[s:e]) > 0 holds from start(e) to e), then the SMEM rule and their counts."""
    items = [(i, e) for i, q in enumerate(reads) for e in range(1, len(q) + 1)]
    lo = np.zeros(len(items), dtype=np.int64)
    hi = np.array([e for _, e in items], dtype=np.int64)
    while True:
        act = np.flatnonzero(lo < hi)
        if act.size == 0:
            break
        mid = (lo[act] + hi[act]) // 2
        got = count([bytes(reads[items[j][0]][int(s):items[j][1]]) for j, s in zip(act.tolist(), mid.tolist())])
        hit = np.asarray(got) > 0
        hi[act[hit]] = mid[hit]
        lo[act[~hit]] = mid[~hit] + 1
    st = [[0] for _ in reads]
    for (i, _), s in zip(items, lo.tolist()):
        st[i].append(s)
    sm = [[x for x in smems_from_starts(s) if x[1] - x[0] >= min_len] for s in st]
    flat = [bytes(reads[i][s:e]) for i, lst in enumerate(sm) for s, e in lst]
    cnt = np.asarray(count(flat)).tolist() if flat else []
    out, j = [], 0
    for lst in sm:
        out.append([(s, e, int(cnt[j + t])) for t, (s, e) in enumerate(lst)])
        j += len(lst)
    return out
