"""CPU reference of BWA-MEM's seed extension (debwt_index_regions), independent of the CUDA path: bwa 0.7.17's
ksw_extend2, the score of ksw_align2, cal_max_gap, bns_fetch_seq's clip, mem_seed_sw, mem_flt_chained_seeds and
mem_chain2aln as include/debwt_b200.h restates them, over any (chains, chain seeds) in the layout of
tests/chain_ref.reference (or BwtBuilder.chains through chain_ref.as_tuples), the reads and the records.

The two DP routines exist twice: cell-by-cell Python loops here, and a scalar C twin (tests/ext_dp.c) that the
reference calls, since the GPU tests' read mixes are too large for Python loops.  The CPU tests check that they agree."""
import ctypes
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

DEFAULTS = dict(a=1, b=4, o_del=6, e_del=1, o_ins=6, e_ins=1, pen_clip5=5, pen_clip3=5, zdrop=100)
F32 = np.float32

_NT4 = np.full(256, 4, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _NT4[_c] = _NT4[_c | 0x20] = _i


def nt4(read) -> np.ndarray:
    """read symbols A, C, G, T in either case to 0..3, anything else to 4"""
    return _NT4[np.frombuffer(bytes(read), dtype=np.uint8)]


def score(o, t, q):
    return -1 if q > 3 else o["a"] if t == q else -o["b"]


# ---- the DP, cell by cell ---------------------------------------------------------------------------------------------
def extend_py(q, t, w, end_bonus, h0, o):
    """ksw_extend2: (max, qle, tle, gtle, gscore, max_off)"""
    qlen, tlen = len(q), len(t)
    oe_del, oe_ins, e_del, e_ins = o["o_del"] + o["e_del"], o["o_ins"] + o["e_ins"], o["e_del"], o["e_ins"]
    H, E = [0] * (qlen + 2), [0] * (qlen + 2)
    H[0] = h0
    if qlen >= 1:
        H[1] = h0 - oe_ins if h0 > oe_ins else 0
    j = 2
    while j <= qlen and H[j - 1] > e_ins:
        H[j] = H[j - 1] - e_ins
        j += 1
    max_ins = max(int((qlen * o["a"] + end_bonus - o["o_ins"]) / e_ins + 1.), 1)
    max_del = max(int((qlen * o["a"] + end_bonus - o["o_del"]) / e_del + 1.), 1)
    w = min(w, max_ins, max_del)
    mx, max_i, max_j, max_ie, gscore, max_off, beg, end = h0, -1, -1, -1, -1, 0, 0, qlen
    for i in range(tlen):
        beg = max(beg, i - w)
        end = min(end, i + w + 1, qlen)
        h1 = max(0, h0 - (o["o_del"] + e_del * (i + 1))) if beg == 0 else 0
        f = m = 0
        mj = -1
        j = beg
        while j < end:
            M, e = H[j], E[j]
            H[j] = h1
            M = M + score(o, t[i], q[j]) if M else 0
            h = max(M, e, f)
            h1 = h
            if m <= h:
                mj, m = j, h
            E[j] = max(e - e_del, M - oe_del, 0)
            f = max(f - e_ins, M - oe_ins, 0)
            j += 1
        H[end], E[end] = h1, 0
        if j == qlen:
            max_ie = max_ie if gscore > h1 else i
            gscore = max(gscore, h1)
        if m == 0:
            break
        if m > mx:
            mx, max_i, max_j = m, i, mj
            max_off = max(max_off, abs(mj - i))
        elif o["zdrop"] > 0:
            di, dj = i - max_i, mj - max_j
            if di > dj:
                if mx - m - (di - dj) * e_del > o["zdrop"]:
                    break
            elif mx - m - (dj - di) * e_ins > o["zdrop"]:
                break
        j = beg
        while j < end and H[j] == 0 and E[j] == 0:
            j += 1
        beg = j
        j = end
        while j >= beg and H[j] == 0 and E[j] == 0:
            j -= 1
        end = min(j + 2, qlen)
    return mx, max_j + 1, max_i + 1, max_ie + 1, gscore, max_off


def seed_sw_py(q, t, o):
    """ksw_align2's score: Gotoh local alignment, H >= 0, gaps open from H"""
    qlen = len(q)
    oe_del, oe_ins = o["o_del"] + o["e_del"], o["o_ins"] + o["e_ins"]
    Hp, E = [0] * (qlen + 1), [0] * qlen                 # Hp[j + 1] = H(i - 1, j)
    best = 0
    for ti in t:
        Hc = [0] * (qlen + 1)
        f = 0
        for j in range(qlen):
            f = 0 if j == 0 else max(f - o["e_ins"], Hc[j] - oe_ins, 0)
            h = max(Hp[j] + score(o, ti, q[j]), E[j], f, 0)
            best = max(best, h)
            E[j] = max(E[j] - o["e_del"], h - oe_del, 0)
            Hc[j + 1] = h
        Hp = Hc
    return best


# ---- the C twin -------------------------------------------------------------------------------------------------------
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ext_dp.c")
        tag = hashlib.sha256(open(src, "rb").read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"debwt_ext_dp_{os.getuid()}_{tag}.so")
        if not os.path.isfile(so):
            tmp = so + f".{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-Wall", "-shared", "-fPIC", "-o", tmp, src])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        vp, i = ctypes.c_void_p, ctypes.c_int
        L.ext_extend.argtypes = [i, vp, i, vp] + [i] * 10 + [vp]
        L.ext_extend.restype = i
        L.ext_seed_sw.argtypes = [i, vp, i, vp] + [i] * 6
        L.ext_seed_sw.restype = i
        L.ext_cells.restype = ctypes.c_ulonglong
        _LIB = L
    return _LIB


def cells() -> int:
    """DP cells the C twin has computed so far (extension rows' band cells and seed SW's full matrices)"""
    return int(_lib().ext_cells())


def _u8(x):
    return np.ascontiguousarray(np.asarray(x, dtype=np.uint8))


def extend_c(q, t, w, end_bonus, h0, o):
    q, t = _u8(q), _u8(t)
    out = np.zeros(5, dtype=np.int32)
    mx = _lib().ext_extend(q.size, q.ctypes.data, t.size, t.ctypes.data, o["a"], o["b"], o["o_del"], o["e_del"], o["o_ins"], o["e_ins"], w,
                           end_bonus, o["zdrop"], h0, out.ctypes.data)
    return (mx,) + tuple(int(x) for x in out)


def seed_sw_c(q, t, o):
    q, t = _u8(q), _u8(t)
    return _lib().ext_seed_sw(q.size, q.ctypes.data, t.size, t.ctypes.data, o["a"], o["b"], o["o_del"], o["e_del"], o["o_ins"], o["e_ins"])


# ---- the reference sequence (bwa's pac) --------------------------------------------------------------------------------
class Pac:
    """the forward records of a both_strands text (ASCII `text`, separators `seps`) as bwa's pac"""

    def __init__(self, text, seps):
        text = np.asarray(text, dtype=np.uint8)
        seps = np.asarray(seps, dtype=np.int64)
        R = seps.size
        starts = np.concatenate(([0], seps[:-1] + 1))
        self.half = R // 2
        self.fwd = np.concatenate([_NT4[text[starts[r]:seps[r]]] for r in range(self.half)] or [np.zeros(0, np.uint8)])
        self.l_pac = int(self.fwd.size)
        self.F = [int(starts[r] - r) for r in range(self.half)]
        self.len = [int(seps[r] - starts[r]) for r in range(self.half)]
        assert self.l_pac == (int(seps[-1]) + 1 - R) // 2

    def seq(self, beg, end):
        """bwa's bns_get_seq of [beg, end) (one strand)"""
        if beg >= end:
            return np.zeros(0, dtype=np.uint8)
        if beg >= self.l_pac:
            lo, hi = 2 * self.l_pac - end, 2 * self.l_pac - beg
            return (3 - self.fwd[lo:hi])[::-1]
        return self.fwd[beg:end]

    def clip(self, rec, beg, mid, end):
        """bns_fetch_seq's clip of [beg, end) to record `rec` on mid's strand"""
        fb, fe = self.F[rec], self.F[rec] + self.len[rec]
        if mid >= self.l_pac:
            fb, fe = 2 * self.l_pac - fe, 2 * self.l_pac - fb
        return max(beg, fb), min(end, fe)


def cal_max_gap(o, w, qlen):
    l_del = int((qlen * o["a"] - o["o_del"]) / o["e_del"] + 1.)
    l_ins = int((qlen * o["a"] - o["o_ins"]) / o["e_ins"] + 1.)
    return min(max(l_del, l_ins, 1), w << 1)


def seed_sw(o, pac, q, L, s, rec, dp=seed_sw_c):
    """mem_seed_sw of seed s = (rbeg, qbeg, len): -1 or the local score"""
    rbeg, qbeg, ln = s
    if ln >= 200:
        return -1
    qb, qe = max(qbeg - 50, 0), min(qbeg + ln + 50, L)
    rb, re = max(rbeg - 50, 0), min(rbeg + ln + 50, 2 * pac.l_pac)
    mid = (rbeg + rbeg + ln) >> 1
    if rb < pac.l_pac < re:
        if mid < pac.l_pac:
            re = pac.l_pac
        else:
            rb = pac.l_pac
    if qe - qb >= 200 or re - rb >= 200:
        return -1
    rb, re = pac.clip(rec, rb, mid, re)
    return dp(q[qb:qe], pac.seq(rb, re), o)


def flt_chained_seeds(o, pac, q, L, chains, min_chain_weight=0, dp=seed_sw_c):
    """mem_flt_chained_seeds: per chain [(rbeg, qbeg, len, score)]; also whether the filter ran"""
    min_l = float(F32(1.1) * F32(min_chain_weight)) if min_chain_weight else float(F32(5.5)) * math.log(L)
    min_hsp = int(o["a"] * min_l + .499)
    if min_l > float(F32(0.05) * F32(L)):
        return [[s + (s[2],) for s in c["seeds"]] for c in chains], False
    out = []
    for c in chains:
        kept = []
        for s in c["seeds"]:
            sc = seed_sw(o, pac, q, L, s, c["record"], dp)
            if sc < 0 or sc >= min_hsp:
                kept.append(s + (s[2] * o["a"] if sc < 0 else sc,))
        out.append(kept)
    return out, True


def _run_band(o, w, q, t, end_bonus, h0, prev, dp, trace):
    aw = w
    for i in range(2):
        aw = w << i
        x = dp(q, t, aw, end_bonus, h0, o)
        if trace is not None:
            trace.append(("try", i))
        if x[0] == prev or x[5] < (aw >> 1) + (aw >> 2):
            break
        prev = x[0]
    return x, aw


def chain2aln(o, w, pac, q, L, c, seeds, regs, ci, dp=extend_c, trace=None):
    """mem_chain2aln of chain c (its record, strand, frac_rep) with its filtered seeds [(rbeg, qbeg, len, score)];
    appends to regs (dicts).  trace (a list) receives the branches taken."""
    n = len(seeds)
    if n == 0:
        if trace is not None:
            trace.append("empty")
        return
    l_pac = pac.l_pac
    rmax0, rmax1 = 2 * l_pac, 0
    for rb, qb, ln, _ in seeds:
        r = L - qb - ln
        rmax0 = min(rmax0, rb - (qb + cal_max_gap(o, w, qb)))
        rmax1 = max(rmax1, rb + ln + (r + cal_max_gap(o, w, r)))
    rmax0, rmax1 = max(rmax0, 0), min(rmax1, 2 * l_pac)
    if rmax0 < l_pac < rmax1:
        if trace is not None:
            trace.append("cross")
        if seeds[0][0] < l_pac:
            rmax1 = l_pac
        else:
            rmax0 = l_pac
    c0 = (rmax0, rmax1)
    rmax0, rmax1 = pac.clip(c["record"], rmax0, seeds[0][0], rmax1)
    if trace is not None and (rmax0, rmax1) != c0:
        trace.append("clip")
    rseq = pac.seq(rmax0, rmax1)
    srt = sorted((sc << 32 | i) for i, (_, _, _, sc) in enumerate(seeds))
    for k in range(n - 1, -1, -1):
        srb, sq, sl, _ = seeds[srt[k] & 0xFFFFFFFF]
        covered = False
        for p in regs:
            if srb < p["rb"] or srb + sl > p["re"] or sq < p["qb"] or sq + sl > p["qe"]:
                continue
            if sl - p["seedlen0"] > .1 * L:
                continue
            qd, rd = sq - p["qb"], srb - p["rb"]
            wd = min(cal_max_gap(o, w, min(qd, rd)), p["w"])
            if qd - rd < wd and rd - qd < wd:
                covered = True
                break
            qd, rd = p["qe"] - (sq + sl), p["re"] - (srb + sl)
            wd = min(cal_max_gap(o, w, min(qd, rd)), p["w"])
            if qd - rd < wd and rd - qd < wd:
                covered = True
                break
        if covered:
            ov = False
            for i in range(k + 1, n):
                if srt[i] == 0:
                    continue
                trb, tq, tl, _ = seeds[srt[i] & 0xFFFFFFFF]
                if tl < sl * .95:
                    continue
                if sq <= tq and sq + sl - tq >= sl >> 2 and tq - sq != trb - srb:
                    ov = True
                    break
                if tq <= sq and tq + tl - sq >= sl >> 2 and sq - tq != srb - trb:
                    ov = True
                    break
            if not ov:
                srt[k] = 0
                if trace is not None:
                    trace.append("skip")
                continue
            if trace is not None:
                trace.append("revived")
        a = dict(w=w)
        aw0 = aw1 = w
        if sq:
            qs = q[:sq][::-1]
            ts = rseq[:srb - rmax0][::-1]
            x, aw0 = _run_band(o, w, qs, ts, o["pen_clip5"], sl * o["a"], -1, dp, trace)
            sc = x[0]
            if x[4] <= 0 or x[4] <= sc - o["pen_clip5"]:
                a["qb"], a["rb"], truesc = sq - x[1], srb - x[2], sc
                tag = "left_local"
            else:
                a["qb"], a["rb"], truesc = 0, srb - x[3], x[4]
                tag = "left_end"
            if trace is not None:
                trace.append(tag)
                if aw0 != w:
                    trace.append("retry")
        else:
            sc = truesc = sl * o["a"]
            a["qb"], a["rb"] = 0, srb
            if trace is not None:
                trace.append("qbeg0")
        if sq + sl != L:
            sc0, qe0, re0 = sc, sq + sl, srb + sl - rmax0
            x, aw1 = _run_band(o, w, q[qe0:], rseq[re0:], o["pen_clip3"], sc0, sc0, dp, trace)
            sc = x[0]
            if x[4] <= 0 or x[4] <= sc - o["pen_clip3"]:
                a["qe"], a["re"] = qe0 + x[1], rmax0 + re0 + x[2]
                truesc += sc - sc0
                tag = "right_local"
            else:
                a["qe"], a["re"] = L, rmax0 + re0 + x[3]
                truesc += x[4] - sc0
                tag = "right_end"
            if trace is not None:
                trace.append(tag)
                if aw1 != w:
                    trace.append("retry")
        else:
            a["qe"], a["re"] = L, srb + sl
            if trace is not None:
                trace.append("qend_L")
        a["seedcov"] = sum(tl for trb, tq, tl, _ in seeds
                           if tq >= a["qb"] and tq + tl <= a["qe"] and trb >= a["rb"] and trb + tl <= a["re"])
        a.update(score=sc, truesc=truesc, w=max(aw0, aw1), seedlen0=sl, chain=ci, record=c["record"], strand=c["strand"],
                 frac_rep=c["frac_rep"])
        regs.append(a)


FIELDS = ("rb", "re", "qb", "qe", "score", "truesc", "w", "seedcov", "seedlen0", "chain", "record", "strand", "frac_rep")


def read_regions(o, w, pac, read, chains, min_chain_weight=0, dp=extend_c, sw=seed_sw_c, trace=None):
    """mem_flt_chained_seeds then mem_chain2aln over one read's chains [{"seeds": [(rbeg, qbeg, len)], "record",
    "strand", "frac_rep"}] in filter order: its regions as dicts"""
    q = nt4(read)
    L = len(q)
    if not chains:
        return []
    fl, ran = flt_chained_seeds(o, pac, q, L, chains, min_chain_weight, sw)
    if trace is not None:
        trace.append("flt" if ran else "noflt")
        if ran and sum(len(c["seeds"]) for c in chains) != sum(len(s) for s in fl):
            trace.append("dropped")
    regs = []
    for ci, (c, seeds) in enumerate(zip(chains, fl)):
        chain2aln(o, w, pac, q, L, c, seeds, regs, ci, dp, trace)
    return regs


def reference(offsets, chains, cseeds, reads, text, seps, w=100, min_chain_weight=0, trace=None, **opts):
    """(offsets, [tuples in FIELDS order]) as debwt_index_regions lays them out, from chains / chain seeds in the layout of
    tests/chain_ref.reference"""
    o = {**DEFAULTS, **{k: v for k, v in opts.items() if k in DEFAULTS}}
    pac = Pac(text, seps)
    offs, out = [0], []
    for i, read in enumerate(reads):
        cs = [dict(seeds=[tuple(s) for s in cseeds[c[1]:c[1] + c[2]]], record=c[4], strand=c[5], frac_rep=c[7])
              for c in chains[offsets[i]:offsets[i + 1]]]
        for a in read_regions(o, w, pac, read, cs, min_chain_weight, trace=trace):
            out.append(tuple(float(F32(a[f])) if f == "frac_rep" else int(a[f]) for f in FIELDS))
        offs.append(len(out))
    return offs, out


def as_tuples(regions):
    """REGION_DTYPE array in the layout of `reference`"""
    return [tuple(float(x[f]) if f == "frac_rep" else int(x[f]) for f in FIELDS) for x in regions]
