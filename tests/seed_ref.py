"""CPU reference of BWA-MEM's seed collection (debwt_index_seeds), independent of the CUDA path: bwa's mem_collect_intv
(round 1 SMEMs, round 2 re-seeding, round 3 LAST-like seeds), its order and the SA sampling of mem_chain, restated over
the FMD-index model of tests/smem_ref.py; and the definitions the restatement is checked against, from the bytes of T."""
import numpy as np

from tests.smem_ref import codes

DEFAULTS = dict(min_len=19, split_factor=1.5, split_width=10, max_mem_intv=20, max_occ=500)


def split_len(min_len: int, split_factor: float) -> int:
    """bwa's (int)(min_seed_len * split_factor + .499): a float product, the sum in double"""
    return int(float(np.float32(min_len) * np.float32(split_factor)) + 0.499)


def smem1(model, q: list, x: int, out: list, min_intv: int = 1) -> int:
    """bwa's bwt_smem1a(x, min_intv, max_intv = 0) over `model` (tests/smem_ref.FmdModel) from q[x], a base that occurs in
    T: FmdModel.smem1 with its two "size 0" tests read as "size below min_intv".  Appends (qbeg, qend, k, l, s) by
    descending qbeg; returns the end of the longest match from x."""
    ik, end = model.single(q[x]), x + 1
    curr = []
    i = x + 1
    while i < len(q):
        if q[i] > 3:
            curr.append((ik, end))
            break
        ok = model.forward(ik, q[i])
        if ok[2] != ik[2]:
            curr.append((ik, end))
            if ok[2] < min_intv:
                break
        ik, end = ok, i + 1
        i += 1
    if i == len(q):
        curr.append((ik, end))
    prev = curr[::-1]                                                 # longest match first
    ret = prev[0][1]
    last_beg = None
    for i in range(x - 1, -2, -1):
        c = q[i] if i >= 0 else 4
        curr = []
        for p, pend in prev:
            ok = model.backward(p, c) if c < 4 else None
            if ok is None or ok[2] < min_intv:
                if not curr and (last_beg is None or i + 1 < last_beg):
                    last_beg = i + 1
                    out.append((i + 1, pend) + p)
            elif not curr or ok[2] != curr[-1][0][2]:
                curr.append((ok, pend))
        if not curr:
            break
        prev = curr
    return ret


def _round3(q: list, single, extend, min_len: int, max_mem_intv: int) -> list:
    """bwa's bwt_seed_strategy1 loop: [(qbeg, qend, interval)] of the seeds that occur"""
    out, x, m = [], 0, len(q)
    while x < m:
        if q[x] > 3 or single(q[x])[-1] == 0:                         # a base T lacks: stepped over as in round 1
            x += 1
            continue
        ik, nxt = single(q[x]), m
        for i in range(x + 1, m):
            if q[i] > 3:
                nxt = i + 1
                break
            ik = extend(ik, q[i], x, i + 1)
            if ik[-1] < max_mem_intv and i - x >= min_len:
                if ik[-1] > 0:
                    out.append((x, i + 1, ik))
                nxt = i + 1
                break
        x = nxt
    return out


def seeds(model, read: bytes, min_len=19, split_factor=1.5, split_width=10, max_mem_intv=20, **_) -> list:
    """[(qbeg, qend, round, row, rc_row, count)] of one read in ascending (qbeg, qend, round)"""
    q = codes(read)
    r1 = model.smems(read, min_len)
    out = [(b, e, 1, k, l, s) for b, e, k, l, s in r1]
    sl = split_len(min_len, split_factor)
    for b, e, _, _, s in r1:
        if e - b >= sl and s <= split_width:
            got = []
            smem1(model, q, (b + e) >> 1, got, s + 1)
            out += [(b2, e2, 2, k2, l2, s2) for b2, e2, k2, l2, s2 in got if e2 - b2 >= min_len]
    if max_mem_intv > 0:
        r3 = _round3(q, model.single, lambda iv, a, lo, hi: model.forward(iv, a), min_len, max_mem_intv)
        out += [(b, e, 3) + iv for b, e, iv in r3]
    return sorted(out, key=lambda t: t[:3])


def hit_rows(row: int, count: int, max_occ: int) -> list:
    """bwa's mem_chain: min(count, max_occ) rows, every step-th from row, step = count // max_occ when count > max_occ"""
    step = count // max_occ if count > max_occ else 1
    return [row + j * step for j in range(min(count, max_occ))]


def reference(model, sa, seps, reads: list, max_occ=500, **opts):
    """(offsets, [(qbeg, qend, round, row, rc_row, count, hit_begin, n_hits)], [(pos, offset, record, strand)]) as
    debwt_index_seeds lays them out; sa: row -> text position, seps: the separators of the both-strands text"""
    from debwt_b200 import api
    offs, out, hits = [0], [], []
    for q in reads:
        for b, e, r, k, l, s in seeds(model, q, **opts):
            rows = hit_rows(k, s, max_occ)
            pos = np.asarray([sa[x] for x in rows], dtype=np.uint64)
            rec, strand, off = api.strand_offsets(pos, e - b, seps)
            out.append((b, e, r, k, l, s, len(hits), len(rows)))
            hits += list(zip(pos.tolist(), off.tolist(), rec.tolist(), strand.tolist()))
        offs.append(len(out))
    return offs, out, hits


# ---- definitions from the bytes of T --------------------------------------------------------------------------------------
def count_in(text: bytes, piece: bytes, stop: int = -1) -> int:
    """occurrences of an A/C/G/T piece in T (overlapping; counting stops at `stop` when it is given); 0 for anything else"""
    if not piece or piece.translate(None, b"ACGT"):
        return 0
    n, i = 0, text.find(piece)
    while i >= 0 and n != stop:
        n += 1
        i = text.find(piece, i + 1)
    return n


def smem1_by_definition(read: bytes, text: bytes, x: int, t: int) -> list:
    """[(qbeg, qend)] ascending: the pieces read[b, e) with b <= x < e, made of A/C/G/T, that occur at least t times in T
    and are contained in no other such piece"""
    r = bytes(read).upper()
    ok = []
    for b in range(x + 1):                                            # the longest such piece from b: a longer one occurs less
        e = x
        while e < len(r) and count_in(text, r[b:e + 1], t) >= t:
            e += 1
        if e > x:
            ok.append((b, e))
    return sorted(p for p in ok if not any(o != p and o[0] <= p[0] and p[1] <= o[1] for o in ok))


def round3_by_walk(read: bytes, text: bytes, min_len: int, max_mem_intv: int) -> list:
    """[(qbeg, qend, count)] of round 3 by its rule, every count taken from the text"""
    r = bytes(read).upper()
    q = codes(read)
    single = lambda a: (count_in(text, b"ACGT"[a:a + 1]),)              # noqa: E731
    extend = lambda iv, a, lo, hi: (count_in(text, r[lo:hi]),)         # noqa: E731
    return [(b, e, iv[0]) for b, e, iv in _round3(q, single, extend, min_len, max_mem_intv)]
