"""TEST INFRASTRUCTURE: numpy restatement of the stage kernels behind debwt_b200.dist (the `ops`
interface of CudaOps), so that the sharded orchestration -- slicing, splitters, the three
all-to-alls, global numbering -- can run on CPU tensors under a world_size-2 gloo group.

Same method signatures and data layouts as debwt_b200.dist.CudaOps; semantics follow
oracle/stages.py (which cites the reference).  Never imported by the product.
"""
from __future__ import annotations

import numpy as np
import torch

from debwt_b200 import dist as D

U = np.uint64
M64 = U(0xFFFFFFFFFFFFFFFF)


def u(t):
    """torch int tensor -> numpy unsigned view (shares memory)"""
    a = t.numpy()
    return a.view({np.dtype(np.int64): np.uint64, np.dtype(np.int32): np.uint32, np.dtype(np.int16): np.uint16}.get(a.dtype, a.dtype))


def window32(words, p):
    """32 symbols starting at position p (vectorised over p)"""
    p = np.asarray(p, dtype=np.uint64)
    i = (p >> U(5)).astype(np.int64)
    s = (p & U(31)) * U(2)
    a = words[i]
    b = words[i + 1]
    with np.errstate(over="ignore"):
        hi = a << s
        lo = np.where(s == 0, U(0), b >> ((U(64) - s) & U(63)))
    return (hi | lo).astype(np.uint64)


def symbol(words, p):
    p = np.asarray(p, dtype=np.uint64)
    return ((words[(p >> U(5)).astype(np.int64)] >> (U(2) * (U(31) - (p & U(31))))) & U(3)).astype(np.int64)


def popc4(x):
    return (x & 1) + ((x >> 1) & 1) + ((x >> 2) & 1) + ((x >> 3) & 1)


def multi_in(m):
    m = m.astype(np.int64)
    return (popc4(m & 15) >= 2) | ((m & 16) != 0)


def multi_out(m):
    m = m.astype(np.int64)
    return (popc4((m >> 8) & 15) >= 2) | ((m & 4096) != 0)


class NumpyOps:
    def __init__(self):
        self.launches = 0

    def empty(self, n, dtype=torch.int64):
        return torch.zeros(max(int(n), 0), dtype=dtype)

    zeros = empty

    def from_numpy(self, a):
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        return torch.from_numpy(np.ascontiguousarray(a).copy())

    def sync(self):
        pass

    # ---- K1 / K2 / K3 ----
    def pack(self, ascii_slice, n_valid, words_out, nwords, err):
        a = ascii_slice.numpy()[:n_valid]
        up = a & 0xDF
        code = np.full(nwords * 32, 0, dtype=np.uint64)
        ok = (up == 0x41) | (up == 0x43) | (up == 0x47) | (up == 0x54)
        sep = (a == 0x23) | (a == 0x24)
        if (~ok & ~sep).any():
            err[0] = 1
        err[1] += int(sep.sum())
        c = ((up >> 1) & 3).astype(np.uint64)
        c ^= c >> U(1)
        code[:n_valid] = np.where(ok, c, U(3))
        code[n_valid:min(n_valid + 32, nwords * 32)] = 3
        sh = (U(2) * (U(31) - (np.arange(nwords * 32, dtype=np.uint64) & U(31))))
        u(words_out)[:nwords] = np.bitwise_or.reduce((code << sh).reshape(nwords, 32), axis=1)

    def extract(self, words, pos_lo, pos_hi, seps, n_rec, idx_base, keys_out, n_symbols):
        w, s = u(words), u(seps)
        p = np.arange(pos_lo, pos_hi, dtype=np.uint64)
        r = np.searchsorted(s, p, side="left")
        okr = r < n_rec
        valid = okr.copy()
        valid[okr] = p[okr] + U(32) <= s[r[okr]]
        pv, rv = p[valid], r[valid].astype(np.uint64)
        u(keys_out)[(pv - U(32) * rv - U(idx_base)).astype(np.int64)] = window32(w, pv)

    def sort(self, keys):
        return torch.from_numpy(np.sort(u(keys)).view(np.int64).copy())

    # ---- K12 ----
    def owner_of_keys(self, items, splitters, mask, drop_marker):
        v = u(items)
        d = np.searchsorted(u(splitters), v & U(mask), side="right").astype(np.uint8)
        if drop_marker:
            d[v == M64] = 255
        return torch.from_numpy(d)

    def owner_of_index(self, idx, bases, n_ranks):
        g, b = u(idx), u(bases)
        r = np.searchsorted(b[:n_ranks], g, side="right") - 1
        g[:] = g - b[r]
        return torch.from_numpy(r.astype(np.uint8))

    def partition_by_splitters(self, items, splitters, n_split, mask, drop_marker, n_ranks):
        dest = self.owner_of_keys(items, splitters[:n_split], mask, drop_marker)
        out, _, counts = self.partition(items, None, dest, n_ranks)
        return out, counts

    def partition(self, a, b, dest, n_ranks):
        d = dest.numpy()
        keep = d < n_ranks
        order = np.argsort(d[keep], kind="stable")
        counts = np.bincount(d[keep], minlength=n_ranks)[:n_ranks].tolist()
        out_a = torch.zeros_like(a)
        out_a[:order.size] = a[torch.from_numpy(np.flatnonzero(keep)[order])]
        out_b = None
        if b is not None:
            out_b = torch.zeros_like(b)
            out_b[:order.size] = b[torch.from_numpy(np.flatnonzero(keep)[order])]
        return out_a, out_b, [int(c) for c in counts]

    # ---- K5..K7 ----
    def key_index(self, sorted_keys):
        return (None, 0)

    def _heads(self, k):
        km = k >> U(2)
        h = np.ones(k.size, dtype=bool)
        h[1:] = km[1:] != km[:-1]
        return h

    def out_edges_queries(self, sorted_keys, gmask):
        k, g = u(sorted_keys), u(gmask)
        q = np.full(k.size, M64, dtype=np.uint64)
        if k.size == 0:
            return torch.from_numpy(q.view(np.int64))
        dist_head = np.ones(k.size, dtype=bool)
        dist_head[1:] = k[1:] != k[:-1]
        gh = np.flatnonzero(self._heads(k))
        grp_head_of = gh[np.searchsorted(gh, np.arange(k.size), side="right") - 1]
        idx = np.flatnonzero(dist_head)
        np.bitwise_or.at(g, grp_head_of[idx], (1 << (8 + (k[idx] & U(3)).astype(np.int64))).astype(np.uint16))
        with np.errstate(over="ignore"):
            qq = (k[idx] << U(2)) | (k[idx] >> U(62))
        polyt = qq == M64
        np.bitwise_or.at(g, grp_head_of[idx[polyt]], np.uint16(8))
        q[idx] = qq
        return torch.from_numpy(q.view(np.int64).copy())

    def apply_in_queries(self, sorted_keys, ki, gmask, q):
        k, g, qq = u(sorted_keys), u(gmask), u(q)
        if qq.size == 0:
            return
        x = qq & U(0xFFFFFFFFFFFFFFFC)
        hs = np.searchsorted(k, x, side="left")
        ok = hs < k.size
        ok[ok] = (k[hs[ok]] & U(0xFFFFFFFFFFFFFFFC)) == x[ok]
        np.bitwise_or.at(g, hs[ok], (1 << (qq[ok] & U(3)).astype(np.int64)).astype(np.uint16))

    def heads_tails(self, words, seps, n_rec, sorted_keys, ki, gmask):
        w, s, k, g = u(words), u(seps), u(sorted_keys), u(gmask)
        starts = np.concatenate(([0], s[:-1] + U(1))).astype(np.uint64)
        for pos, bit in ((starts, 16), (s - U(31), 4096)):
            x = window32(w, pos) & U(0xFFFFFFFFFFFFFFFC)
            h = np.searchsorted(k, x, side="left")
            ok = h < k.size
            ok[ok] = (k[h[ok]] & U(0xFFFFFFFFFFFFFFFC)) == x[ok]
            np.bitwise_or.at(g, h[ok], np.uint16(bit))

    def propagate(self, sorted_keys, gmask):
        k, g = u(sorted_keys), u(gmask)
        gh = np.flatnonzero(self._heads(k))
        head_of = gh[np.searchsorted(gh, np.arange(k.size), side="right") - 1]
        g[:k.size] = g[head_of]

    def branch_table(self, sorted_keys, gmask):
        k, g = u(sorted_keys), u(gmask)[:sorted_keys.numel()]
        if k.size == 0:
            return {"kmer": self.empty(0), "head": self.empty(0, torch.int32), "blue": self.zeros(1, torch.int32), "B": 0, "M": 0}
        h = self._heads(k)
        gh = np.flatnonzero(h)
        size = np.diff(np.append(gh, k.size))
        mi, mo = multi_in(g[gh]), multi_out(g[gh])
        br = mi | mo
        kmer = (k[gh[br]] & U(0xFFFFFFFFFFFFFFFC)) | mo[br].astype(np.uint64) | (mi[br].astype(np.uint64) << U(1))
        sz = np.where(mi[br], size[br], 0)
        blue = np.concatenate(([0], np.cumsum(sz))).astype(np.int32)
        return {"kmer": torch.from_numpy(kmer.view(np.int64).copy()), "head": torch.from_numpy(gh[br].astype(np.int32)),
                "blue": torch.from_numpy(blue), "B": int(br.sum()), "M": int(sz.sum())}

    def branch_index(self, gkmer):
        return (None, 0)

    # ---- sentinel-window suffixes ----
    def special_scan(self, words, seps, n_rec, sorted_keys, ki):
        import functools
        w, s, k = u(words), u(seps), u(sorted_keys)
        n = int(s[-1]) + 1
        sym = symbol(w, np.arange(n, dtype=np.uint64)).astype(np.uint8)
        sym[s.astype(np.int64)] = 4
        sym[n - 1] = 5
        b = bytes(sym.tolist())
        m = 32 * n_rec
        pos = [int(s[t >> 5]) - (t & 31) for t in range(m)]
        order = sorted(range(m), key=lambda t: b[pos[t]:])
        rank = np.zeros(m, dtype=np.uint32)
        rank[order] = np.arange(m, dtype=np.uint32)
        out = np.zeros((m, 4), dtype=np.uint64)
        for t in range(m):
            p, j = pos[t], t & 31
            w0 = window32(w, [p])[0]
            w1 = window32(w, [p + j + 1])[0]
            if j:
                pad = (w0 & ~(M64 >> U(2 * j))) | (M64 >> U(2 * j))
                ins = int(np.searchsorted(k, pad, side="right"))
            else:
                ins = k.size
            out[t, 0], out[t, 1], out[t, 2] = w0, w1, ins
            out[t, 3] = U(int(rank[t])) | (U(int(symbol(w, [p - 1])[0])) << U(32)) | (U(int(symbol(w, [p + 31])[0])) << U(40))
        return out.reshape(-1).view(np.int64).copy()

    def special_tables(self, info_np, ins_by_t, seps_np, n_rec):
        return D.special_tables_host(info_np, ins_by_t, seps_np, n_rec)

    # ---- K9 ----
    def flag_slice(self, words, pos_lo, pos_hi, seps, n_rec, gkmer, gbidx, nbw, cap):
        w, s, gk = u(words), u(seps), u(gkmer)
        mo = np.zeros(nbw + 2, dtype=np.uint32)
        ent, ind = [], []
        p = np.arange(pos_lo, pos_hi, dtype=np.uint64)
        if p.size:
            r = np.searchsorted(s, p, side="left")
            okr = r < n_rec
            valid = okr.copy()
            valid[okr] = p[okr] + U(32) <= s[r[okr]]
            pv, rv = p[valid], r[valid]
            x = window32(w, pv) & U(0xFFFFFFFFFFFFFFFC)
            tab = gk & U(0xFFFFFFFFFFFFFFFC)
            b = np.searchsorted(tab, x, side="left")
            found = b < tab.size
            found[found] = tab[b[found]] == x[found]
            for pp, rr, bb in zip(pv[found].tolist(), rv[found].tolist(), b[found].tolist()):
                f = int(gk[bb]) & 3
                if f & 1:
                    l = pp - pos_lo
                    mo[l >> 5] |= np.uint32(1 << (l & 31))
                if f & 2:
                    start = int(s[rr - 1]) + 1 if rr else 0
                    prev = (4 if rr else 5) if pp == start else int(symbol(w, [pp - 1])[0])
                    ent.append((pp << 4) | prev)
                    ind.append(bb)
        return (torch.from_numpy(mo.view(np.int32).copy()), torch.tensor(ent, dtype=torch.int64), torch.tensor(ind, dtype=torch.int64))

    def patch_bits_slice(self, mo, pos_lo, pos_hi, positions):
        m = u(mo)
        for p in u(positions).tolist():
            if pos_lo <= p < pos_hi:
                l = p - pos_lo
                m[l >> 5] |= np.uint32(1 << (l & 31))

    def scan_popc(self, mo, nbw):
        m = u(mo)[:nbw]
        pc = np.array([bin(int(x)).count("1") for x in m], dtype=np.int64)
        wp = np.zeros(nbw + 2, dtype=np.int32)
        wp[:nbw] = np.cumsum(pc) - pc
        return torch.from_numpy(wp), int(pc.sum())

    def _sp_index(self, mo, wp, pos_lo, code_base, p):
        l = p - pos_lo
        bits = int(u(mo)[l >> 5]) & ((1 << (l & 31)) - 1)
        return code_base + int(wp[l >> 5]) + bin(bits).count("1")

    def emit_codes_slice(self, words, word_lo, nbw, mo, wp, code_base, codes):
        w, m, c = u(words), u(mo), u(codes)
        for wl in range(nbw):
            bits = int(m[wl])
            ci = code_base + int(wp[wl])
            for b in range(32):
                if bits >> b & 1:
                    p = (word_lo + wl) * 32 + b
                    code = int(symbol(w, [p + 31])[0])
                    c[ci >> 5] |= U(code) << U(2 * (31 - (ci & 31)))
                    ci += 1

    def mark_sep_slice(self, mo, wp, pos_lo, pos_hi, code_base, tail_pos, sep):
        out = np.zeros(tail_pos.numel(), dtype=np.int64)
        sp = u(sep)
        for t, p in enumerate(u(tail_pos).tolist()):
            if pos_lo <= p < pos_hi:
                ci = self._sp_index(mo, wp, pos_lo, code_base, p)
                sp[ci >> 5] |= np.uint32(1 << (ci & 31))
                out[t] = ci
        return torch.from_numpy(out)

    def fix_records(self, rec_entry, mo, wp, pos_lo, code_base):
        e = u(rec_entry)
        for i in range(e.size):
            v = int(e[i])
            e[i] = U((self._sp_index(mo, wp, pos_lo, code_base, v >> 4) << 4) | (v & 15))

    # ---- K10 / K11 ----
    def scatter_blue(self, rec_entry, rec_local, bt):
        blue = np.zeros(bt["M"] + 1, dtype=np.int64)
        cur = np.zeros(bt["B"] + 1, dtype=np.int64)
        off = bt["blue"].numpy()
        for e, b in zip(rec_entry.tolist(), rec_local.tolist()):
            blue[int(off[b]) + cur[b]] = e
            cur[b] += 1
        return torch.from_numpy(blue)

    def sort_blue(self, blue, bt, codes, sep, dollar_index, n_codes):
        c, s = u(codes), u(sep)
        syms = []
        for i in range(n_codes):
            v = int(c[i >> 5] >> U(2 * (31 - (i & 31)))) & 3
            if int(s[i >> 5]) >> (i & 31) & 1:
                v = 5 if i == dollar_index else 4
            syms.append(v)
        sb = bytes(syms)
        off = bt["blue"].numpy()
        bl = blue.numpy()
        km = u(bt["kmer"])
        for b in range(bt["B"]):
            if int(km[b]) & 2:
                lo, hi = int(off[b]), int(off[b + 1])
                seg = sorted(bl[lo:hi].tolist(), key=lambda e: sb[(e >> 4):])
                bl[lo:hi] = seg

    def release_cached(self, m):
        pass

    def bwt_segment(self, word_lo, word_hi):
        """numpy restatement: the segment is a view into a full-size array, which is also the handle"""
        full = torch.zeros(word_hi + 2, dtype=torch.int64)
        return full[word_lo:word_hi + 1], full

    def fill_range(self, gmask, n_keys, key_base, n_symbols, spec_rows, word_lo, word_hi, bwt):
        g, rows, out = u(gmask), u(spec_rows), u(bwt)
        for wd in range(word_lo, word_hi):
            val = 0
            for lane in range(32):
                row = wd * 32 + lane
                code = 0
                if row < n_symbols:
                    t = int(np.searchsorted(rows, U(row), side="left"))
                    special = t < rows.size and int(rows[t]) == row
                    i = row - t
                    if not special and key_base <= i < key_base + n_keys:
                        mk = int(g[i - key_base])
                        if not bool(multi_in(np.array([mk]))[0]) and (mk & 15):
                            code = (mk & 15).bit_length() - 1
                val |= code << (2 * (31 - lane))
            out[wd] = U(val)

    def emit_blue(self, blue, bt, key_base, spec_ins, bwt, n_rec):
        out, ins = u(bwt), u(spec_ins)
        off, head, bl = bt["blue"].numpy(), bt["head"].numpy(), blue.numpy()
        km = u(bt["kmer"])
        sharp, dollar = [], -1
        for b in range(bt["B"]):
            if not int(km[b]) & 2:
                continue
            for t, e in enumerate(bl[int(off[b]):int(off[b + 1])].tolist()):
                i = key_base + int(head[b]) + t
                row = i + int(np.searchsorted(ins, U(i), side="right"))
                c = e & 15
                if c == 4:
                    sharp.append(row)
                elif c == 5:
                    dollar = row
                code = min(c, 3)
                out[row >> 5] |= U(code) << U(2 * (31 - (row & 31)))
        return torch.tensor(sharp, dtype=torch.int64), torch.tensor([dollar], dtype=torch.int64)

    def emit_special(self, spec_rows, spec_chr, bwt):
        out = u(bwt)
        for row, c in zip(u(spec_rows).tolist(), spec_chr.numpy().tolist()):
            out[row >> 5] |= U(c) << U(2 * (31 - (row & 31)))
