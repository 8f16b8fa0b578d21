"""CPU reference of BWA-MEM's seed chaining (debwt_index_chains), independent of the CUDA path: bwa 0.7.17's mem_chain
(chain set ordered by pos, test_and_merge), mem_chain_weight and mem_chain_flt as include/debwt_b200.h restates them,
over any (seeds, hits) pair in the layout of debwt_index_seeds: tests/seed_ref.reference's tuples or the arrays of
BwtBuilder.seeds."""
import bisect

import numpy as np

DEFAULTS = dict(w=100, max_chain_gap=10000, min_chain_weight=0, mask_level=0.5, drop_ratio=0.5, max_chain_extend=1 << 30)

F32 = np.float32


def tuples(seeds, hits):
    """SEED_DTYPE / HIT_DTYPE arrays as the tuples of tests/seed_ref.reference"""
    s = [(int(x["qbeg"]), int(x["qend"]), int(x["round"]), int(x["row"]), int(x["rc_row"]), int(x["count"]), int(x["hit_begin"]),
          int(x["n_hits"])) for x in seeds]
    h = [(int(x["pos"]), int(x["offset"]), int(x["record"]), int(x["strand"])) for x in hits]
    return s, h


def frac_rep(seeds, read_len: int, max_occ: int):
    """bwa's l_rep sweep over the seeds (qbeg, qend, count) above max_occ, over the read length, in float32"""
    b = e = l_rep = 0
    for qb, qe, cnt in seeds:
        if cnt <= max_occ:
            continue
        if qb > e:
            l_rep += e - b
            b, e = qb, qe
        else:
            e = max(e, qe)
    l_rep += e - b
    return F32(l_rep) / F32(read_len) if read_len else F32(0)


def test_and_merge(c, p, rid, l_pac, w, max_chain_gap):
    """0: not merged; 1: contained (not added); 2: appended.  c: {"seeds": [(rbeg, qbeg, len)], "rid"}"""
    if rid != c["rid"]:
        return 0
    first, last = c["seeds"][0], c["seeds"][-1]
    rb, qb, ln = p
    if qb >= first[1] and qb + ln <= last[1] + last[2] and rb >= first[0] and rb + ln <= last[0] + last[2]:
        return 1
    if (last[0] < l_pac or first[0] < l_pac) and rb >= l_pac:
        return 0
    x, y = qb - last[1], rb - last[0]
    if y >= 0 and x - y <= w and y - x <= w and x - last[2] < max_chain_gap and y - last[2] < max_chain_gap:
        c["seeds"].append(p)
        return 2
    return 0


def weight(seeds) -> int:
    """mem_chain_weight: the smaller of the query and reference sweeps"""
    out = []
    for k in (1, 0):
        end = w = 0
        for s in seeds:
            if s[k] >= end:
                w += s[2]
            elif s[k] + s[2] > end:
                w += s[k] + s[2] - end
            end = max(end, s[k] + s[2])
        out.append(w)
    return min(out)


def chain_set(shits, l_pac, w=100, max_chain_gap=10000, trace=None, **_):
    """mem_chain over [(rbeg, qbeg, len, rid)] in visiting order: the chains [{"pos", "seeds", "rid", "cid"}] in chain-set
    order (pos, then creation).  trace (a list) receives per hit (outcome 0 new / 1 contained / 2 appended, cid tested or
    None, (first, last) of that chain when tested)."""
    chains, keys = [], []                                             # keys: (pos, cid) ascending
    for rb, qb, ln, rid in shits:
        p = (rb, qb, ln)
        i = bisect.bisect_right(keys, (rb, float("inf"))) - 1
        got, cid, ends = 0, None, None
        if i >= 0:
            cid = keys[bisect.bisect_left(keys, (keys[i][0], -1))][1]  # the first created chain at that pos
            c = chains[cid]
            ends = (c["seeds"][0], c["seeds"][-1])
            got = test_and_merge(c, p, rid, l_pac, w, max_chain_gap)
        if trace is not None:
            trace.append((got, cid, ends))
        if not got:
            bisect.insort(keys, (rb, len(chains)))
            chains.append({"pos": rb, "seeds": [p], "rid": rid, "cid": len(chains)})
    return [chains[c] for _, c in keys]


def chain_filter(chains, min_seed_len, min_chain_weight=0, mask_level=0.5, drop_ratio=0.5, max_chain_gap=10000,
                 max_chain_extend=1 << 30, **_):
    """mem_chain_flt over chains in chain-set order: the kept chains in output order, each with "w" and "kept" set"""
    a = []
    for c in chains:
        c = dict(c, w=weight(c["seeds"]), first=-1, kept=0)
        if c["w"] >= min_chain_weight:
            a.append(c)
    a.sort(key=lambda c: -c["w"])                                     # stable: ties keep chain-set order
    if not a:
        return []
    beg = lambda c: c["seeds"][0][1]                                  # noqa: E731
    end = lambda c: c["seeds"][-1][1] + c["seeds"][-1][2]             # noqa: E731
    a[0]["kept"] = 3
    kept = [0]
    for i in range(1, len(a)):
        large, dropped = False, False
        for j in kept:
            b, e = max(beg(a[i]), beg(a[j])), min(end(a[i]), end(a[j]))
            if e <= b:
                continue
            min_l = min(end(a[i]) - beg(a[i]), end(a[j]) - beg(a[j]))
            if F32(e - b) >= F32(min_l) * F32(mask_level) and min_l < max_chain_gap:
                large = True
                if a[j]["first"] < 0:
                    a[j]["first"] = i
                if F32(a[i]["w"]) < F32(a[j]["w"]) * F32(drop_ratio) and a[j]["w"] - a[i]["w"] >= 2 * min_seed_len:
                    dropped = True
                    break
        if not dropped:
            kept.append(i)
            a[i]["kept"] = 2 if large else 3
    for j in kept:
        if a[j]["first"] >= 0:
            a[a[j]["first"]]["kept"] = 1
    i = k = 0
    while i < len(a):
        if a[i]["kept"] not in (0, 3):
            k += 1
            if k >= max_chain_extend:
                break
        i += 1
    for c in a[i:]:
        if c["kept"] < 3:
            c["kept"] = 0
    return [c for c in a if c["kept"]]


def read_chains(shits, l_pac, min_seed_len, **opts):
    """mem_chain then mem_chain_flt for one read's chain seeds [(rbeg, qbeg, len, rid)]"""
    o = {**DEFAULTS, **opts}
    return chain_filter(chain_set(shits, l_pac, **o), min_seed_len, **o)


def read_hits(seeds, hits, seps):
    """[(rbeg, qbeg, len, rid)] of seeds [(qbeg, qend, ...)] with hits [hit_begin, hit_begin + n_hits) in visiting order"""
    from debwt_b200 import api
    out = []
    for s in seeds:
        qb, qe, hb, nh = s[0], s[1], s[6], s[7]
        h = hits[hb:hb + nh]
        if not h:
            continue
        rb = api.bwa_rbeg([x[2] for x in h], [x[3] for x in h], [x[1] for x in h], qe - qb, seps)
        out += [(int(r), qb, qe - qb, x[2]) for r, x in zip(rb.tolist(), h)]
    return out


def reference(offsets, seeds, hits, seps, read_lens, min_len=19, max_occ=500, **opts):
    """(offsets, [(pos, seed_begin, n_seeds, weight, record, strand, kept, frac_rep)], [(rbeg, qbeg, len)]) as
    debwt_index_chains lays them out, from seeds / hits in the tuple layout of tests/seed_ref.reference"""
    seps = np.asarray(seps, dtype=np.uint64)
    l_pac = (int(seps[-1]) + 1 - seps.size) // 2
    offs, out, cseeds = [0], [], []
    for i, L in enumerate(read_lens):
        sd = seeds[offsets[i]:offsets[i + 1]]
        fr = frac_rep([(s[0], s[1], s[5]) for s in sd], L, max_occ)
        for c in read_chains(read_hits(sd, hits, seps), l_pac, min_len, **opts):
            strand = int(c["pos"] >= l_pac)
            out.append((c["pos"], len(cseeds), len(c["seeds"]), c["w"], c["rid"], strand, c["kept"], float(fr)))
            cseeds += c["seeds"]
        offs.append(len(out))
    return offs, out, cseeds


def as_tuples(chains, cseeds):
    """CHAIN_DTYPE / CHAIN_SEED_DTYPE arrays in the layout of `reference`"""
    c = [(int(x["pos"]), int(x["seed_begin"]), int(x["n_seeds"]), int(x["weight"]), int(x["record"]), int(x["strand"]), int(x["kept"]),
          float(x["frac_rep"])) for x in chains]
    s = [(int(x["rbeg"]), int(x["qbeg"]), int(x["len"])) for x in cseeds]
    return c, s
