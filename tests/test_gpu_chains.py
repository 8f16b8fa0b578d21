"""BWA-MEM seed chaining (debwt_index_chains, BwtBuilder.chains) through the C ABI against tests/chain_ref.py, exactly
(chains and chain seeds), on both strands of the seeded cases and read mix of tests/test_gpu_smem.py at three option
sets; chain seeds against the hits of seeds() through api.bwa_rbeg; chains() against chain_ref over the GPU's own
seeds(); a repeat above max_occ; poly-A and 1-Mbp reads; a loaded result of another text; and the error paths."""
import ctypes

import numpy as np
import pytest

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from tests import chain_ref as cr
from tests import seed_ref as sr
from tests import smem_ref as ref
from tests.locate_ref import suffix_array
from tests.test_gpu_seeds import _sa
from tests.test_gpu_smem import _LUT, CASES, _case, _mutate, _reads
from tests.util import golden

pytestmark = pytest.mark.gpu

NO_FILTER = dict(cr.DEFAULTS, mask_level=1.5)
STRICT = dict(cr.DEFAULTS, w=5, max_chain_gap=50, min_chain_weight=25, drop_ratio=0.9, max_chain_extend=2)
OPTS = {"defaults": dict(cr.DEFAULTS), "no_filter": NO_FILTER, "strict": STRICT}


def _want(model, sa, seps, reads, **o):
    offs, seeds, hits = sr.reference(model, sa, seps, reads, **sr.DEFAULTS)
    return cr.reference(offs, seeds, hits, seps, [len(r) for r in reads], **{**sr.DEFAULTS, **o})


def _check_against_hits(reads, offs, chains, cseeds, s_offs, seeds, hits, seps):
    """every chain seed is a hit of one of its read's seeds, in bwa's coordinate"""
    for i in range(len(reads)):
        sd = seeds[int(s_offs[i]):int(s_offs[i + 1])]
        have = set()
        for x in sd:
            h = hits[int(x["hit_begin"]):int(x["hit_begin"]) + int(x["n_hits"])]
            L = int(x["qend"] - x["qbeg"])
            rb = api.bwa_rbeg(h["record"], h["strand"], h["offset"], L, seps)
            have.update((int(r), int(x["qbeg"]), L, int(rec)) for r, rec in zip(rb.tolist(), h["record"].tolist()))
        for c in chains[int(offs[i]):int(offs[i + 1])]:
            for s in cseeds[int(c["seed_begin"]):int(c["seed_begin"]) + int(c["n_seeds"])]:
                assert (int(s["rbeg"]), int(s["qbeg"]), int(s["len"]), int(c["record"])) in have, (i, s)


@pytest.mark.parametrize("name", CASES)
def test_chains_equal_reference(name):
    both, text, seps, model = _case(name)
    reads = _reads(both, np.random.default_rng(31))
    seen = {"kept": set(), "strand": set(), "multi": False}
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(16)
        s_offs, seeds, hits = b.seeds(reads)
        for label, o in OPTS.items():
            want = _want(model, _sa(name), seps, reads, **o)
            offs, chains, cseeds = b.chains(reads, **o)
            assert chains.dtype == api.CHAIN_DTYPE and cseeds.dtype == api.CHAIN_SEED_DTYPE
            assert offs.tolist() == want[0], label
            got = cr.as_tuples(chains, cseeds)
            assert got[0] == want[1], label
            assert got[1] == want[2], label
            _check_against_hits(reads, offs, chains, cseeds, s_offs, seeds, hits, seps)
            if label == "no_filter":
                assert (chains["kept"] == 3).all()
                mine = cr.reference(s_offs.tolist(), *cr.tuples(seeds, hits), seps, [len(r) for r in reads], **{**sr.DEFAULTS, **o})
                assert (offs.tolist(), got[0], got[1]) == mine
            if label == "strict":
                assert (chains["weight"] >= 25).all()
                assert all(((c["kept"] == 1) | (c["kept"] == 2)).sum() <= 1 for c in np.split(chains, offs[1:-1].astype(np.int64)))
            seen["kept"].update(chains["kept"].tolist())
            seen["strand"].update(chains["strand"].tolist())
            seen["multi"] |= bool((np.diff(offs.astype(np.int64)) > 1).any())
    assert {1, 3} <= seen["kept"] and seen["strand"] == {0, 1} and seen["multi"], seen
    assert 2 in seen["kept"] or name != "c3_like_600k_3rec", seen                # kept 2 occurs on the three-record case


def test_repeat_above_default_max_occ():
    """a 40-base unit in 1100 copies: reads on it have hundreds of chains and frac_rep > 0"""
    rng = np.random.default_rng(9)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    unit = acgt[rng.integers(0, 4, 40)].tobytes()
    recs = [bytearray(acgt[rng.integers(0, 4, 150_000)].tobytes()) for _ in range(2)]
    for j in range(1100):
        r = recs[j % 2]
        p = 100 * (j // 2) + 30
        r[p:p + 40] = unit
    recs = [bytes(r) for r in recs]
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    model = ref.FmdModel(_LUT[text])
    sa = suffix_array(_LUT[text])
    reads = [recs[0][100 * k:100 * k + 150] for k in (3, 40, 200)] + [_mutate(recs[1][100 * k + 10:100 * k + 130], rng, 2) for k in (7, 77)]
    reads += [b"GATTACA" + unit + b"CAT", unit]
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(32)
        for o in (cr.DEFAULTS, NO_FILTER):
            want = _want(model, sa, seps, reads, **o)
            offs, chains, cseeds = b.chains(reads, **o)
            assert offs.tolist() == want[0] and cr.as_tuples(chains, cseeds) == (want[1], want[2])
        assert np.diff(offs.astype(np.int64)).max() >= 200 and (chains["frac_rep"] > 0).any()


def test_poly_a_and_megabase_reads():
    rng = np.random.default_rng(4)
    acgt = b"ACGT"
    rnd = lambda k: bytes(acgt[int(x)] for x in rng.integers(0, 4, k))  # noqa: E731
    recs = [rnd(40_000), b"A" * 3000 + rnd(500), rnd(200) + b"A" * 2500 + rnd(300), b"C" + b"A" * 2100]
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    model = ref.FmdModel(_LUT[text])
    sa = suffix_array(_LUT[text])
    reads = [b"A" * 2000, b"G" + b"A" * 2000 + b"C", b"A" * 1000 + b"N" + b"A" * 999, b"C" + b"A" * 2101, b"A" * 2400, rnd(150)]
    want = _want(model, sa, seps, reads)
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(8)
        offs, chains, cseeds = b.chains(reads)
        assert offs.tolist() == want[0] and cr.as_tuples(chains, cseeds) == (want[1], want[2])
        assert chains.size

    both, text, seps, model = _case("c2_like_1m")
    rec = both[0]
    short = [_mutate(rec[a:a + 150], rng, int(rng.integers(0, 3))) for a in rng.integers(0, len(rec) - 150, 300).tolist()]
    reads = short[:150] + [rec] + short[150:]
    for o in (cr.DEFAULTS, STRICT):
        want = _want(model, _sa("c2_like_1m"), seps, reads, **o)
        with api.BwtBuilder() as b:
            b.set_records(both)
            b.build()
            b.sample_sa(16)
            offs, chains, cseeds = b.chains(reads, **o)
        assert offs.tolist() == want[0] and cr.as_tuples(chains, cseeds) == (want[1], want[2])
        mega = chains[int(offs[150]):int(offs[151])]
        assert mega.size >= 1 and int(mega[0]["weight"]) >= len(rec) // 2


def test_loaded_result_of_another_text(tmp_path):
    both, text, seps, model = _case("c4_like_5x100k")
    reads = _reads(both, np.random.default_rng(77))
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        b.sample_sa(32)
        want = b.chains(reads)
        words, sharp, dollar = b.result()
    api.write_outputs(str(tmp_path / "c4.bwt"), words, sharp, dollar)
    both2, text2, seps2, model2 = _case("c3_like_600k_3rec")
    reads2 = _reads(both2, np.random.default_rng(78))
    with api.BwtBuilder() as c:
        w, s, d = api.read_outputs(str(tmp_path / "c4.bwt"), text.size)
        c.set_result(w, text.size, s, d)
        c.sample_sa(16)
        got = c.chains(reads)
        assert all((x == y).all() for x, y in zip(got, want))
        with api.BwtBuilder() as e:
            e.set_records(both2)
            e.build()
            w2, s2, d2 = e.result()
        c.set_result(w2, text2.size, s2, d2)
        c.sample_sa(32)
        offs, chains, cseeds = c.chains(reads2)
    ref2 = _want(model2, _sa("c3_like_600k_3rec"), seps2, reads2)
    assert offs.tolist() == ref2[0] and cr.as_tuples(chains, cseeds) == (ref2[1], ref2[2])


def test_errors():
    recs = [r.upper().encode() for r in golden()["small"]["haplotypes_6x1500"]["records"]]
    both = api.both_strands(recs)
    L = binding.lib()
    SENT = 0xA5A5A5A5A5A5A5A5

    def raw(b, reads, cap=100, scap=1000, offs=None, null="", seed_kw=None, **kw):
        so = {**dict(min_len=19, split_width=10, max_mem_intv=20, max_occ=500, split_factor=1.5), **(seed_kw or {})}
        sopts = api.SeedOpts(so["min_len"], so["split_width"], so["max_mem_intv"], so["max_occ"], so["split_factor"])
        o = {**cr.DEFAULTS, **kw}
        copts = api.ChainOpts(o["w"], o["max_chain_gap"], o["min_chain_weight"], o["max_chain_extend"], o["mask_level"], o["drop_ratio"])
        blob = np.frombuffer(b"".join(reads) + b"\0", dtype=np.uint8)
        if offs is None:
            offs = np.concatenate(([0], np.cumsum([len(r) for r in reads]))).astype(np.uint64)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        co = np.full(len(reads) + 1, SENT, dtype=np.uint64)
        ns = np.full(1, SENT, dtype=np.uint64)
        ch = np.zeros(max(cap, 1) + 4, dtype=api.CHAIN_DTYPE)
        ch["pos"] = SENT
        cs = np.zeros(max(scap, 1) + 4, dtype=api.CHAIN_SEED_DTYPE)
        cs["rbeg"] = SENT
        P = lambda name, a: None if null == name else api._ptr(a)  # noqa: E731
        rc = L.debwt_index_chains(b._h, P("reads", blob), P("offsets", offs), len(reads),
                                  None if null == "seed_opts" else ctypes.addressof(sopts),
                                  None if null == "chain_opts" else ctypes.addressof(copts), P("chain_offsets", co),
                                  P("n_chain_seeds", ns), P("chains", ch), cap, P("chain_seeds", cs), scap)
        return rc, co, ns, ch, cs, L.debwt_last_error().decode()

    def untouched(co, ns, ch, cs):
        return (co == SENT).all() and (ns == SENT).all() and (ch["pos"] == SENT).all() and (cs["rbeg"] == SENT).all()

    reads = [q[100:180] for q in both] + [b"ACGTN" * 9]
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.index()
        rc, co, ns, ch, cs, msg = raw(b, reads)                       # no samples
        assert rc != 0 and "debwt_index_sample_sa" in msg and untouched(co, ns, ch, cs)
        with pytest.raises(DebwtError, match="sample_sa"):
            b.chains(reads)
        b.sample_sa(32)
        offs, chains, cseeds = b.chains(reads)
        total, ts = int(offs[-1]), cseeds.size
        assert total >= len(reads) - 1 and ts >= total
        for cap, scap in ((total - 1, ts), (total, ts - 1)):          # too small: names both totals, writes no chain or seed
            rc, co, ns, ch, cs, msg = raw(b, reads, cap, scap)
            assert rc != 0 and str(total) in msg and str(ts) in msg and (co == offs).all() and int(ns[0]) == ts
            assert (ch["pos"] == SENT).all() and (cs["rbeg"] == SENT).all()
        rc, co, ns, ch, cs, msg = raw(b, reads, total, ts)
        assert rc == 0 and (co == offs).all() and (ch[:total] == chains).all() and (cs[:ts] == cseeds).all()
        assert (ch["pos"][total:] == SENT).all() and (cs["rbeg"][ts:] == SENT).all()
        rc, co, ns, ch, cs, msg = raw(b, reads, 0, 0, null="chains")  # size query
        assert rc == 0 and (co == offs).all() and int(ns[0]) == ts and (ch["pos"] == SENT).all() and (cs["rbeg"] == SENT).all()
        bad = [(dict(w=-1), "w"), (dict(max_chain_gap=-1), "max_chain_gap"), (dict(min_chain_weight=-5), "min_chain_weight"),
               (dict(max_chain_extend=-1), "max_chain_extend"), (dict(mask_level=-0.5), "mask_level"),
               (dict(mask_level=float("nan")), "mask_level"), (dict(drop_ratio=float("inf")), "drop_ratio"),
               (dict(drop_ratio=-1.0), "drop_ratio")]
        for kw, word in bad:
            rc, co, ns, ch, cs, msg = raw(b, reads, **kw)
            assert rc != 0 and word in msg and "index_chains" in msg and untouched(co, ns, ch, cs), kw
        for kw, word in ((dict(min_len=0), "min_seed_len"), (dict(max_occ=0), "max_occ"), (dict(split_factor=-1.0), "split_factor"),
                         (dict(split_factor=float("nan")), "split_factor")):
            rc, co, ns, ch, cs, msg = raw(b, reads, seed_kw=kw)
            assert rc != 0 and word in msg and "index_chains" in msg and untouched(co, ns, ch, cs), kw
        for null in ("reads", "offsets", "chain_offsets", "n_chain_seeds", "seed_opts", "chain_opts", "chain_seeds"):
            rc, co, ns, ch, cs, msg = raw(b, reads, null=null)
            assert rc != 0 and "null argument" in msg and (ch["pos"] == SENT).all() and (cs["rbeg"] == SENT).all(), null
            assert (co == SENT).all() and (ns == SENT).all(), null
        rc, co, ns, ch, cs, msg = raw(b, [b"A" * 40] * 3, offs=np.array([0, 60, 50, 120], dtype=np.uint64))
        assert rc != 0 and "read 1" in msg and untouched(co, ns, ch, cs)
        rc, co, ns, ch, cs, msg = raw(b, [b"ACGT" * 10, b"A" * (1 << 24)])    # the seeding scratch: 72 * 2^24 + 64 bytes > 1 GiB
        assert rc != 0 and "index_chains" in msg and "read 1" in msg and str(((1 << 30) - 64) // 72) in msg and untouched(co, ns, ch, cs)
        rc, co, ns, ch, cs, msg = raw(b, [], 0, 0)                    # no reads
        assert rc == 0 and int(co[0]) == 0 and int(ns[0]) == 0 and (co[1:] == SENT).all()
        o, c, s = b.chains([])
        assert o.tolist() == [0] and c.size == 0 and s.size == 0
        o, c, s = b.chains([b"", b"NNNN", b"ACG"])                     # no hits at all
        assert o.tolist() == [0, 0, 0, 0] and c.size == 0 and s.size == 0
        o, c, s = b.chains(reads, min_chain_weight=10 ** 6)           # every chain below the weight
        assert (o == 0).all() and c.size == 0

    with api.BwtBuilder() as b:                                       # one strand only: unbalanced
        b.set_records(recs)
        b.build()
        b.sample_sa(32)
        rc, co, ns, ch, cs, msg = raw(b, reads)
        assert rc != 0 and "reverse complement" in msg and untouched(co, ns, ch, cs)
    with api.BwtBuilder() as b:                                       # balanced, but an odd number of records
        b.set_records(both + [b"ACGT" * 16])
        b.build()
        b.sample_sa(32)
        rc, co, ns, ch, cs, msg = raw(b, reads)
        assert rc != 0 and str(len(both) + 1) in msg and untouched(co, ns, ch, cs)
