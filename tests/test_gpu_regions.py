"""BWA-MEM seed extension (debwt_index_regions, BwtBuilder.regions) through the C ABI against tests/ext_ref.py, exactly,
on both strands of the seeded cases and read mix of tests/test_gpu_smem.py at five option sets (reads -> seed_ref ->
chain_ref -> ext_ref, and ext_ref over the GPU's own chains()); the 1100-copy repeat; poly-A, 1-Mbp and long mutated
reads with indels; a loaded result of another text; and the error paths."""
import ctypes

import numpy as np
import pytest

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from tests import chain_ref as cr
from tests import ext_ref as er
from tests.test_gpu_chains import _want
from tests.test_gpu_seeds import _sa
from tests.test_gpu_smem import CASES, _case, _mutate, _reads
from tests.util import golden

pytestmark = pytest.mark.gpu

ASYM = dict(w=6, o_del=2, e_del=3, o_ins=5, e_ins=1)
OPTS = {"defaults": {}, "asym_small_w": ASYM, "zdrop1": dict(zdrop=1), "clip0": dict(pen_clip5=0, pen_clip3=0),
        "clip1000": dict(pen_clip5=1000, pen_clip3=1000)}
_CHAIN_KEYS = set(cr.DEFAULTS)


def _split(o):
    return {k: v for k, v in o.items() if k in _CHAIN_KEYS}


def _over_chains(b, reads, text, seps, trace=None, **o):
    """ext_ref over the GPU's own chains() with the same options"""
    offs, chains, cseeds = b.chains(reads, **_split(o))
    c, s = cr.as_tuples(chains, cseeds)
    return er.reference(offs.tolist(), c, s, reads, text, seps, trace=trace, **o)


_SEEN = set()


@pytest.mark.parametrize("name", CASES)
def test_regions_equal_reference(name):
    both, text, seps, model = _case(name)
    reads = _reads(both, np.random.default_rng(31))
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(16)
        for label, o in OPTS.items():
            co = _split(o)
            c_offs, chains, cseeds = _want(model, _sa(name), seps, reads, **co)
            trace = []
            want = er.reference(c_offs, chains, cseeds, reads, text, seps, trace=trace, **o)
            offs, regs = b.regions(reads, **o)
            assert regs.dtype == api.REGION_DTYPE
            assert offs.tolist() == want[0], label
            assert er.as_tuples(regs) == want[1], label
            assert _over_chains(b, reads, text, seps, **o) == want, label
            _SEEN.update(x for x in trace if isinstance(x, str))
            _SEEN.update(f"strand{s}" for s in set(regs["strand"].tolist()))
            if label == "asym_small_w":
                assert (regs["w"] > ASYM["w"]).any() or "retry" not in trace
    if name == CASES[-1]:
        want = {"skip", "left_local", "left_end", "right_local", "right_end", "qbeg0", "qend_L", "flt", "strand0", "strand1"}
        assert want <= _SEEN, want - _SEEN


def test_repeat_poly_a_megabase_and_indels():
    rng = np.random.default_rng(9)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    unit = acgt[rng.integers(0, 4, 40)].tobytes()
    recs = [bytearray(acgt[rng.integers(0, 4, 150_000)].tobytes()) for _ in range(2)]
    for j in range(1100):
        r = recs[j % 2]
        p = 100 * (j // 2) + 30
        r[p:p + 40] = unit
    recs = [bytes(r) for r in recs]
    recs += [b"A" * 3000 + recs[0][:500], recs[1][:200] + b"A" * 2500 + recs[1][200:500]]
    big = acgt[rng.integers(0, 4, 1_100_000)].tobytes()
    recs.append(big)
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    reads = [recs[0][100 * k:100 * k + 150] for k in (3, 40, 200)] + [_mutate(recs[1][100 * k + 10:100 * k + 130], rng, 2) for k in (7, 77)]
    reads += [b"GATTACA" + unit + b"CAT", unit, b"A" * 2000, b"G" + b"A" * 2000 + b"C", big[50_000:1_050_000]]
    for k in range(3):                                                          # a 20-base piece of another record: its seed is dropped
        a = int(rng.integers(0, len(big) - 1000))
        p = int(rng.integers(0, 100_000))
        reads.append(big[a:a + 400] + recs[0][p:p + 20] + big[a + 400:a + 800])
    for k, indel in enumerate((5, 10, 60, 120) * 3):                               # 2-20 kbp reads with an insertion or a deletion
        L = int(rng.integers(2000, 20_000))
        a = int(rng.integers(0, len(big) - L - indel))
        seg = bytearray(big[a:a + L + indel])
        mid = L // 2
        q = seg[:mid] + seg[mid + indel:] if k % 2 else seg[:mid] + acgt[rng.integers(0, 4, indel)].tobytes() + seg[mid:L]
        q = _mutate(bytes(q), rng, L // 200)
        reads.append(q if k % 3 else api.both_strands([q])[1])
    trace = []
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(32)
        for o in ({}, ASYM):
            want = _over_chains(b, reads, text, seps, trace=trace, **o)
            offs, regs = b.regions(reads, **o)
            assert offs.tolist() == want[0] and er.as_tuples(regs) == want[1]
        c_offs = b.chains(reads)[0]
    n_chains, n_regs = np.diff(c_offs.astype(np.int64)), np.diff(offs.astype(np.int64))
    assert n_chains[:7].max() >= 100 and n_regs[:7].max() >= 100                # reads on the repeat: hundreds of chains
    assert {"skip", "revived", "retry", "flt", "dropped", "empty"} <= set(x for x in trace if isinstance(x, str))
    mega = regs[int(offs[9]):int(offs[10])]
    assert mega.size and int(mega["qe"][0] - mega["qb"][0]) == 1_000_000


def test_loaded_result_of_another_text(tmp_path):
    both, text, seps, model = _case("c4_like_5x100k")
    reads = _reads(both, np.random.default_rng(77))
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        b.sample_sa(32)
        want = b.regions(reads)
        words, sharp, dollar = b.result()
    api.write_outputs(str(tmp_path / "c4.bwt"), words, sharp, dollar)
    both2, text2, seps2, _ = _case("c3_like_600k_3rec")
    reads2 = _reads(both2, np.random.default_rng(78))
    with api.BwtBuilder() as c:
        w, s, d = api.read_outputs(str(tmp_path / "c4.bwt"), text.size)
        c.set_result(w, text.size, s, d)
        c.sample_sa(16)
        got = c.regions(reads)
        assert all((x == y).all() for x, y in zip(got, want))
        with api.BwtBuilder() as e:
            e.set_records(both2)
            e.build()
            w2, s2, d2 = e.result()
        c.set_result(w2, text2.size, s2, d2)                                    # the pac is derived again after sample_sa
        c.sample_sa(32)
        offs, regs = c.regions(reads2)
        assert (offs.tolist(), er.as_tuples(regs)) == _over_chains(c, reads2, text2, seps2)


def test_errors():
    recs = [r.upper().encode() for r in golden()["small"]["haplotypes_6x1500"]["records"]]
    both = api.both_strands(recs)
    L = binding.lib()
    SENT = 0xA5A5A5A5A5A5A5A5

    def raw(bld, reads, cap=1000, offs=None, null="", seed_kw=None, chain_kw=None, **kw):
        so = {**dict(min_len=19, split_width=10, max_mem_intv=20, max_occ=500, split_factor=1.5), **(seed_kw or {})}
        sopts = api.SeedOpts(so["min_len"], so["split_width"], so["max_mem_intv"], so["max_occ"], so["split_factor"])
        c = {**cr.DEFAULTS, **(chain_kw or {})}
        copts = api.ChainOpts(c["w"], c["max_chain_gap"], c["min_chain_weight"], c["max_chain_extend"], c["mask_level"], c["drop_ratio"])
        e = {**er.DEFAULTS, **kw}
        eopts = api.ExtOpts(*(e[f] for f, _ in api.ExtOpts._fields_))
        blob = np.frombuffer(b"".join(reads) + b"\0", dtype=np.uint8)
        if offs is None:
            offs = np.concatenate(([0], np.cumsum([len(r) for r in reads]))).astype(np.uint64)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        ro = np.full(len(reads) + 1, SENT, dtype=np.uint64)
        rg = np.zeros(max(cap, 1) + 4, dtype=api.REGION_DTYPE)
        rg["rb"] = SENT
        P = lambda name, a: None if null == name else api._ptr(a)  # noqa: E731
        rc = L.debwt_index_regions(bld._h, P("reads", blob), P("offsets", offs), len(reads),
                                   None if null == "seed_opts" else ctypes.addressof(sopts),
                                   None if null == "chain_opts" else ctypes.addressof(copts),
                                   None if null == "ext_opts" else ctypes.addressof(eopts), P("region_offsets", ro), P("regions", rg), cap)
        return rc, ro, rg, L.debwt_last_error().decode()

    def untouched(ro, rg):
        return (ro == SENT).all() and (rg["rb"] == SENT).all()

    reads = [q[100:180] for q in both] + [b"ACGTN" * 9]
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.index()
        rc, ro, rg, msg = raw(b, reads)                                         # no samples
        assert rc != 0 and "debwt_index_sample_sa" in msg and untouched(ro, rg)
        with pytest.raises(DebwtError, match="sample_sa"):
            b.regions(reads)
        b.sample_sa(32)
        offs, regs = b.regions(reads)
        total = int(offs[-1])
        assert total >= len(reads) - 1
        rc, ro, rg, msg = raw(b, reads, total - 1)                              # too small: names the total, writes offsets only
        assert rc != 0 and str(total) in msg and (ro == offs).all() and (rg["rb"] == SENT).all()
        rc, ro, rg, msg = raw(b, reads, total)
        assert rc == 0 and (ro == offs).all() and (rg[:total] == regs).all() and (rg["rb"][total:] == SENT).all()
        rc, ro, rg, msg = raw(b, reads, 0, null="regions")                      # size query
        assert rc == 0 and (ro == offs).all() and (rg["rb"] == SENT).all()
        bad = [(dict(a=0), "a"), (dict(e_del=0), "e_del"), (dict(e_ins=0), "e_ins"), (dict(b=-1), "b"), (dict(o_del=-1), "o_del"),
               (dict(o_ins=-2), "o_ins"), (dict(pen_clip5=-1), "pen_clip5"), (dict(pen_clip3=-1), "pen_clip3"), (dict(zdrop=-1), "zdrop"),
               (dict(a=128), "a"), (dict(b=200), "b"), (dict(e_del=1 << 24), "2^31")]
        for kw, word in bad:
            rc, ro, rg, msg = raw(b, reads, **kw)
            assert rc != 0 and word in msg and "index_regions" in msg and untouched(ro, rg), kw
        for kw, word in ((dict(w=1025), "w"), (dict(w=-1), "w"), (dict(max_chain_gap=-1), "max_chain_gap"),
                         (dict(mask_level=float("nan")), "mask_level")):
            rc, ro, rg, msg = raw(b, reads, chain_kw=kw)
            assert rc != 0 and word in msg and "index_regions" in msg and untouched(ro, rg), kw
        rc, ro, rg, msg = raw(b, reads, chain_kw=dict(w=1024))
        assert rc == 0 and int(ro[-1]) >= 1
        for kw, word in ((dict(min_len=0), "min_seed_len"), (dict(max_occ=0), "max_occ"), (dict(split_factor=-1.0), "split_factor")):
            rc, ro, rg, msg = raw(b, reads, seed_kw=kw)
            assert rc != 0 and word in msg and "index_regions" in msg and untouched(ro, rg), kw
        for null in ("reads", "offsets", "region_offsets", "seed_opts", "chain_opts", "ext_opts"):
            rc, ro, rg, msg = raw(b, reads, null=null)
            assert rc != 0 and "null argument" in msg and untouched(ro, rg), null
        rc, ro, rg, msg = raw(b, [b"A" * 40] * 3, offs=np.array([0, 60, 50, 120], dtype=np.uint64))
        assert rc != 0 and "read 1" in msg and untouched(ro, rg)
        rc, ro, rg, msg = raw(b, [], 0)                                         # no reads
        assert rc == 0 and int(ro[0]) == 0 and (ro[1:] == SENT).all()
        o, r = b.regions([])
        assert o.tolist() == [0] and r.size == 0
        o, r = b.regions([b"", b"NNNN", b"ACG"])                                 # no hits
        assert o.tolist() == [0, 0, 0, 0] and r.size == 0
        o, r = b.regions(reads, min_chain_weight=10 ** 6)                        # no chains
        assert (o == 0).all() and r.size == 0
    with api.BwtBuilder() as b:                                                 # one strand only: unbalanced
        b.set_records(recs)
        b.build()
        b.sample_sa(32)
        rc, ro, rg, msg = raw(b, reads)
        assert rc != 0 and "reverse complement" in msg and "index_regions" in msg and untouched(ro, rg)


def test_steady_batches_run_once():
    """a stream of batches that fit the builder's buffer costs one pass each: the launch count per call does not change"""
    both, text, seps, _ = _case("c4_like_5x100k")
    reads = _reads(both, np.random.default_rng(5))
    L = binding.lib()
    with api.BwtBuilder() as b:
        b.set_records(both)
        b.build()
        b.sample_sa(32)
        b.regions(reads)
        n0 = L.debwt_launch_count()
        b.regions(reads)
        n1 = L.debwt_launch_count()
        b.regions(reads[:100])
        n2 = L.debwt_launch_count()
    assert n1 - n0 == n2 - n1
