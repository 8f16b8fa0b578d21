"""CPU side of BWA-MEM seed collection: the restatement of tests/seed_ref.py against definitions computed from the bytes of
T (round 1 = the SMEMs, each round-2 smem1 call = the maximal pieces through its middle that occur often enough, round 3 =
a brute-force walk of its rule, hit rows = row + j step), on texts with repeats where every round fires; split_len and
the SEED_DTYPE / HIT_DTYPE / SeedOpts mirrors of include/debwt_b200.h against a C compiler."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from debwt_b200 import api, binding
from tests import seed_ref as sr
from tests import smem_ref as ref
from tests.locate_ref import suffix_array

_LUT = np.full(256, 255, dtype=np.uint8)
for _c, _v in ((b"A", 0), (b"C", 1), (b"G", 2), (b"T", 3), (b"#", 4), (b"$", 5)):
    _LUT[_c[0]] = _v


def _rand(rng, k):
    return bytes(b"ACGT"[int(x)] for x in rng.integers(0, 4, k))


def _repeat_records(rng):
    """six 1500-base records holding 14 copies of a 60-base unit and 30 copies of a 24-base unit"""
    recs = [bytearray(_rand(rng, 1500)) for _ in range(6)]
    for unit, copies in ((_rand(rng, 60), 14), (_rand(rng, 24), 30)):
        for j in range(copies):
            r = recs[j % 6]
            p = int(rng.integers(0, len(r) - len(unit)))
            r[p:p + len(unit)] = unit
    return [bytes(r) for r in recs]


def _reads(both, rng, k):
    """pieces of either strand, some with substitutions, an 'N' or lower case, and poly-A"""
    out = []
    for j in range(k):
        r = both[int(rng.integers(0, len(both)))]
        L = int(rng.integers(40, 150))
        a = int(rng.integers(0, len(r) - L))
        q = bytearray(r[a:a + L])
        if j % 4 == 1:
            for p in rng.integers(0, L, int(rng.integers(1, 3))).tolist():
                q[p] = b"ACGT"[(b"ACGT".index(q[p]) + 1) % 4]
        elif j % 4 == 2:
            q[int(rng.integers(0, L))] = ord("N")
            q = bytearray(bytes(q[:L // 2]).lower() + bytes(q[L // 2:]))
        out.append(bytes(q))
    return out + [b"A" * 45, b"", b"NNNN", b"acgt"]


def _setup(seed):
    rng = np.random.default_rng(seed)
    recs = _repeat_records(rng)
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    sym = _LUT[text]
    return both, text.tobytes(), seps, ref.FmdModel(sym), sym, _reads(both, rng, 60)


OPTS = [dict(sr.DEFAULTS), dict(min_len=12, split_factor=1.0, split_width=20, max_mem_intv=0, max_occ=3)]


@pytest.mark.parametrize("seed", range(3))
@pytest.mark.parametrize("opt", range(len(OPTS)))
def test_rounds_against_definitions(seed, opt):
    o = OPTS[opt]
    both, text, seps, model, sym, reads = _setup(500 + seed)
    fired = {1: 0, 2: 0, 3: 0}
    sl = sr.split_len(o["min_len"], o["split_factor"])
    for q in reads:
        got = sr.seeds(model, q, **o)
        assert got == sorted(got, key=lambda t: t[:3])
        for b, e, r, k, l, s in got:
            fired[r] += 1
            assert (k, l, s) == model.interval(q[b:e].upper()) and s == sr.count_in(text, q[b:e].upper()) >= 1
            assert e - b >= o["min_len"]
        # round 1: the SMEMs
        r1 = [t for t in got if t[2] == 1]
        assert [(b, e, 1, k, l, s) for b, e, k, l, s in model.smems(q, o["min_len"])] == r1
        # round 2: every smem1 call through a middle, where the middle base occurs often enough
        want2 = []
        for b, e, _, _, _, s in r1:
            if e - b < sl or s > o["split_width"]:
                continue
            x, t = (b + e) >> 1, s + 1
            out = []
            sr.smem1(model, ref.codes(q), x, out, t)
            if sr.count_in(text, q[x:x + 1].upper()) >= t:
                assert sorted((p[0], p[1]) for p in out) == sr.smem1_by_definition(q, text, x, t), (q, x, t)
            want2 += [(p[0], p[1]) for p in out if p[1] - p[0] >= o["min_len"]]
        assert sorted(want2) == [(b, e) for b, e, r, *_ in got if r == 2]
        # round 3: a walk of its rule with counts from the text
        want3 = sr.round3_by_walk(q, text, o["min_len"], o["max_mem_intv"]) if o["max_mem_intv"] > 0 else []
        assert want3 == [(b, e, s) for b, e, r, k, l, s in got if r == 3]
    assert fired[1] and fired[2], fired
    assert bool(fired[3]) == (o["max_mem_intv"] > 0), fired


def test_hits_are_sampled_rows():
    both, text, seps, model, sym, reads = _setup(600)
    sa = suffix_array(sym)
    for mo in (500, 7, 3, 1):
        offs, seeds, hits = sr.reference(model, sa, seps, reads, **{**sr.DEFAULTS, "max_occ": mo})
        assert offs[-1] == len(seeds) and len(hits) == sum(s[7] for s in seeds)
        stepped = 0
        for b, e, r, k, l, s, hb, nh in seeds:
            rows = sr.hit_rows(k, s, mo)
            step = s // mo if s > mo else 1
            stepped += step > 1
            assert nh == min(s, mo) and rows == [k + j * step for j in range(nh)] and rows[-1] < k + s
            for j, (pos, off, rec, strand) in enumerate(hits[hb:hb + nh]):
                assert pos == int(sa[rows[j]])
                piece = text[pos:pos + e - b]
                fwd = both[rec][off:off + e - b]
                assert (ref.revcomp(piece) if strand else piece) == fwd
                assert rec < len(both) // 2
        assert stepped or mo > 3                                     # step > 1 fires at the small max_occ


def test_base_missing_from_text():
    """a base that T does not hold is stepped over in every round"""
    recs = [b"AT" * 40 + b"AAT" * 30, b"TTA" * 50]
    both = api.both_strands(recs)
    text, _ = api.join_records(both)
    model = ref.FmdModel(_LUT[text])
    t = text.tobytes()
    for q in [b"ATATATATATCATATATATATATATAT", b"GGGGATTAATTAATTAATTAATT", b"AATAATAATAATAATAATGAATAATAATAATAATAAT"]:
        got = sr.seeds(model, q, min_len=5, split_factor=1.0, split_width=10, max_mem_intv=4)
        assert [(b, e, s) for b, e, r, k, l, s in got if r == 3] == sr.round3_by_walk(q, t, 5, 4)
        assert all(b"C" not in q[b:e] and b"G" not in q[b:e] for b, e, *_ in got)


@pytest.mark.parametrize("seed", range(3))
def test_smem1_at_threshold_one_is_the_model_loop(seed):
    """min_intv = 1 is Li's smem1 of tests/smem_ref.py, call by call"""
    both, text, seps, model, sym, reads = _setup(700 + seed)
    for q in reads:
        c = ref.codes(q)
        for x in range(len(c)):
            if c[x] > 3 or model.single(c[x])[2] == 0:
                continue
            a, b = [], []
            assert sr.smem1(model, c, x, a) == model.smem1(c, x, b) and a == b, (q, x)


def test_split_len_is_a_float_product():
    assert sr.split_len(19, 1.5) == 28
    assert sr.split_len(1, 2.501) == 2                               # 3 in double arithmetic


def test_dtypes_match_header_layout(tmp_path):
    structs = {"debwt_seed": api.SEED_DTYPE, "debwt_seed_hit": api.HIT_DTYPE}
    body = ""
    for name, dt in structs.items():
        body += f'printf("%zu ", sizeof({name}));' + "".join(f'printf("%zu ", offsetof({name}, {f}));' for f in dt.names)
    opts = [f for f, _ in api.SeedOpts._fields_]
    body += 'printf("%zu ", sizeof(debwt_seed_opts));' + "".join(f'printf("%zu ", offsetof(debwt_seed_opts, {f}));' for f in opts)
    pairs = [(19, 1.5), (1, 2.501), (7, 1.3), (33, 0.55), (10, 2.45)]
    body += "".join(f'{{uint32_t k = {k}; float s = {s}f; printf("%d ", (int)(k * s + .499));}}' for k, s in pairs)
    src = tmp_path / "seeds.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "debwt_b200.h"\nint main(void){' + body + "return 0;}\n")
    exe = tmp_path / "seeds"
    subprocess.check_call(["gcc", "-I", os.path.dirname(binding.HEADER), "-o", str(exe), str(src)])
    out = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert list(api.SEED_DTYPE.names) == ["row", "rc_row", "count", "qbeg", "qend", "hit_begin", "n_hits", "round"]
    assert list(api.HIT_DTYPE.names) == ["pos", "offset", "record", "strand"]
    for name, dt in structs.items():
        assert out[0] == dt.itemsize and out[1:1 + len(dt.names)] == [dt.fields[f][1] for f in dt.names], name
        out = out[1 + len(dt.names):]
    assert out[0] == ctypes.sizeof(api.SeedOpts) and out[1:1 + len(opts)] == [getattr(api.SeedOpts, f).offset for f in opts]
    assert out[1 + len(opts):] == [sr.split_len(k, s) for k, s in pairs]
