"""CPU side of SMEM search: the FMD-index model of tests/smem_ref.py against the brute-force definition, Li's MEM definition,
the suffix array and reverse-complement symmetry; both_strands, strand_offsets and the SMEM_DTYPE mirror of debwt_smem."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from tests import smem_ref as ref
from tests.locate_ref import suffix_array
from tests.util import golden

_LUT = np.full(256, 255, dtype=np.uint8)
for _c, _v in ((b"A", 0), (b"C", 1), (b"G", 2), (b"T", 3), (b"#", 4), (b"$", 5)):
    _LUT[_c[0]] = _v


def _fmd_text(records):
    """(upper-case text bytes, symbol codes) of T built from `records` and their reverse complements"""
    text, _ = api.join_records(api.both_strands(records))
    return text.tobytes(), _LUT[text]


def _reads(records, rng, k):
    """k seeded reads: pieces of either strand, some with substitutions, 'N' or lower case, pieces across two records,
    random bases and poly-A"""
    both = api.both_strands(records)
    acgt = b"ACGT"
    out = []
    for j in range(k):
        r = both[int(rng.integers(0, len(both)))]
        a = int(rng.integers(0, len(r)))
        q = bytearray(r[a:a + int(rng.integers(1, 40))])
        kind = j % 6
        if kind == 1 and q:
            for _ in range(int(rng.integers(1, 4))):
                q[int(rng.integers(0, len(q)))] = acgt[int(rng.integers(0, 4))]
        elif kind == 2 and q:
            q[int(rng.integers(0, len(q)))] = ord("N")
            q = bytearray(bytes(q[:len(q) // 2]).lower() + bytes(q[len(q) // 2:]))
        elif kind == 3:
            nxt = both[int(rng.integers(0, len(both)))]
            q = bytearray(r[-int(rng.integers(1, 15)):] + nxt[:int(rng.integers(1, 15))])
        elif kind == 4:
            q += bytes(acgt[int(x)] for x in rng.integers(0, 4, int(rng.integers(0, 10))))
        elif kind == 5:
            q = bytearray(b"A" * int(rng.integers(1, 45)))
        out.append(bytes(q))
    return out + [b"", b"N", b"A", b"acgtNNacgt"]


def _random_records(rng):
    recs = []
    for _ in range(int(rng.integers(1, 5))):
        r = bytes(b"ACGT"[int(x)] for x in rng.integers(0, 4, int(rng.integers(5, 70))))
        if rng.random() < 0.3:
            r = b"A" * int(rng.integers(3, 30)) + r
        recs.append(r)
    return recs


def _check_model_against_brute(records, reads):
    text, sym = _fmd_text(records)
    model = ref.FmdModel(sym)
    for q in reads:
        got = model.smems(q)
        assert [(s, e) for s, e, *_ in got] == ref.brute_smems(q, text), q
        for s, e, k, l, cnt in got:
            assert (k, l, cnt) == model.interval(q[s:e].upper()), q
            assert cnt == sum(1 for i in range(len(text)) if text.startswith(q[s:e].upper(), i))
    return model


@pytest.mark.parametrize("name", sorted(golden()["small"]))
def test_model_equals_brute_force_golden(name):
    recs = [r.encode() for r in golden()["small"][name]["records"]]
    _check_model_against_brute(recs, _reads(recs, np.random.default_rng(len(name)), 60))


@pytest.mark.parametrize("seed", range(12))
def test_model_equals_brute_force_random(seed):
    rng = np.random.default_rng(100 + seed)
    recs = _random_records(rng)
    _check_model_against_brute(recs, _reads(recs, rng, 40))


def test_text_without_some_bases():
    """a base that T does not hold ends every match: no interval starts from it"""
    recs = [b"AT" * 20, b"AAT" * 12]
    text, sym = _fmd_text(recs)
    model = ref.FmdModel(sym)
    for q in [b"ACA", b"ATATGATAT", b"GGGG", b"CATATATC", b"TAAT"]:
        assert [(s, e) for s, e, *_ in model.smems(q)] == ref.brute_smems(q, text)
    assert [(s, e) for s, e, *_ in model.smems(b"ACA")] == [(0, 1), (2, 3)]


@pytest.mark.parametrize("seed", range(6))
def test_bi_intervals_against_suffix_array(seed):
    """backward-only and forward-only extension give the rows that the suffix array shows for P and rc(P)"""
    rng = np.random.default_rng(200 + seed)
    recs = _random_records(rng)
    text, sym = _fmd_text(recs)
    model = ref.FmdModel(sym)
    sa = suffix_array(sym).astype(np.int64)
    suf = [text[p:] for p in sa.tolist()]

    def rows(p):
        r = [i for i, s in enumerate(suf) if s.startswith(p)]
        assert r == list(range(r[0], r[0] + len(r))) if r else True
        return (r[0] if r else None), len(r)

    for _ in range(60):
        p = bytes(b"ACGT"[int(x)] for x in rng.integers(0, 4, int(rng.integers(1, 7))))
        if rng.random() < 0.5:                                   # a piece of T
            a = int(rng.integers(0, len(text) - 6))
            p = text[a:a + int(rng.integers(1, 6))]
            if p.translate(None, b"ACGT"):
                continue
        (k, cnt), (l, cnt_rc) = rows(p), rows(ref.revcomp(p))
        assert cnt == cnt_rc
        back = model.interval(p)
        fwd = model.empty()
        for a in ref.codes(p):
            fwd = model.forward(fwd, a)
        assert back[2] == fwd[2] == cnt, p
        if cnt:
            assert back[:2] == fwd[:2] == (k, l), p
    # every SMEM's rows
    for q in _reads(recs, rng, 30):
        for s, e, k, l, cnt in model.smems(q):
            assert rows(q[s:e].upper()) == (k, cnt) and rows(ref.revcomp(q[s:e]).upper()) == (l, cnt)


@pytest.mark.parametrize("seed", range(8))
def test_li_definition_equals_start_characterisation(seed):
    rng = np.random.default_rng(300 + seed)
    recs = _random_records(rng)
    text, _ = _fmd_text(recs)
    for q in _reads(recs, rng, 30):
        assert ref.li_smems(q, text) == ref.brute_smems(q, text), q


@pytest.mark.parametrize("seed", range(6))
def test_reverse_complement_symmetry(seed):
    """the SMEMs of rc(q) are [m - e, m - s) with row and rc_row swapped"""
    rng = np.random.default_rng(400 + seed)
    recs = _random_records(rng)
    _, sym = _fmd_text(recs)
    model = ref.FmdModel(sym)
    for q in _reads(recs, rng, 40):
        m = len(q)
        want = sorted((m - e, m - s, l, k, c) for s, e, k, l, c in model.smems(q))
        assert model.smems(ref.revcomp(q)) == want, q


def test_min_len_filters():
    rng = np.random.default_rng(5)
    recs = _random_records(rng)
    _, sym = _fmd_text(recs)
    model = ref.FmdModel(sym)
    for q in _reads(recs, rng, 40):
        full = model.smems(q)
        for k in (2, 5, 19):
            assert model.smems(q, k) == [x for x in full if x[1] - x[0] >= k]


def test_smems_by_count_equals_model():
    rng = np.random.default_rng(6)
    recs = _random_records(rng) + [b"ACGTTGCAGT" * 4]
    text, sym = _fmd_text(recs)
    model = ref.FmdModel(sym)
    reads = _reads(recs, rng, 50)

    def count(pats):
        return [sum(1 for i in range(len(text)) if text.startswith(p.upper(), i)) if not p.upper().translate(None, b"ACGT") else 0
                for p in pats]

    got = ref.smems_by_count(count, reads, 3)
    assert got == [[(s, e, c) for s, e, _, _, c in model.smems(q, 3)] for q in reads]


def test_both_strands_layout():
    recs = ["ACGTTa", b"ggCAT", np.frombuffer(b"TTTTAC", dtype=np.uint8)]
    assert api.both_strands(recs) == [b"ACGTTA", b"GGCAT", b"TTTTAC", b"TAACGT", b"ATGCC", b"GTAAAA"]
    assert api.both_strands([]) == []
    for bad in (["ACGN"], ["ACGT", "AC-T"], ["acgtr"], [b"ACGT\n"]):
        with pytest.raises(DebwtError, match="both_strands"):
            api.both_strands(bad)


def test_strand_offsets_round_trip():
    rng = np.random.default_rng(8)
    recs = [bytes(b"ACGT"[int(x)] for x in rng.integers(0, 4, n)) for n in (50, 33, 80)]
    both = api.both_strands(recs)
    text, seps = api.join_records(both)
    t = text.tobytes()
    starts = np.concatenate(([0], seps[:-1] + 1)).astype(np.int64)
    for L in (1, 5, 33):
        pos, want = [], []
        for j, r in enumerate(both):
            for o in (0, len(r) - L, (len(r) - L) // 3):
                pos.append(int(starts[j]) + o)
                i = j % 3
                want.append((i, int(j >= 3), o if j < 3 else len(recs[i]) - o - L))
        rec, strand, off = api.strand_offsets(np.array(pos, dtype=np.uint64), L, seps)
        assert list(zip(rec.tolist(), strand.tolist(), off.tolist())) == want
        for p, (i, s, o) in zip(pos, want):                          # the hit's bases on the forward strand
            hit = t[p:p + L]
            assert (ref.revcomp(hit) if s else hit) == recs[i][o:o + L]
    with pytest.raises(ValueError):
        api.strand_offsets([int(seps[0]) - 2], 5, seps)
    with pytest.raises(ValueError):
        api.strand_offsets([0], 1, seps[:3])
    r, s, o = api.strand_offsets(np.array([], dtype=np.uint64), 4, seps)
    assert r.size == s.size == o.size == 0


def test_smem_dtype_matches_header_layout(tmp_path):
    fields = list(api.SMEM_DTYPE.names)
    src = tmp_path / "smem.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "debwt_b200.h"\nint main(void){printf("%zu", sizeof(debwt_smem));'
                   + "".join('printf(" %%zu", offsetof(debwt_smem, %s));' % f for f in fields) + "return 0;}\n")
    exe = tmp_path / "smem"
    subprocess.check_call(["gcc", "-I", os.path.dirname(binding.HEADER), "-o", str(exe), str(src)])
    out = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert fields == ["row", "rc_row", "count", "qbeg", "qend"]
    assert out[0] == api.SMEM_DTYPE.itemsize == 32
    assert out[1:] == [api.SMEM_DTYPE.fields[f][1] for f in fields]
    assert ctypes.sizeof(ctypes.c_uint64) * 3 + 8 == 32
