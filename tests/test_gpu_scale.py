"""The single-GPU path at the size limit of one device call: N < 2^32 - 64 symbols and N - 32 R < 2^32 - 65536 keys.

Nearly every index on the hot path is a u32 sized for that limit (sort offsets, key index, branch table, list-ranking
nodes, sampled SA values), and several branches only switch at large N (28-bit key index, bitonic sentinel sort, key
histograms when 2048 R > N).  These tests
  a. check that the input calls accept exactly the texts the sort can take (nothing large is allocated),
  b. sort 2^32 - 65537 keys with the library's radix sort and check order, permutation and the 28-bit key index,
  c. build three texts above 2^31 symbols (one at the limit) and check the BWT, the FM-index tables, the sampled SA and
     locate against references computed here from the text (numpy / torch), not by the library.
A sort test needs about 75 GB of HBM; a whole-path case up to about 115 GB (measured at the limit: the build's arena,
then the verifier's and the sampler's scratch in a second context) and 25 GB of host memory.  A test skips, naming the
amount, when that memory is not free."""
import bisect
import ctypes
import gc
import json
import time

import numpy as np
import pytest
import torch

from debwt_b200 import api, binding
from debwt_b200.binding import DebwtError
from oracle import stages as st

pytestmark = [pytest.mark.gpu, pytest.mark.slow]

GB = 1 << 30
SORT_MAX_KEYS = (1 << 32) - 65537          # radix_sort_u64 takes fewer than 2^32 - 65536 keys
M64 = (1 << 64) - 1


def n_max(R):
    """largest N one device call takes for R records"""
    return min(SORT_MAX_KEYS + 32 * R, (1 << 32) - 65)


def _s64(v):
    v &= M64
    return v - (1 << 64) if v >> 63 else v


def _release_device_memory():
    """hand memory that earlier tests left cached back to the driver: torch's cache, builders still waiting for the
    garbage collector, and the stream-ordered allocations the library returned to the device's default pool (whose
    release threshold it raises so that repeated builds keep it)"""
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    cu = ctypes.CDLL("libcuda.so.1")
    dev, pool = ctypes.c_int(), ctypes.c_void_p()
    assert cu.cuDeviceGet(ctypes.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(ctypes.byref(pool), dev) == 0
    assert cu.cuMemPoolTrimTo(pool, ctypes.c_size_t(0)) == 0


def _need(dev_gb, host_gb=0):
    _release_device_memory()
    free, _ = torch.cuda.mem_get_info(0)
    if free < dev_gb * GB:
        pytest.skip(f"needs about {dev_gb} GB of free device memory, {free / GB:.1f} GB free")
    if host_gb:
        avail = 0
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    avail = int(line.split()[1]) * 1024
        if avail < host_gb * GB:
            pytest.skip(f"needs about {host_gb} GB of free host memory, {avail / GB:.1f} GB available")


class _Peak:
    """highest device memory in use seen at the checkpoints of one test (the library's arena is not torch's, so the
    driver's view is sampled)"""

    def __init__(self):
        self.peak = 0

    def __call__(self):
        free, total = torch.cuda.mem_get_info(0)
        self.peak = max(self.peak, total - free)


def _report(name, t0, peak, **kw):
    print(json.dumps({"test": name, "wall_s": round(time.time() - t0, 1), "peak_device_gb": round(peak.peak / GB, 1), **kw}))


def _even_seps(n, R):
    return ((np.arange(1, R + 1, dtype=np.uint64) * np.uint64(n)) // np.uint64(R) - np.uint64(1)).astype(np.uint64)


# ---- a. the size limit ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("R", [1, 24, 1000])
def test_input_size_limit(R):
    """set_text_device checks the separators and keeps the pointer; it never reads the text, so a 64-byte buffer stands
    in for a text of any claimed length"""
    buf = torch.zeros(64, dtype=torch.uint8, device="cuda:0")
    top = n_max(R)
    assert top == min((1 << 32) - 65537 + 32 * R, (1 << 32) - 65)
    if R == 1:
        assert top == (1 << 32) - 65505
    with api.BwtBuilder(0) as b:
        b.set_text_device(buf.data_ptr(), top, _even_seps(top, R))
        for n in (top + 1, (1 << 32) - 65):
            if n <= top:
                continue
            with pytest.raises(DebwtError, match=r"2\^32 - 65536") as e:
                b.set_text_device(buf.data_ptr(), n, _even_seps(n, R))
            msg = str(e.value)
            assert str(n) in msg and f"R = {R} " in msg and "2^32 - 64" in msg
        with pytest.raises(DebwtError, match="no input"):          # a refused input leaves nothing to build
            b.build()


# ---- b. the sort at its limit -----------------------------------------------------------------------------------------
_GOLD, _C1, _C2 = 0x9E3779B97F4A7C15, 0xBF58476D1CE4E5B9, 0x94D049BB133111EB
_CHUNK = 1 << 27


def _srl(x, k):
    """logical right shift of int64 values"""
    return (x >> k) & ((1 << (64 - k)) - 1)


def _splitmix(z):
    """splitmix64 finaliser on int64 tensors (wrapping arithmetic)"""
    z = (z ^ _srl(z, 30)) * _s64(_C1)
    z = (z ^ _srl(z, 27)) * _s64(_C2)
    return z ^ _srl(z, 31)


def _xor_all(x):
    while x.numel() > 1:
        if x.numel() & 1:
            x = torch.cat([x, x.new_zeros(1)])
        h = x.numel() // 2
        x = x[:h] ^ x[h:]
    return int(x[0]) if x.numel() else 0


def _fingerprint(keys):
    """(count, wrapping sum, xor, wrapping sum of splitmix(key)): equal for two arrays that are permutations of each
    other, and a lost, duplicated or altered key changes them"""
    s = x = h = 0
    for i in range(0, keys.numel(), _CHUNK):
        c = keys[i:i + _CHUNK]
        s += int(c.sum())
        x ^= _xor_all(c)
        h += int(_splitmix(c).sum())
    return keys.numel(), s & M64, x & M64, h & M64


def _fill_keys(keys, kind):
    n = keys.numel()
    for i in range(0, n, _CHUNK):
        m = min(_CHUNK, n - i)
        z = _splitmix(torch.arange(i + 1, i + m + 1, dtype=torch.int64, device=keys.device) * _s64(_GOLD) + 12345)
        if kind == "top16_constant":
            z = (z & ((1 << 48) - 1)) | _s64(0xA5C3 << 48)
        elif kind == "three_values":
            z = torch.tensor([0, _s64(1 << 63), -1], dtype=torch.int64, device=keys.device)[_srl(z, 62) % 3]
        keys[i:i + m] = z


@pytest.mark.parametrize("kind", ["uniform", "top16_constant", "three_values"])
def test_sort_at_limit(kind):
    from debwt_b200 import dist
    _need(75)
    t0, peak = time.time(), _Peak()
    n = SORT_MAX_KEYS
    ops = dist.CudaOps(0)
    keys = torch.empty(n, dtype=torch.int64, device="cuda:0")
    _fill_keys(keys, kind)
    want = _fingerprint(keys)
    out = ops.sort(keys, timed=True)
    torch.cuda.synchronize()
    peak()
    sweeps = ops.sort_stats["sweeps"]
    assert sweeps == (6 if kind == "top16_constant" else 8)
    del keys
    idx, bits = ops.key_index(out)
    assert bits == 28
    torch.cuda.synchronize()
    assert _fingerprint(out) == want
    out.bitwise_xor_(_s64(1 << 63))                     # unsigned order == signed order of the flipped keys
    for i in range(0, n - 1, _CHUNK):
        c = out[i:i + _CHUNK + 1]
        assert bool((c[1:] >= c[:-1]).all()), f"not sorted in [{i}, {i + c.numel()})"
    nb = 1 << bits
    for t in range(0, nb, _CHUNK):
        q = (torch.arange(t, min(t + _CHUNK, nb), dtype=torch.int64, device=out.device) << (64 - bits)) ^ _s64(1 << 63)
        ref = torch.searchsorted(out, q)
        got = idx[t:t + q.numel()].to(torch.int64) & 0xFFFFFFFF
        bad = torch.nonzero(got != ref)
        assert bad.numel() == 0, f"key index differs at bucket {t + int(bad[0])}"
    assert int(idx[nb]) & 0xFFFFFFFF == n
    peak()
    del out, idx
    torch.cuda.empty_cache()
    # one key more than the limit: refused before any memory is touched (the buffers are a few bytes)
    small = torch.zeros(64, dtype=torch.int64, device="cuda:0")
    in_b = ctypes.c_int(0)
    rc = ops.L.debwt_dev_sort(dist._p(small), dist._p(small), dist._u64(n + 1), ops.sort_cfg, dist._p(small), ctypes.byref(in_b),
                              ops._st())
    assert rc != 0 and "2^32 - 65536" in binding.lib().debwt_last_error().decode()
    torch.cuda.synchronize()
    _report(f"sort_{kind}", t0, peak, sweeps=sweeps)


# ---- host references over the packed BWT ------------------------------------------------------------------------------
_LUT = np.full(256, 255, dtype=np.uint8)
for _c, _v in ((b"A", 0), (b"C", 1), (b"G", 2), (b"T", 3), (b"#", 4), (b"$", 5)):
    _LUT[_c[0]] = _v
_PAT = [0, 0x5555555555555555, 0xAAAAAAAAAAAAAAAA, M64]
_LO = 0x5555555555555555


def host_occ(words, n, sharp, dollar):
    """occ[w][c] = rows < 32 w holding base c (separator rows, stored as T, not counted), w = 0 .. ceil(N/32): a per-word
    popcount of the packed words and a cumsum, as an index with int64 counts"""
    nw = words.size
    tail = n - 32 * (nw - 1)                           # valid symbols of the last word
    valid = np.full(nw, M64, dtype=np.uint64)
    valid[-1] = np.uint64((M64 << (64 - 2 * tail)) & M64) & np.uint64(_LO | (_LO << 1))
    per = np.empty((nw, 4), dtype=np.int64)
    for c in range(4):
        x = words ^ np.uint64(_PAT[c])
        m = ~(x | (x >> np.uint64(1))) & np.uint64(_LO) & valid
        per[:, c] = np.bitwise_count(m)
    seprows = np.append(np.asarray(sharp, dtype=np.int64), int(dollar))
    per[:, 3] -= np.bincount(seprows >> 5, minlength=nw)
    occ = np.zeros((nw + 1, 4), dtype=np.int64)
    np.cumsum(per, axis=0, out=occ[1:])
    return occ


def c_array(occ, n, R):
    tot = occ[-1]
    return np.array([0, tot[0], tot[0] + tot[1], tot[0] + tot[1] + tot[2], n - R, n - 1], dtype=np.int64)


def bwt_at(words, sharp_sorted, dollar, rows):
    """BWT symbol codes (0..3 bases, 4 '#', 5 '$') of the given rows"""
    rows = np.asarray(rows, dtype=np.int64)
    w = words[rows >> 5]
    code = ((w >> (2 * (31 - (rows & 31))).astype(np.uint64)) & np.uint64(3)).astype(np.uint8)
    i = np.searchsorted(sharp_sorted, rows)
    is_sharp = (i < sharp_sorted.size) & (sharp_sorted[np.minimum(i, sharp_sorted.size - 1)] == rows)
    code[is_sharp] = 4
    code[rows == dollar] = 5
    return code


class HostLF:
    """LF mapping on the host from the packed words and host occ checkpoints (independent of index.cu)"""

    def __init__(self, words, occ, C, sharp_sorted, dollar):
        self.words, self.occ, self.C = words, occ, [int(x) for x in C]
        self.sharp = [int(x) for x in sharp_sorted]
        self.sharp_set = set(self.sharp)
        self.dollar = int(dollar)

    def step(self, r):
        """(BWT[r], LF(r))"""
        if r == self.dollar:
            return 5, self.C[5]
        if r in self.sharp_set:
            return 4, self.C[4] + bisect.bisect_left(self.sharp, r)
        w = int(self.words[r >> 5])
        j = r & 31
        c = (w >> (2 * (31 - j))) & 3
        x = w ^ _PAT[c]
        m = ~(x | (x >> 1)) & _LO
        before = (m >> (64 - 2 * j)).bit_count() if j else 0
        if c == 3:                                     # separator rows before r in this word are stored as T
            lo = r & ~31
            before -= bisect.bisect_left(self.sharp, r) - bisect.bisect_left(self.sharp, lo)
            before -= lo <= self.dollar < r
        return c, self.C[c] + int(self.occ[r >> 5][c]) + before

    def walk(self, sym, r, p, steps):
        """from row r with SA[r] = p, `steps` LF steps: each must read T[p - 1]; returns (row, position) reached"""
        n = sym.size
        for _ in range(steps):
            c, nxt = self.step(r)
            p = p - 1 if p else n - 1
            assert c == sym[p], f"LF walk: row {r} holds {c}, T[{p}] = {sym[p]}"
            r = nxt
        return r, p


def check_sa_rows(b, words, sharp_sorted, dollar, sym, rows):
    """SA values of `rows` (and of the row after each): below N, BWT[r] = T[SA[r] - 1], and the suffixes of consecutive
    rows in suffix order"""
    n = sym.size
    rows = np.unique(np.asarray(rows, dtype=np.int64))
    q = np.unique(np.concatenate([rows, rows[rows + 1 < n] + 1]))
    sa = b.sa(q.astype(np.uint64)).astype(np.int64)
    assert (sa < n).all()
    assert np.unique(sa).size == sa.size
    prev = np.where(sa > 0, sa - 1, n - 1)
    bad = np.flatnonzero(bwt_at(words, sharp_sorted, dollar, q) != sym[prev])
    assert bad.size == 0, f"BWT[{q[bad[0]]}] != T[SA - 1] (SA = {sa[bad[0]]})"
    val = dict(zip(q.tolist(), sa.tolist()))
    for r in rows.tolist():
        if r + 1 < n:
            assert st.suffix_less(sym, val[r], val[r + 1]), f"rows {r}, {r + 1}: suffixes {val[r]}, {val[r + 1]} out of order"
    return q, sa


def sa_probe_rows(n, sharp_sorted, rng):
    parts = [rng.integers(0, n, 10_000), np.arange(64), np.arange((1 << 31) - 64, (1 << 31) + 64), np.arange(n - 64, n)]
    k = rng.integers(1, n // 32, 2_000) * 32
    parts += [k - 1, k]
    s = sharp_sorted[::1000].astype(np.int64)
    parts += [s - 1, s, s + 1]
    rows = np.concatenate([np.asarray(p, dtype=np.int64) for p in parts])
    return rows[(rows >= 0) & (rows < n)]


def _find_all(raw, p):
    out, i = [], raw.find(p)
    while i >= 0:
        out.append(i)
        i = raw.find(p, i + 1)
    return out


def pick_patterns(sym, n, rng):
    """(origin, length) of base-only windows: spread over T, and some within 2^23 of its end"""
    out = []
    los = [int(x) for x in np.linspace(0, n - 400, 28)] + [int(x) for x in rng.integers(max(n - (1 << 23), 0), n - 400, 8)]
    for lo in los:
        L = int(rng.integers(16, 201))
        o = lo
        while (sym[o:o + L] > 3).any():
            o = int(rng.integers(max(lo - (1 << 20), 0), lo + 1))
        out.append((o, L))
    return out


def check_locate(b, raw, tnp, sym, seps, rng):
    n = sym.size
    origins = pick_patterns(sym, n, rng)
    pats = [raw[o:o + L] for o, L in origins]
    # repeat families: the 20-mers with the most hits among random candidates
    cand = []
    for o in rng.integers(0, n - 64, 256).tolist():
        if (sym[o:o + 20] < 4).all():
            cand.append(raw[o:o + 20])
    cnt = b.count(cand)
    top = np.argsort(-cnt.astype(np.int64), kind="stable")[:4]
    assert int(cnt[top[0]]) > 1, "no repeated 20-mer found among the candidates"
    pats += [cand[i] for i in top]
    hits, pos = b.locate(pats)
    counts = b.count(pats)
    assert (np.diff(hits.astype(np.int64)) == counts.astype(np.int64)).all()
    pos = pos.astype(np.int64)
    assert (pos < n).all()
    starts = np.concatenate([[0], seps[:-1].astype(np.int64) + 1])
    for i, p in enumerate(pats):
        got = pos[int(hits[i]):int(hits[i + 1])]
        L = len(p)
        assert got.size == np.unique(got).size, f"pattern {i}: duplicate positions"
        if i < len(origins):
            assert origins[i][0] in set(got.tolist()), f"pattern {i}: origin {origins[i][0]} not located"
        assert (got + L <= n).all()
        win = tnp[got[:, None] + np.arange(L)]
        assert (win == np.frombuffer(p, dtype=np.uint8)).all(), f"pattern {i}: a located position does not match T"
        rec, off = api.record_offsets(got.astype(np.uint64), seps)
        off = off.astype(np.int64)
        assert (starts[rec] + off == got).all() and (got + L <= seps[rec].astype(np.int64)).all()
    # no hit missing: a full scan of T for a few of them (random, near the end, repeated)
    for i in [0, 13, 27, len(origins) - 1] + list(range(len(origins), len(pats))):
        got = np.sort(pos[int(hits[i]):int(hits[i + 1])])
        assert got.tolist() == _find_all(raw, pats[i]), f"pattern {i}: located positions differ from a scan of T"
    return hits, pos, pats


# ---- c. the whole path at scale -------------------------------------------------------------------------------------
def _text_c3_at_limit():
    from debwt_b200 import synth_gpu
    R = 24
    text, seps = synth_gpu.config3(n_max(R) - R, R)
    assert text.numel() == n_max(R) and seps.size == R
    return text, seps


def _text_records():
    from debwt_b200 import synth_gpu
    seq = synth_gpu.genome_like((1 << 31) + (1 << 22), 7)
    per = seq.numel() // 4096
    text, seps = synth_gpu.join_records_device([seq[i * per:(i + 1) * per] for i in range(4096)])
    return text, seps


def _text_reads():
    from debwt_b200 import synth_gpu
    R, L = 1_400_000, 1550
    seq = synth_gpu.genome_like(R * L, 11)
    t = torch.empty((R, L + 1), dtype=torch.uint8, device=seq.device)
    t[:, :L] = seq.view(R, L)
    t[:, L] = ord("#")
    del seq
    text = t.view(-1)
    text[-1] = ord("$")
    seps = (np.arange(R, dtype=np.uint64) * np.uint64(L + 1) + np.uint64(L)).astype(np.uint64)
    return text, seps


CASES = {"c3_at_limit": _text_c3_at_limit, "records_past_2^31": _text_records, "reads_past_2^31": _text_reads}


@pytest.mark.parametrize("case", list(CASES))
def test_whole_path_at_scale(case):
    _need(116, 25)
    t0, peak = time.time(), _Peak()
    rng = np.random.default_rng(2024)
    text, seps = CASES[case]()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    n, R = text.numel(), seps.size
    assert n > (1 << 31) + 64 and n <= n_max(R)

    # 1. build, copy the result out, free the context
    with api.BwtBuilder(0) as b:
        b.set_text_device(text.data_ptr(), n, seps)
        b.build()
        peak()
        words, sharp, dollar = b.result()
        stats = b.stats()
    torch.cuda.empty_cache()
    nk = stats["n_keys"]
    assert nk == n - 32 * R and stats["n_special"] == 32 * R
    if case == "c3_at_limit":
        assert nk > (1 << 32) - (1 << 17)
        assert stats["sort_sweeps"] == 8
        assert binding.lib().debwt_dev_key_index_bits(ctypes.c_uint64(nk)) == 28
    else:
        assert 32 * R > 16384                               # the sentinel-window suffixes go through the bitonic network
    if case == "reads_past_2^31":
        assert 2048 * R > n                                 # the sort counts its digits from the keys, not the text

    # 2. base counts and separator rows
    raw = text.cpu().numpy().tobytes()
    tnp = np.frombuffer(raw, dtype=np.uint8)
    sym = _LUT[tnp]
    tcount = np.zeros(6, dtype=np.int64)
    for i in range(0, n, 1 << 28):
        tcount += np.bincount(sym[i:i + (1 << 28)], minlength=6)[:6]
    assert tcount[4] == R - 1 and tcount[5] == 1
    sharp = np.sort(sharp.astype(np.int64))
    dollar = int(dollar[0])
    assert sharp.size == R - 1 and np.unique(sharp).size == R - 1
    assert sharp[-1] < n and dollar < n and dollar not in set(sharp.tolist())
    if case == "records_past_2^31":
        assert (sharp > (1 << 31)).any()
    occ = host_occ(words, n, sharp, dollar)
    assert (occ[-1] == tcount[:4]).all(), f"BWT base counts {occ[-1]} != text base counts {tcount[:4]}"
    C = c_array(occ, n, R)

    words_dev = torch.from_numpy(words.view(np.int64)).to("cuda:0")
    with api.BwtBuilder(0) as c:
        c.set_result(words, n, sharp.astype(np.uint64), dollar)
        # 3. index tables
        docc, dC = c.index()
        assert (dC.astype(np.int64) == C).all(), f"C array {dC} != {C}"
        rows = docc.shape[0]
        assert rows == (n >> 5) + 1
        assert (docc.view(np.int64) == occ[:rows]).all(), "occ checkpoints differ from a host recount"
        del docc

        # 4. host LF walks from the '$' row and from separator rows
        lf = HostLF(words, occ, C, sharp, dollar)
        lf.walk(sym, dollar, 0, 100_000)
        del occ

        # 5. the library's verifiers, on the true text and on texts with one base changed
        bad, _ = c.verify(device_ptr=text.data_ptr(), n_symbols=n)
        peak()
        assert bad == 0
        for p in (1 << 16, (1 << 31) + 12345, n - (1 << 19)):
            while sym[p] > 3:
                p += 1
            old = int(text[p])
            text[p] = ord("A") if old != ord("A") else ord("C")
            try:
                bad, _ = c.verify(device_ptr=text.data_ptr(), n_symbols=n)
            finally:
                text[p] = old
            assert bad > 0, f"verify missed a changed base at {p}"
        steps = 5_000_000
        wbad, wc = api.verify_walk_device(words_dev.data_ptr(), n, sharp.astype(np.uint64), dollar,
                                          text[n - steps:].data_ptr(), steps)
        assert wbad == 0 and (wc.astype(np.int64) == C).all()
        del words_dev

        # 6. sampled SA
        c.sample_sa(32)
        peak()
        sep_rows = np.arange(n - R, n, dtype=np.uint64)
        sep_sa = c.sa(sep_rows).astype(np.int64)
        assert (np.sort(sep_sa) == seps.astype(np.int64)).all(), "SA of the separator rows is not the separator positions"
        assert int(sep_sa[-1]) == n - 1                     # '$' sorts last
        for i in sorted(set(rng.integers(0, R, 9).tolist()) | {R - 1}):
            r, p = lf.walk(sym, n - R + i, int(sep_sa[i]), 20_000)
            assert int(c.sa([r])[0]) == p
        probe = sa_probe_rows(n, sharp, rng)
        q, sa32 = check_sa_rows(c, words, sharp, dollar, sym, probe)

        # 7. count and locate
        hits, pos, pats = check_locate(c, raw, tnp, sym, seps, rng)

        if case == "c3_at_limit":                           # every row sampled: the same SA values and hits
            c.sample_sa(1)
            peak()
            assert (c.sa(q.astype(np.uint64)).astype(np.int64) == sa32).all()
            h1, p1 = c.locate(pats)
            assert (h1 == hits).all() and (p1.astype(np.int64) == pos).all()
    del text
    torch.cuda.empty_cache()
    _report(case, t0, peak, n_symbols=n, n_records=R, n_keys=nk, sort_sweeps=stats["sort_sweeps"], hits=int(hits[-1]),
            arena_gb=round(stats["arena_bytes"] / GB, 1), ms_build=round(stats["ms_total"], 1))
