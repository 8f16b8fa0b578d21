"""Host-side mirror of the reference's stage interface, on top of the C ABI.

The reference exposes the hot path as a chain of C stage functions driven by main()
(reference src/main.h:1-8, src/main.c:83-149).  `BwtBuilder` keeps that shape: set the FASTA
records (collect), build (mySort .. sortBlue), fetch the three outputs (insertCase3), and
`write_outputs` writes the reference's three files byte for byte (src/insertCase3.c:115-131).
Everything that computes runs in libdebwt_b200.so on the GPU.
"""
from __future__ import annotations

import ctypes
from typing import Sequence

import numpy as np

from . import binding
from .binding import DebwtError, ShardStats, Stats, c_p, c_u64, check, lib


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(c_p)


def join_records(records: Sequence) -> tuple[np.ndarray, np.ndarray]:
    """T = S1 # S2 # ... Sn $ as one ASCII byte array + separator offsets (src/collect#$.c:56-90)."""
    arrs = [np.frombuffer(r.encode() if isinstance(r, str) else bytes(r), dtype=np.uint8)
            if not isinstance(r, np.ndarray) else r.astype(np.uint8, copy=False) for r in records]
    if not arrs:
        raise DebwtError("no records")
    n = sum(a.size for a in arrs) + len(arrs)
    text = np.empty(n, dtype=np.uint8)
    seps = np.empty(len(arrs), dtype=np.uint64)
    pos = 0
    for i, a in enumerate(arrs):
        text[pos:pos + a.size] = a
        pos += a.size
        text[pos] = ord("#")
        seps[i] = pos
        pos += 1
    text[-1] = ord("$")
    return text, seps


class BwtBuilder:
    """One context == one GPU (replaces the reference's process-wide state)."""

    def __init__(self, device: int = 0, sort_config: int = 0, blue_grouping: int = 0):
        self._h = c_p()
        check(lib().debwt_create(ctypes.byref(self._h), device))
        if sort_config:
            lib().debwt_set_sort_config(self._h, sort_config)
        if blue_grouping:
            lib().debwt_set_blue_grouping(self._h, blue_grouping)
        self._keep = None

    def close(self):
        if self._h:
            lib().debwt_destroy(self._h)
            self._h = c_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_ambiguity_policy(self, resolve: bool, seed: int = 0):
        """IUPAC codes: reject (default) or resolve to a seeded pseudo-random compatible base (otherTool/transferN.c)"""
        check(lib().debwt_set_ambiguity_policy(self._h, int(bool(resolve)), seed))

    # -- input -------------------------------------------------------------------------------
    def set_records(self, records: Sequence):
        """Per-record host buffers (what a kseq loop yields)."""
        arrs = [np.ascontiguousarray(np.frombuffer(r.encode() if isinstance(r, str) else bytes(r), dtype=np.uint8)
                                     if not isinstance(r, np.ndarray) else r, dtype=np.uint8) for r in records]
        n = len(arrs)
        ptrs = (c_p * max(n, 1))(*[a.ctypes.data for a in arrs])
        lens = (c_u64 * max(n, 1))(*[a.size for a in arrs])
        self._keep = arrs
        check(lib().debwt_set_records(self._h, ptrs, lens, n))

    def set_text(self, text: np.ndarray, seps: np.ndarray):
        """One host buffer that already holds T (use pinned memory for the fastest H2D copy)."""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        seps = np.ascontiguousarray(seps, dtype=np.uint64)
        self._keep = (text, seps)
        check(lib().debwt_set_text(self._h, _ptr(text), text.size, _ptr(seps), seps.size))

    def set_text_ptr(self, host_ptr: int, n_symbols: int, seps: np.ndarray):
        seps = np.ascontiguousarray(seps, dtype=np.uint64)
        self._keep = seps
        check(lib().debwt_set_text(self._h, c_p(host_ptr), n_symbols, _ptr(seps), seps.size))

    def set_text_device(self, device_ptr: int, n_symbols: int, seps: np.ndarray):
        """T already resident in HBM (e.g. a torch.uint8 CUDA tensor's data_ptr())."""
        seps = np.ascontiguousarray(seps, dtype=np.uint64)
        self._keep = seps
        check(lib().debwt_set_text_device(self._h, c_p(device_ptr), n_symbols, _ptr(seps), seps.size))

    def ingest(self, chunks, seps: np.ndarray, n_hint: int = 0):
        """Streaming input (debwt_ingest_*): `chunks` yields consecutive pieces of T as bytes / uint8 arrays"""
        seps = np.ascontiguousarray(seps, dtype=np.uint64)
        check(lib().debwt_ingest_begin(self._h, n_hint))
        for ch in chunks:
            a = np.ascontiguousarray(np.frombuffer(ch, dtype=np.uint8) if not isinstance(ch, np.ndarray) else ch, dtype=np.uint8)
            if a.size:
                check(lib().debwt_ingest_append(self._h, _ptr(a), a.size))
        check(lib().debwt_ingest_end(self._h, _ptr(seps), seps.size))

    # -- build / output -------------------------------------------------------------------------
    def build(self, k: int = 32):
        check(lib().debwt_build(self._h, k))

    def result(self, out_words: np.ndarray | None = None):
        n, nw, ns = c_u64(), c_u64(), c_u64()
        check(lib().debwt_result_sizes(self._h, ctypes.byref(n), ctypes.byref(nw), ctypes.byref(ns)))
        words = out_words if out_words is not None else np.empty(nw.value, dtype=np.uint64)
        sharp = np.empty(ns.value, dtype=np.uint64)
        dollar = np.empty(1, dtype=np.uint64)
        check(lib().debwt_result_copy(self._h, _ptr(words), _ptr(sharp), _ptr(dollar)))
        return words, sharp, dollar

    def result_into(self, host_ptr: int):
        """Copy the packed BWT into caller-owned (e.g. pinned) host memory; returns (sharp, dollar)."""
        n, nw, ns = c_u64(), c_u64(), c_u64()
        check(lib().debwt_result_sizes(self._h, ctypes.byref(n), ctypes.byref(nw), ctypes.byref(ns)))
        sharp = np.empty(ns.value, dtype=np.uint64)
        dollar = np.empty(1, dtype=np.uint64)
        check(lib().debwt_result_copy(self._h, c_p(host_ptr), _ptr(sharp), _ptr(dollar)))
        return sharp, dollar

    # -- FM-index tables / verifier (reference "developer mode", src/insertCase3.c:139-208, src/LFsearch.c) ----
    def index(self):
        """(occ[(N>>5)+1][4], C[6]) in the reference's layout, built on the device"""
        check(lib().debwt_index_build(self._h))
        rows = c_u64()
        check(lib().debwt_index_sizes(self._h, ctypes.byref(rows)))
        occ = np.empty((rows.value, 4), dtype=np.uint64)
        carr = np.empty(6, dtype=np.uint64)
        check(lib().debwt_index_copy(self._h, _ptr(occ), _ptr(carr)))
        return occ, carr

    def count(self, patterns: Sequence) -> np.ndarray:
        """occurrences of each ACGT pattern in T, by backward search on the device"""
        check(lib().debwt_index_build(self._h))
        pats = [p.encode() if isinstance(p, str) else bytes(p) for p in patterns]
        offs = np.zeros(len(pats) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(p) for p in pats])
        blob = np.frombuffer(b"".join(pats) + b"\0", dtype=np.uint8)
        out = np.zeros(len(pats), dtype=np.uint64)
        check(lib().debwt_index_count(self._h, _ptr(blob), _ptr(offs), len(pats), _ptr(out)))
        return out

    def set_result(self, words: np.ndarray, n_symbols: int, sharp: np.ndarray, dollar):
        """Load a finished result (the reference's three outputs, e.g. from `read_outputs` or `build_multi`) in place of a
        build, to query it with count / sample_sa / sa / locate / extract / verify."""
        words = np.ascontiguousarray(words, dtype=np.uint64)
        sharp = np.ascontiguousarray(sharp, dtype=np.uint64)
        if words.size != (n_symbols + 31) // 32:
            raise DebwtError(f"set_result: {words.size} words for {n_symbols} symbols (expected {(n_symbols + 31) // 32})")
        dollar = int(np.asarray(dollar).reshape(-1)[0])
        check(lib().debwt_set_result(self._h, _ptr(words), n_symbols, _ptr(sharp), sharp.size, dollar))

    def sample_sa(self, rate: int = 32) -> float:
        """Sample the suffix array every `rate` text positions (power of two, 1..1024); returns the device ms."""
        ms = ctypes.c_float()
        check(lib().debwt_index_sample_sa(self._h, rate, ctypes.byref(ms)))
        return float(ms.value)

    def sa(self, rows) -> np.ndarray:
        """SA[r] (text position of the suffix in row r) for every row in `rows`; needs sample_sa"""
        rows = np.ascontiguousarray(rows, dtype=np.uint64)
        out = np.empty(rows.size, dtype=np.uint64)
        check(lib().debwt_index_sa(self._h, _ptr(rows), rows.size, _ptr(out)))
        return out

    def locate(self, patterns: Sequence) -> tuple[np.ndarray, np.ndarray]:
        """(hit_offsets u64[len + 1], positions u64[hits]): pattern i occurs at positions[hit_offsets[i]:hit_offsets[i+1]],
        in suffix-array order; needs sample_sa"""
        pats = [p.encode() if isinstance(p, str) else bytes(p) for p in patterns]
        offs = np.zeros(len(pats) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(p) for p in pats])
        blob = np.frombuffer(b"".join(pats) + b"\0", dtype=np.uint8)
        hits = np.zeros(len(pats) + 1, dtype=np.uint64)
        check(lib().debwt_index_locate(self._h, _ptr(blob), _ptr(offs), len(pats), _ptr(hits), c_p(0), 0))
        pos = np.empty(int(hits[-1]), dtype=np.uint64)
        if pos.size:
            check(lib().debwt_index_locate(self._h, _ptr(blob), _ptr(offs), len(pats), _ptr(hits), _ptr(pos), pos.size))
        return hits, pos

    def _sizes(self) -> tuple[int, int]:
        """(N, R) of the result"""
        n, nw, ns = c_u64(), c_u64(), c_u64()
        check(lib().debwt_result_sizes(self._h, ctypes.byref(n), ctypes.byref(nw), ctypes.byref(ns)))
        return int(n.value), int(ns.value) + 1

    def extract(self, starts, ends) -> tuple[np.ndarray, np.ndarray]:
        """(offsets u64[m + 1], symbols u8[total]): T[starts[i]:ends[i]] as ASCII (A, C, G, T upper case, '#', '$') is
        symbols[offsets[i]:offsets[i+1]], decoded from the index alone; needs sample_sa"""
        starts = np.ascontiguousarray(starts, dtype=np.uint64).reshape(-1)
        ends = np.ascontiguousarray(ends, dtype=np.uint64).reshape(-1)
        if starts.size != ends.size:
            raise DebwtError(f"extract: {starts.size} starts but {ends.size} ends")
        n, _ = self._sizes()
        # an interval the library will refuse counts 0 here, so that the buffer stays small and the call names it
        lens = np.where((starts <= ends) & (ends <= np.uint64(n)), ends - starts, np.uint64(0))
        offs = np.zeros(starts.size + 1, dtype=np.uint64)
        np.cumsum(lens, out=offs[1:])
        out = np.empty(int(offs[-1]), dtype=np.uint8)
        check(lib().debwt_index_extract(self._h, _ptr(starts), _ptr(ends), starts.size, _ptr(out), out.size))
        return offs, out

    def text(self) -> np.ndarray:
        """the whole text T (u8[N], ASCII) inverted from the index; needs sample_sa"""
        n, _ = self._sizes()
        return self.extract([0], [n])[1]

    def separators(self) -> np.ndarray:
        """the R separator positions of T ('#' ... '$', ascending; the `seps` of join_records) from the index alone: the
        rows [N - R, N) hold the suffixes that start with a separator; needs sample_sa"""
        n, r = self._sizes()
        return np.sort(self.sa(np.arange(n - r, n, dtype=np.uint64)))

    def smem(self, reads: Sequence, min_len: int = 19) -> tuple[np.ndarray, np.ndarray]:
        """(offsets u64[m + 1], smems SMEM_DTYPE[total]): the super-maximal exact matches of at least `min_len` bases of read
        i are smems[offsets[i]:offsets[i+1]], in ascending qbeg.  The text must hold both strands (`both_strands`); rows
        [row, row + count) are the suffixes that start with the match, for `sa`.  Builds the index tables if needed."""
        check(lib().debwt_index_build(self._h))
        rs = [r.encode() if isinstance(r, str) else bytes(r) for r in reads]
        offs = np.zeros(len(rs) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(r) for r in rs])
        blob = np.frombuffer(b"".join(rs) + b"\0", dtype=np.uint8)
        so = np.zeros(len(rs) + 1, dtype=np.uint64)
        check(lib().debwt_index_smem(self._h, _ptr(blob), _ptr(offs), len(rs), min_len, _ptr(so), c_p(0), 0))
        out = np.zeros(int(so[-1]), dtype=SMEM_DTYPE)
        if out.size:
            check(lib().debwt_index_smem(self._h, _ptr(blob), _ptr(offs), len(rs), min_len, _ptr(so), _ptr(out), out.size))
        return so, out

    def seeds(self, reads: Sequence, min_len: int = 19, split_factor: float = 1.5, split_width: int = 10, max_mem_intv: int = 20,
              max_occ: int = 500) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(offsets u64[m + 1], seeds SEED_DTYPE[total], hits HIT_DTYPE[all hits]): BWA-MEM's seeds of read i (bwa's -k, -r,
        split_width, -y, -c; SMEMs, re-seeded SMEMs and LAST-like seeds, `round` 1 / 2 / 3) are seeds[offsets[i]:offsets[i+1]],
        in ascending (qbeg, qend, round); seed s has hits[s.hit_begin : s.hit_begin + s.n_hits], at most max_occ evenly
        spaced rows of its interval, each with its text position, record, strand and forward offset (`strand_offsets`).
        The text must hold both strands (`both_strands`); needs sample_sa."""
        rs = [r.encode() if isinstance(r, str) else bytes(r) for r in reads]
        offs = np.zeros(len(rs) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(r) for r in rs])
        blob = np.frombuffer(b"".join(rs) + b"\0", dtype=np.uint8)
        for name, v in (("min_len", min_len), ("split_width", split_width), ("max_mem_intv", max_mem_intv), ("max_occ", max_occ)):
            if not 0 <= v < 1 << 32:
                raise DebwtError(f"seeds: {name} = {v} is not a 32-bit unsigned integer")
        opts = SeedOpts(min_len, split_width, max_mem_intv, max_occ, split_factor)
        so = np.zeros(len(rs) + 1, dtype=np.uint64)
        nh = c_u64()
        args = (self._h, _ptr(blob), _ptr(offs), len(rs), ctypes.addressof(opts), _ptr(so), ctypes.addressof(nh))
        check(lib().debwt_index_seeds(*args, c_p(0), 0, c_p(0), 0))
        seeds = np.zeros(int(so[-1]), dtype=SEED_DTYPE)
        hits = np.zeros(int(nh.value), dtype=HIT_DTYPE)
        if seeds.size:
            check(lib().debwt_index_seeds(*args, _ptr(seeds), seeds.size, _ptr(hits), hits.size))
        return so, seeds, hits

    def chains(self, reads: Sequence, min_len: int = 19, split_factor: float = 1.5, split_width: int = 10, max_mem_intv: int = 20,
               max_occ: int = 500, w: int = 100, max_chain_gap: int = 10000, min_chain_weight: int = 0, mask_level: float = 0.5,
               drop_ratio: float = 0.5, max_chain_extend: int = 1 << 30) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(offsets u64[m + 1], chains CHAIN_DTYPE[total], chain_seeds CHAIN_SEED_DTYPE[all chain seeds]): BWA-MEM's chains of
        read i (bwa's mem_chain and mem_chain_flt over the seeds of `seeds` with the same seed options; bwa's w,
        max_chain_gap, -W, mask_level, -D, max_chain_extend) are chains[offsets[i]:offsets[i+1]], in the filter's order;
        chain c has chain_seeds[c.seed_begin : c.seed_begin + c.n_seeds] in insertion order, in bwa's coordinate
        (`bwa_rbeg`).  The text must hold both strands (`both_strands`); needs sample_sa."""
        rs = [r.encode() if isinstance(r, str) else bytes(r) for r in reads]
        offs = np.zeros(len(rs) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(r) for r in rs])
        blob = np.frombuffer(b"".join(rs) + b"\0", dtype=np.uint8)
        for name, v in (("min_len", min_len), ("split_width", split_width), ("max_mem_intv", max_mem_intv), ("max_occ", max_occ)):
            if not 0 <= v < 1 << 32:
                raise DebwtError(f"chains: {name} = {v} is not a 32-bit unsigned integer")
        for name, v in (("w", w), ("max_chain_gap", max_chain_gap), ("min_chain_weight", min_chain_weight),
                        ("max_chain_extend", max_chain_extend)):
            if not -(1 << 31) <= v < 1 << 31:
                raise DebwtError(f"chains: {name} = {v} is not a 32-bit signed integer")
        so = SeedOpts(min_len, split_width, max_mem_intv, max_occ, split_factor)
        co = ChainOpts(w, max_chain_gap, min_chain_weight, max_chain_extend, mask_level, drop_ratio)
        co_offs = np.zeros(len(rs) + 1, dtype=np.uint64)
        ns = c_u64()
        args = (self._h, _ptr(blob), _ptr(offs), len(rs), ctypes.addressof(so), ctypes.addressof(co), _ptr(co_offs), ctypes.addressof(ns))
        check(lib().debwt_index_chains(*args, c_p(0), 0, c_p(0), 0))
        chains = np.zeros(int(co_offs[-1]), dtype=CHAIN_DTYPE)
        seeds = np.zeros(int(ns.value), dtype=CHAIN_SEED_DTYPE)
        if chains.size:
            check(lib().debwt_index_chains(*args, _ptr(chains), chains.size, _ptr(seeds), seeds.size))
        return co_offs, chains, seeds

    def regions(self, reads: Sequence, min_len: int = 19, split_factor: float = 1.5, split_width: int = 10, max_mem_intv: int = 20,
                max_occ: int = 500, w: int = 100, max_chain_gap: int = 10000, min_chain_weight: int = 0, mask_level: float = 0.5,
                drop_ratio: float = 0.5, max_chain_extend: int = 1 << 30, a: int = 1, b: int = 4, o_del: int = 6, e_del: int = 1,
                o_ins: int = 6, e_ins: int = 1, pen_clip5: int = 5, pen_clip3: int = 5, zdrop: int = 100) -> tuple[np.ndarray, np.ndarray]:
        """(offsets u64[m + 1], regions REGION_DTYPE[total]): BWA-MEM's alignment regions of read i (bwa's
        mem_flt_chained_seeds and mem_chain2aln over the chains of `chains` with the same seed and chain options; w is
        also the band; bwa's -A, -B, -O, -E, -L and -d) are regions[offsets[i]:offsets[i+1]], chain by chain in the
        order of extension, in bwa's coordinate.  One device pass per call: the regions land in a buffer the builder
        keeps, and only a batch with more regions than it holds runs a second time.  Needs sample_sa."""
        rs = [r.encode() if isinstance(r, str) else bytes(r) for r in reads]
        offs = np.zeros(len(rs) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(r) for r in rs])
        blob = np.frombuffer(b"".join(rs) + b"\0", dtype=np.uint8)
        for name, v in (("min_len", min_len), ("split_width", split_width), ("max_mem_intv", max_mem_intv), ("max_occ", max_occ)):
            if not 0 <= v < 1 << 32:
                raise DebwtError(f"regions: {name} = {v} is not a 32-bit unsigned integer")
        ints = dict(w=w, max_chain_gap=max_chain_gap, min_chain_weight=min_chain_weight, max_chain_extend=max_chain_extend, a=a, b=b,
                    o_del=o_del, e_del=e_del, o_ins=o_ins, e_ins=e_ins, pen_clip5=pen_clip5, pen_clip3=pen_clip3, zdrop=zdrop)
        for name, v in ints.items():
            if not -(1 << 31) <= v < 1 << 31:
                raise DebwtError(f"regions: {name} = {v} is not a 32-bit signed integer")
        so = SeedOpts(min_len, split_width, max_mem_intv, max_occ, split_factor)
        co = ChainOpts(w, max_chain_gap, min_chain_weight, max_chain_extend, mask_level, drop_ratio)
        eo = ExtOpts(a, b, o_del, e_del, o_ins, e_ins, pen_clip5, pen_clip3, zdrop)
        r_offs = np.zeros(len(rs) + 1, dtype=np.uint64)
        args = (self._h, _ptr(blob), _ptr(offs), len(rs), ctypes.addressof(so), ctypes.addressof(co), ctypes.addressof(eo), _ptr(r_offs))
        buf = getattr(self, "_regions_buf", None)
        if buf is None:
            buf = self._regions_buf = np.zeros(1 << 16, dtype=REGION_DTYPE)
        rc = lib().debwt_index_regions(*args, _ptr(buf), buf.size)
        if rc != 0 and int(r_offs[-1]) > buf.size:                    # too small: grow once, run again
            buf = self._regions_buf = np.zeros(int(r_offs[-1]) * 5 // 4, dtype=REGION_DTYPE)
            rc = lib().debwt_index_regions(*args, _ptr(buf), buf.size)
        check(rc)
        return r_offs, buf[:int(r_offs[-1])].copy()

    def verify(self, text=None, device_ptr: int | None = None, n_symbols: int | None = None):
        """LF-inversion check of the last build against T; returns (bad rows, device ms).  0 bad rows <=> BWT(T)."""
        bad, ms = c_u64(), ctypes.c_float()
        if device_ptr is not None:
            check(lib().debwt_verify_text_device(self._h, c_p(device_ptr), n_symbols, ctypes.byref(bad), ctypes.byref(ms)))
        else:
            text = np.ascontiguousarray(text, dtype=np.uint8)
            check(lib().debwt_verify_text(self._h, _ptr(text), text.size, ctypes.byref(bad), ctypes.byref(ms)))
        return int(bad.value), float(ms.value)

    def stats(self) -> dict:
        s = Stats()
        check(lib().debwt_get_stats(self._h, ctypes.byref(s)))
        return s.as_dict()


def build_bwt(records: Sequence, device: int = 0, k: int = 32):
    """FASTA records in, (bwt_words, sharp_rows, dollar_row) out -- the whole hot path."""
    with BwtBuilder(device) as b:
        b.set_records(records)
        b.build(k)
        return b.result()


def write_outputs(path: str, words: np.ndarray, sharp: np.ndarray, dollar: np.ndarray):
    """The reference's three output files (src/insertCase3.c:115-131)."""
    words.astype("<u8", copy=False).tofile(path)
    sharp.astype("<u8", copy=False).tofile(path + ".#")
    dollar.astype("<u8", copy=False).tofile(path + ".$")


def read_outputs(path: str, n_symbols: int):
    """The inverse of `write_outputs`: (words, sharp, dollar) from the three files.  The files do not hold N, so the
    caller passes it; the word file must hold exactly ceil(N / 32) words."""
    words = np.fromfile(path, dtype="<u8").astype(np.uint64, copy=False)
    if words.size != (n_symbols + 31) // 32:
        raise DebwtError(f"{path}: {words.size} words, but {n_symbols} symbols need {(n_symbols + 31) // 32}")
    sharp = np.fromfile(path + ".#", dtype="<u8").astype(np.uint64, copy=False)
    dollar = np.fromfile(path + ".$", dtype="<u8").astype(np.uint64, copy=False)
    if dollar.size != 1:
        raise DebwtError(f"{path}.$: {dollar.size} values, expected 1")
    return words, sharp, dollar


def record_offsets(positions, seps) -> tuple[np.ndarray, np.ndarray]:
    """Text positions in T = S1 # S2 # ... Sn $ to (record index, offset in that record).  `seps` are the separator
    positions (join_records); a separator maps to its record with offset = the record's length."""
    pos = np.asarray(positions, dtype=np.uint64)
    seps = np.asarray(seps, dtype=np.uint64)
    if pos.size and int(pos.max()) > int(seps[-1]):
        raise ValueError(f"position {int(pos.max())} is beyond the text ({int(seps[-1]) + 1} symbols)")
    rec = np.searchsorted(seps, pos, side="left")
    starts = np.concatenate(([0], seps[:-1] + 1)).astype(np.uint64)
    return rec.astype(np.int64), pos - starts[rec]


# ---- SMEM seeding over both strands (debwt_index_smem) ---------------------------------------------------------------
SMEM_DTYPE = np.dtype([("row", np.uint64), ("rc_row", np.uint64), ("count", np.uint64), ("qbeg", np.uint32), ("qend", np.uint32)],
                      align=True)                      # debwt_smem of include/debwt_b200.h

# ---- BWA-MEM seed collection over both strands (debwt_index_seeds) ---------------------------------------------------
SEED_DTYPE = np.dtype([("row", np.uint64), ("rc_row", np.uint64), ("count", np.uint64), ("qbeg", np.uint32), ("qend", np.uint32),
                       ("hit_begin", np.uint64), ("n_hits", np.uint32), ("round", np.uint32)], align=True)    # debwt_seed
HIT_DTYPE = np.dtype([("pos", np.uint64), ("offset", np.uint64), ("record", np.uint32), ("strand", np.uint32)], align=True)  # debwt_seed_hit


class SeedOpts(ctypes.Structure):
    """debwt_seed_opts of include/debwt_b200.h"""
    _fields_ = [("min_seed_len", ctypes.c_uint32), ("split_width", ctypes.c_uint32), ("max_mem_intv", ctypes.c_uint32),
                ("max_occ", ctypes.c_uint32), ("split_factor", ctypes.c_float)]


# ---- BWA-MEM seed chaining over both strands (debwt_index_chains) ----------------------------------------------------
CHAIN_DTYPE = np.dtype([("pos", np.uint64), ("seed_begin", np.uint64), ("n_seeds", np.uint32), ("weight", np.uint32),
                        ("record", np.uint32), ("strand", np.uint32), ("kept", np.uint32), ("frac_rep", np.float32)],
                       align=True)                     # debwt_chain
CHAIN_SEED_DTYPE = np.dtype([("rbeg", np.uint64), ("qbeg", np.uint32), ("len", np.uint32)], align=True)  # debwt_chain_seed


class ChainOpts(ctypes.Structure):
    """debwt_chain_opts of include/debwt_b200.h"""
    _fields_ = [("w", ctypes.c_int32), ("max_chain_gap", ctypes.c_int32), ("min_chain_weight", ctypes.c_int32),
                ("max_chain_extend", ctypes.c_int32), ("mask_level", ctypes.c_float), ("drop_ratio", ctypes.c_float)]


# ---- BWA-MEM seed extension over both strands (debwt_index_regions) --------------------------------------------------
REGION_DTYPE = np.dtype([("rb", np.uint64), ("re", np.uint64), ("qb", np.uint32), ("qe", np.uint32), ("score", np.int32),
                         ("truesc", np.int32), ("w", np.uint32), ("seedcov", np.uint32), ("seedlen0", np.uint32), ("chain", np.uint32),
                         ("record", np.uint32), ("strand", np.uint32), ("frac_rep", np.float32), ("pad_", np.uint32)],
                        align=True)                    # debwt_region


class ExtOpts(ctypes.Structure):
    """debwt_ext_opts of include/debwt_b200.h"""
    _fields_ = [(n, ctypes.c_int32) for n in ("a", "b", "o_del", "e_del", "o_ins", "e_ins", "pen_clip5", "pen_clip3", "zdrop")]


_COMP = bytes.maketrans(b"ACGT", b"TGCA")


def both_strands(records: Sequence) -> list[bytes]:
    """records + their reverse complements, upper case, in that order: a text closed under reverse complement, which SMEM
    search needs (Li 2012's FMD-index).  Only A, C, G, T (either case) are accepted; ambiguity codes resolved at random
    per position would break the closure."""
    fwd = []
    for i, r in enumerate(records):
        b = (r.encode() if isinstance(r, str) else bytes(np.asarray(r, dtype=np.uint8)) if isinstance(r, np.ndarray) else bytes(r)).upper()
        bad = b.translate(None, b"ACGT")
        if bad:
            raise DebwtError(f"both_strands: record {i} holds {bad[:1]!r}; only A, C, G and T have a reverse complement here")
        fwd.append(b)
    return fwd + [b.translate(_COMP)[::-1] for b in fwd]


def strand_offsets(positions, length: int, seps) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Hits of `length` symbols at text positions of a `both_strands` text (separators `seps`, 2 R records) to (record in
    0..R-1, strand 0 forward / 1 reverse, offset of the hit's first base on the forward strand).  A hit at offset o of the
    reverse copy of record i covers forward bases [len_i - o - length, len_i - o)."""
    seps = np.asarray(seps, dtype=np.uint64)
    if seps.size % 2:
        raise ValueError(f"{seps.size} records: a both_strands text has an even number")
    rec, off = record_offsets(positions, seps)
    off = off.astype(np.int64)
    R = seps.size // 2
    lens = (seps - np.concatenate(([0], seps[:-1] + 1)).astype(np.uint64)).astype(np.int64)
    if rec.size and (off + length > lens[rec]).any():
        raise ValueError(f"a hit of {length} symbols runs past the end of its record")
    rev = rec >= R
    return rec % R, rev.astype(np.int8), np.where(rev, lens[rec] - off - length, off)


def bwa_rbeg(record, strand, offset, length, seps) -> np.ndarray:
    """bwa's forward-reverse coordinate (int64) of hits of `length` bases at (record, strand, forward offset) of a
    `both_strands` text with separators `seps`: with l_pac = (N - R) / 2 forward bases and F[r] the bases of the forward
    records before r, F[r] + offset on strand 0 (the text position - r), 2 l_pac - (F[r] + offset + length) on strand 1."""
    seps = np.asarray(seps, dtype=np.int64)
    if seps.size % 2:
        raise ValueError(f"{seps.size} records: a both_strands text has an even number")
    R = seps.size
    l_pac = (int(seps[-1]) + 1 - R) // 2
    F = np.concatenate(([0], seps[:R // 2 - 1] + 1 - np.arange(1, R // 2))).astype(np.int64)
    rec = np.asarray(record, dtype=np.int64)
    f = F[rec] + np.asarray(offset, dtype=np.int64)
    return np.where(np.asarray(strand) != 0, 2 * l_pac - (f + np.asarray(length, dtype=np.int64)), f)


# ---- per-kernel entry points (parity tests) -------------------------------------------------------
def k_pack(text: np.ndarray, device: int = 0) -> np.ndarray:
    text = np.ascontiguousarray(text, dtype=np.uint8)
    out = np.empty((text.size + 32 + 31) // 32, dtype=np.uint64)
    check(lib().debwt_k_pack(device, _ptr(text), text.size, _ptr(out)))
    return out


def k_extract(text: np.ndarray, seps: np.ndarray, device: int = 0) -> np.ndarray:
    text = np.ascontiguousarray(text, dtype=np.uint8)
    seps = np.ascontiguousarray(seps, dtype=np.uint64)
    out = np.empty(text.size - 32 * seps.size, dtype=np.uint64)
    check(lib().debwt_k_extract(device, _ptr(text), text.size, _ptr(seps), seps.size, _ptr(out)))
    return out


def k_radix_sort(keys: np.ndarray, device: int = 0, cfg: int = 0):
    k = np.ascontiguousarray(keys, dtype=np.uint64).copy()
    ms = ctypes.c_float()
    check(lib().debwt_k_radix_sort_u64(device, _ptr(k), k.size, cfg, ctypes.byref(ms)))
    return k, ms.value


def k_rle(sorted_keys: np.ndarray, device: int = 0):
    s = np.ascontiguousarray(sorted_keys, dtype=np.uint64)
    km = np.empty(s.size, dtype=np.uint64)
    ct = np.empty(s.size, dtype=np.uint64)
    d = c_u64()
    check(lib().debwt_k_rle(device, _ptr(s), s.size, _ptr(km), _ptr(ct), ctypes.byref(d)))
    return km[:d.value].copy(), ct[:d.value].copy()


def k_group_masks(text: np.ndarray, seps: np.ndarray, device: int = 0) -> np.ndarray:
    text = np.ascontiguousarray(text, dtype=np.uint8)
    seps = np.ascontiguousarray(seps, dtype=np.uint64)
    out = np.empty(text.size - 32 * seps.size, dtype=np.uint16)
    check(lib().debwt_k_group_masks(device, _ptr(text), text.size, _ptr(seps), seps.size, _ptr(out)))
    return out


def k_branch_kmers(text: np.ndarray, seps: np.ndarray, device: int = 0):
    """K7: the branch table, (entries u64[B] = k-mer << 2 | multi_in << 1 | multi_out ascending, group head key index u64[B])"""
    text = np.ascontiguousarray(text, dtype=np.uint8)
    seps = np.ascontiguousarray(seps, dtype=np.uint64)
    cap = max(text.size - 32 * seps.size, 1)
    kmer, head = np.empty(cap, dtype=np.uint64), np.empty(cap, dtype=np.uint64)
    nb = c_u64()
    check(lib().debwt_k_branch_kmers(device, _ptr(text), text.size, _ptr(seps), seps.size, _ptr(kmer), _ptr(head), cap, ctypes.byref(nb)))
    return kmer[:nb.value].copy(), head[:nb.value].copy()


def bench_sort(n: int, device: int = 0, cfg: int = 0, iters: int = 5) -> float:
    ms = ctypes.c_float()
    check(lib().debwt_bench_sort(device, n, cfg, iters, ctypes.byref(ms)))
    return ms.value


def bench_sort_passes(n: int, device: int = 0, cfg: int = 0, iters: int = 5):
    """(mean ms per whole sort, mean ms per digit pass) on `n` device-generated pseudo-random keys"""
    ms, msp = ctypes.c_float(), ctypes.c_float()
    check(lib().debwt_bench_sort_passes(device, n, cfg, iters, ctypes.byref(ms), ctypes.byref(msp)))
    return ms.value, msp.value


def verify_bwt_device(bwt_ptr: int, n_symbols: int, sharp_rows: np.ndarray, dollar_row: int, text_ptr: int, device: int = 0):
    """LF-inversion check of a packed BWT in device memory against the ASCII text in device memory: (bad rows, ms)"""
    sharp = np.ascontiguousarray(sharp_rows, dtype=np.uint64)
    bad, ms = c_u64(), ctypes.c_float()
    check(lib().debwt_verify_bwt_device(device, c_p(bwt_ptr), n_symbols, _ptr(sharp), sharp.size, int(dollar_row), c_p(text_ptr),
                                        ctypes.byref(bad), ctypes.byref(ms)))
    return int(bad.value), float(ms.value)


def k_codes(text: np.ndarray, seps: np.ndarray, device: int = 0):
    """K9: (codes u8[S], blue entries as (group head key index u64[M], spIndex u64[M], prev u8[M]))"""
    text = np.ascontiguousarray(text, dtype=np.uint8)
    seps = np.ascontiguousarray(seps, dtype=np.uint64)
    cap = text.size + 64
    codes = np.empty(cap, dtype=np.uint8)
    head, spi, prev = np.empty(cap, dtype=np.uint64), np.empty(cap, dtype=np.uint64), np.empty(cap, dtype=np.uint8)
    nc, nb = c_u64(), c_u64()
    check(lib().debwt_k_codes(device, _ptr(text), text.size, _ptr(seps), seps.size, _ptr(codes), cap, ctypes.byref(nc), _ptr(head),
                              _ptr(spi), _ptr(prev), cap, ctypes.byref(nb)))
    return codes[:nc.value].copy(), head[:nb.value].copy(), spi[:nb.value].copy(), prev[:nb.value].copy()


def k_sort_blue(codes: np.ndarray, seg_offsets: np.ndarray, spindex: np.ndarray, prev: np.ndarray, device: int = 0):
    """K10 alone: returns (spindex, prev) with every segment ordered by its code strings"""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    offs = np.ascontiguousarray(seg_offsets, dtype=np.uint64)
    spi = np.ascontiguousarray(spindex, dtype=np.uint64).copy()
    prv = np.ascontiguousarray(prev, dtype=np.uint8).copy()
    check(lib().debwt_k_sort_blue(device, _ptr(codes), codes.size, _ptr(offs), offs.size - 1, _ptr(spi), _ptr(prv)))
    return spi, prv


def verify_walk_device(bwt_ptr: int, n_symbols: int, sharp_rows: np.ndarray, dollar_row: int, tail_ptr: int, steps: int, device: int = 0):
    """sequential LF walk of `steps` rows from the '$' row against the last `steps` symbols of T (device pointers);
    returns (mismatches, C-array).  For texts beyond the list-ranking verifier's 2^32 symbols."""
    sharp = np.ascontiguousarray(sharp_rows, dtype=np.uint64)
    bad = c_u64()
    carr = np.zeros(6, dtype=np.uint64)
    check(lib().debwt_verify_walk_device(device, c_p(bwt_ptr), n_symbols, _ptr(sharp), sharp.size, int(dollar_row), c_p(tail_ptr), steps,
                                         ctypes.byref(bad), _ptr(carr)))
    return int(bad.value), carr


# ---- multi-GPU: the sharded build behind the C ABI (csrc/shard.cu) ---------------------------------------------------
class Shard:
    """One rank of the sharded build (one per GPU; a process under torchrun, or a thread)."""

    def __init__(self, device: int, rank: int, world: int, group_tag: str, same_process: bool = False, sort_config: int = 0):
        self._h = c_p()
        self.rank, self.world, self.device = rank, world, device
        check(lib().debwt_shard_create(ctypes.byref(self._h), device, rank, world, group_tag.encode(), int(same_process)))
        if sort_config:
            lib().debwt_shard_set_sort_config(self._h, sort_config)

    def close(self):
        if self._h:
            lib().debwt_shard_destroy(self._h)
            self._h = c_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def slice(self, n_symbols: int):
        lo, hi = c_u64(), c_u64()
        check(lib().debwt_shard_slice(self.rank, self.world, n_symbols, ctypes.byref(lo), ctypes.byref(hi)))
        return int(lo.value), int(hi.value)

    def build(self, slice_ptr: int, on_device: bool, n_symbols: int, seps: np.ndarray):
        seps = np.ascontiguousarray(seps, dtype=np.uint64)
        check(lib().debwt_shard_build(self._h, c_p(slice_ptr), int(on_device), n_symbols, _ptr(seps), seps.size))
        self._n, self._r = n_symbols, int(seps.size)

    def build_host(self, text: np.ndarray, seps: np.ndarray):
        """every rank passes the whole T; only its slice is read"""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        lo, hi = self.slice(text.size)
        sl = np.ascontiguousarray(text[lo:hi]) if hi > lo else np.zeros(1, np.uint8)
        self.build(sl.ctypes.data, False, text.size, seps)

    def result(self):
        """(words, sharp, dollar) on rank 0, None elsewhere"""
        if self.rank != 0:
            check(lib().debwt_shard_result_copy(self._h, c_p(0), c_p(0), c_p(0)))
            return None
        words = np.empty((self._n + 31) // 32, dtype=np.uint64)
        sharp = np.empty(max(self._r - 1, 0), dtype=np.uint64)
        dollar = np.empty(1, dtype=np.uint64)
        check(lib().debwt_shard_result_copy(self._h, _ptr(words), _ptr(sharp), _ptr(dollar)))
        return words, sharp, dollar

    def result_device_ptr(self) -> int:
        p, nw = c_p(), c_u64()
        check(lib().debwt_shard_result_device(self._h, ctypes.byref(p), ctypes.byref(nw)))
        return p.value or 0

    def result_into(self, host_ptr: int):
        sharp = np.empty(max(self._r - 1, 0), dtype=np.uint64)
        dollar = np.empty(1, dtype=np.uint64)
        check(lib().debwt_shard_result_copy(self._h, c_p(host_ptr), _ptr(sharp), _ptr(dollar)))
        return sharp, dollar

    def stats(self) -> dict:
        s = ShardStats()
        check(lib().debwt_shard_get_stats(self._h, ctypes.byref(s)))
        return s.as_dict()


def build_multi(text: np.ndarray, seps: np.ndarray, devices: Sequence[int]):
    """one process, one thread per GPU (debwt_build_multi): (words, sharp, dollar, stats of rank 0)"""
    text = np.ascontiguousarray(text, dtype=np.uint8)
    seps = np.ascontiguousarray(seps, dtype=np.uint64)
    devs = (ctypes.c_int * len(devices))(*devices)
    words = np.empty((text.size + 31) // 32, dtype=np.uint64)
    sharp = np.empty(seps.size - 1, dtype=np.uint64)
    dollar = np.empty(1, dtype=np.uint64)
    st = ShardStats()
    check(lib().debwt_build_multi(devs, len(devices), _ptr(text), text.size, _ptr(seps), seps.size, _ptr(words), _ptr(sharp), _ptr(dollar),
                                  ctypes.byref(st)))
    return words, sharp, dollar, st.as_dict()
