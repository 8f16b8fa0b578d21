"""Sharded (multi-GPU) BWT build: one process per GPU, torch.distributed for the plumbing.

SURVEY.md section 8e / K12.  The reference has no distributed code; this is the B200 design:

  1. the text is split by position into G 32-aligned slices; every rank packs its slice and the packed
     text (N/4 bytes in total) is all-gathered;
  2. every rank extracts the 64-bit keys of its slice; G-1 splitters are chosen from an all-gathered
     sample, rounded to k-mer boundaries so that a k-mer is never split between two ranks;
  3. ONE all-to-all moves every key to its owner; each rank then owns a contiguous key range, i.e. a
     contiguous run of BWT rows, and sorts / classifies it locally.  In-edges cX -> X that cross a range
     boundary travel as a second, smaller all-to-all of queries;
  4. branch tables are all-gathered (small), branch codes are produced per position slice at global
     code indices and summed (disjoint bits), blue entries travel to the owner of their k-mer in a third
     all-to-all, and every rank emits its own BWT rows; the segments are summed onto rank 0.

The orchestration is written against two small interfaces so that it also runs on CPU tensors:
  * `Comm`  -- the collectives (torch.distributed, NCCL on CUDA tensors, gloo staged through host memory);
  * `ops`   -- the stage kernels: `CudaOps` (libdebwt_b200.so, include/debwt_b200_dev.h) in production;
               tests/numpy_ops.py restates them in numpy for the world_size-2 gloo tests.
All u64 payloads live in torch.int64 tensors (bit containers).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import binding

SAMPLES_PER_RANK = 4096
I64_ALL_ONES = -1


# --------------------------------------------------------------------------------------------------
# collectives
# --------------------------------------------------------------------------------------------------
class Comm:
    """torch.distributed wrapper; `staged=True` moves device tensors through host memory so that a
    gloo group can drive CUDA ranks (used by the single-GPU two-process test)."""

    def __init__(self, group=None, staged: bool | None = None):
        import torch.distributed as dist
        self.dist = dist if dist.is_available() and dist.is_initialized() else None
        self.group = group
        self.rank = self.dist.get_rank(group) if self.dist else 0
        self.size = self.dist.get_world_size(group) if self.dist else 1
        if staged is None:
            staged = bool(self.dist) and self.dist.get_backend(group) == "gloo"
        self.staged = staged
        self.bytes_sent = 0
        gloo = bool(self.dist) and self.dist.get_backend(group) == "gloo"
        self.coll_device = torch.device("cpu") if (gloo or not torch.cuda.is_available()) else torch.device("cuda", torch.cuda.current_device())

    def to_coll(self, t: torch.Tensor) -> torch.Tensor:
        """a tensor the backend can run a collective on"""
        return t.to(self.coll_device)

    def _h(self, t):
        return t.cpu() if (self.staged and t.is_cuda) else t

    def all_gather_equal(self, t: torch.Tensor) -> torch.Tensor:
        """concatenation of every rank's `t` (same length everywhere)"""
        if self.size == 1:
            return t.clone()
        src = self._h(t.contiguous())
        out = torch.empty(self.size * src.numel(), dtype=src.dtype, device=src.device)
        self.dist.all_gather_into_tensor(out, src, group=self.group)
        self.bytes_sent += src.numel() * src.element_size() * (self.size - 1)
        return out.to(t.device)

    def all_gather_scalar(self, v: int) -> list[int]:
        if self.size == 1:
            return [int(v)]
        out = self.all_gather_equal(self.to_coll(torch.tensor([int(v)], dtype=torch.int64)))
        return [int(x) for x in out.cpu().tolist()]

    def all_gather_var(self, t: torch.Tensor):
        """concatenation of variable-length tensors + the per-rank lengths"""
        lens = self.all_gather_scalar(t.numel())
        if self.size == 1:
            return t.clone(), lens
        mx = max(max(lens), 1)
        pad = torch.zeros(mx, dtype=t.dtype, device=t.device)
        pad[:t.numel()] = t
        allp = self.all_gather_equal(pad)
        return torch.cat([allp[i * mx:i * mx + lens[i]] for i in range(self.size)]), lens

    def all_reduce_sum(self, t: torch.Tensor) -> torch.Tensor:
        if self.size == 1:
            return t
        h = self._h(t)
        self.dist.all_reduce(h, op=self.dist.ReduceOp.SUM, group=self.group)
        self.bytes_sent += h.numel() * h.element_size()
        if h is not t:
            t.copy_(h)
        return t

    def all_reduce_max(self, t: torch.Tensor) -> torch.Tensor:
        if self.size == 1:
            return t
        h = self._h(t)
        self.dist.all_reduce(h, op=self.dist.ReduceOp.MAX, group=self.group)
        if h is not t:
            t.copy_(h)
        return t

    def reduce_sum_to0(self, t: torch.Tensor) -> torch.Tensor:
        if self.size == 1:
            return t
        h = self._h(t)
        self.dist.reduce(h, dst=0, op=self.dist.ReduceOp.SUM, group=self.group)
        self.bytes_sent += h.numel() * h.element_size()
        if h is not t:
            t.copy_(h)
        return t

    def gather_to0(self, t: torch.Tensor):
        """rank 0 gets the list of every rank's `t` (same length everywhere); others get None"""
        if self.size == 1:
            return [t]
        src = self._h(t.contiguous())
        outs = [torch.empty_like(src) for _ in range(self.size)] if self.rank == 0 else None
        self.dist.gather(src, outs, dst=0, group=self.group)
        if self.rank != 0:
            self.bytes_sent += src.numel() * src.element_size()
            return None
        return [o.to(t.device) for o in outs]

    def all_to_all_v(self, t: torch.Tensor, send_counts) -> tuple[torch.Tensor, list[int]]:
        """`t` is grouped by destination rank with `send_counts[r]` items for rank r"""
        send_counts = [int(c) for c in send_counts]
        if self.size == 1:
            return t[:send_counts[0]].clone(), send_counts
        sc = torch.tensor(send_counts, dtype=torch.int64)
        dev = t.device if not self.staged else torch.device("cpu")
        sc_d = sc.to(dev)
        rc_d = torch.empty_like(sc_d)
        self.dist.all_to_all_single(rc_d, sc_d, group=self.group)
        recv_counts = [int(x) for x in rc_d.cpu().tolist()]
        src = self._h(t[:sum(send_counts)].contiguous())
        out = torch.empty(sum(recv_counts), dtype=src.dtype, device=src.device)
        self.dist.all_to_all_single(out, src, output_split_sizes=recv_counts, input_split_sizes=send_counts, group=self.group)
        self.bytes_sent += (sum(send_counts) - send_counts[self.rank]) * src.element_size()
        return out.to(t.device), recv_counts

    def barrier(self):
        if self.size > 1:
            self.dist.barrier(group=self.group)


# --------------------------------------------------------------------------------------------------
# CUDA ops: torch tensors -> include/debwt_b200_dev.h
# --------------------------------------------------------------------------------------------------
_DEV_SIGS_DONE = False


def _dev_lib():
    global _DEV_SIGS_DONE
    L = binding.lib()
    if not _DEV_SIGS_DONE:
        for name in dir(L):
            pass
        # every debwt_dev_* function returns int; arguments are passed explicitly typed below
        _DEV_SIGS_DONE = True
    return L


def _p(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def _u64(v):
    return ctypes.c_uint64(int(v))


class CudaOps:
    """Stage kernels of libdebwt_b200.so on torch CUDA tensors (current device, current stream)."""

    def __init__(self, device: int, sort_cfg: int = 8):
        self.device = torch.device("cuda", device)
        self.L = _dev_lib()
        self.sort_cfg = sort_cfg
        self.launches = 0
        binding.check(self.L.debwt_dev_init(device))

    # -- helpers --
    def _st(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _ck(self, rc):
        binding.check(rc)
        self.launches += 1

    def _bytes(self, fn, *args):
        f = getattr(self.L, fn)
        f.restype = ctypes.c_uint64
        return int(f(*args))

    def empty(self, n, dtype=torch.int64):
        return torch.empty(max(int(n), 0), dtype=dtype, device=self.device)

    def zeros(self, n, dtype=torch.int64):
        return torch.zeros(max(int(n), 0), dtype=dtype, device=self.device)

    def from_numpy(self, a):
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        return torch.from_numpy(np.ascontiguousarray(a)).to(self.device)

    # -- stages --
    def pack(self, ascii_slice, n_valid, words_out, nwords, err):
        self._ck(self.L.debwt_dev_pack(_p(ascii_slice), _u64(n_valid), _p(words_out), _u64(nwords), _p(err), self._st()))

    def extract(self, words, pos_lo, pos_hi, seps, n_rec, idx_base, keys_out, n_symbols):
        self._ck(self.L.debwt_dev_extract_slice(_p(words), _u64(n_symbols), _u64(pos_lo), _u64(pos_hi), _p(seps), _u64(n_rec),
                                                _u64(idx_base), _p(keys_out), self._st()))

    def sort(self, keys, timed: bool = False):
        n = keys.numel()
        if n <= 1:
            return keys
        tmp = torch.empty_like(keys)
        ws = self.empty(self._bytes("debwt_dev_sort_workspace_bytes", _u64(n), self.sort_cfg), torch.uint8)
        in_b = ctypes.c_int(0)
        if timed:
            ms, msw, nsw = ctypes.c_float(), ctypes.c_float(), ctypes.c_int()
            self._ck(self.L.debwt_dev_sort_timed(_p(keys), _p(tmp), _u64(n), self.sort_cfg, _p(ws), ctypes.byref(in_b),
                                                 ctypes.byref(ms), ctypes.byref(msw), ctypes.byref(nsw), self._st()))
            self.sort_stats = {"n": n, "ms": ms.value, "ms_sweeps": msw.value, "sweeps": nsw.value}
        else:
            self._ck(self.L.debwt_dev_sort(_p(keys), _p(tmp), _u64(n), self.sort_cfg, _p(ws), ctypes.byref(in_b), self._st()))
        return tmp if in_b.value else keys

    def owner_of_keys(self, items, splitters, mask, drop_marker):
        dest = self.empty(items.numel(), torch.uint8)
        self._ck(self.L.debwt_dev_owner_of_keys(_p(items), _u64(items.numel()), _p(splitters), ctypes.c_uint32(splitters.numel()),
                                                _u64(mask), int(bool(drop_marker)), _p(dest), self._st()))
        return dest

    def owner_of_index(self, idx, bases, n_ranks):
        dest = self.empty(idx.numel(), torch.uint8)
        self._ck(self.L.debwt_dev_owner_of_index(_p(idx), _u64(idx.numel()), _p(bases), ctypes.c_uint32(n_ranks), _p(dest),
                                                 self._st()))
        return dest

    def partition(self, a, b, dest, n_ranks):
        n = a.numel()
        out_a = torch.empty_like(a)
        out_b = torch.empty_like(b) if b is not None else None
        counts = (ctypes.c_uint64 * 16)()
        ws = self.empty(32)
        self._ck(self.L.debwt_dev_partition(_p(a), _p(b) if b is not None else ctypes.c_void_p(0), _p(dest), _u64(n),
                                            ctypes.c_uint32(n_ranks), _p(out_a),
                                            _p(out_b) if out_b is not None else ctypes.c_void_p(0), counts, _p(ws), self._st()))
        return out_a, out_b, [int(counts[i]) for i in range(n_ranks)]

    def partition_by_splitters(self, items, splitters, n_split, mask, drop_marker, n_ranks):
        out = torch.empty_like(items)
        counts = (ctypes.c_uint64 * 16)()
        ws = self.empty(32)
        self._ck(self.L.debwt_dev_partition_by_splitters(_p(items), _u64(items.numel()), _p(splitters), ctypes.c_uint32(n_split),
                                                         _u64(mask), int(bool(drop_marker)), ctypes.c_uint32(n_ranks), _p(out),
                                                         counts, _p(ws), self._st()))
        return out, [int(counts[i]) for i in range(n_ranks)]

    def partition_count(self, items, splitters, n_split, mask, drop_marker, n_ranks):
        counts = (ctypes.c_uint64 * 16)()
        ws = self.empty(32)
        self._ck(self.L.debwt_dev_partition_count(_p(items), _u64(items.numel()), _p(splitters), ctypes.c_uint32(n_split), _u64(mask),
                                                  int(bool(drop_marker)), ctypes.c_uint32(n_ranks), counts, _p(ws), self._st()))
        return [int(counts[i]) for i in range(n_ranks)]

    def partition_scatter_p2p(self, items, splitters, n_split, mask, drop_marker, n_ranks, dst):
        ws = self.empty(32)
        self._ck(self.L.debwt_dev_partition_scatter_p2p(_p(items), _u64(items.numel()), _p(splitters), ctypes.c_uint32(n_split),
                                                        _u64(mask), int(bool(drop_marker)), ctypes.c_uint32(n_ranks), dst, _p(ws),
                                                        self._st()))

    def key_index(self, sorted_keys):
        n = sorted_keys.numel()
        bits = int(self.L.debwt_dev_key_index_bits(_u64(n)))
        idx = self.empty((1 << bits) + 2, torch.int32)
        self._ck(self.L.debwt_dev_key_index(_p(sorted_keys), _u64(n), _p(idx), bits, self._st()))
        return idx, bits

    def out_edges_queries(self, sorted_keys, gmask):
        q = self.empty(sorted_keys.numel())
        self._ck(self.L.debwt_dev_out_edges_queries(_p(sorted_keys), _u64(sorted_keys.numel()), _p(gmask), _p(q), self._st()))
        return q

    def apply_in_queries(self, sorted_keys, ki, gmask, q):
        self._ck(self.L.debwt_dev_apply_in_queries(_p(sorted_keys), _u64(sorted_keys.numel()), _p(ki[0]), ki[1], _p(gmask),
                                                   _p(q), _u64(q.numel()), self._st()))

    def heads_tails(self, words, seps, n_rec, sorted_keys, ki, gmask):
        self._ck(self.L.debwt_dev_heads_tails(_p(words), _p(seps), _u64(n_rec), _p(sorted_keys), _u64(sorted_keys.numel()),
                                              _p(ki[0]), ki[1], _p(gmask), self._st()))

    def propagate(self, sorted_keys, gmask):
        self._ck(self.L.debwt_dev_propagate(_p(sorted_keys), _u64(sorted_keys.numel()), _p(gmask), self._st()))

    def branch_table(self, sorted_keys, gmask):
        n = sorted_keys.numel()
        nb, nblue = ctypes.c_uint64(), ctypes.c_uint64()
        if n == 0:
            return {"kmer": self.empty(0), "head": self.empty(0, torch.int32), "blue": self.zeros(1, torch.int32), "B": 0, "M": 0}
        ws = self.empty(self._bytes("debwt_dev_branch_workspace_bytes", _u64(n)), torch.uint8)
        self._ck(self.L.debwt_dev_branch_count(_p(sorted_keys), _u64(n), _p(gmask), ctypes.byref(nb), ctypes.byref(nblue),
                                               _p(ws), self._st()))
        B, M = nb.value, nblue.value
        kmer, head, blue = self.empty(B + 1), self.empty(B + 1, torch.int32), self.zeros(B + 2, torch.int32)
        self._ck(self.L.debwt_dev_branch_write(_p(sorted_keys), _u64(n), _p(gmask), _p(ws), _p(kmer), _p(head), _p(blue), _u64(B),
                                               _u64(M), self._st()))
        return {"kmer": kmer[:B], "head": head[:B], "blue": blue[:B + 1], "B": B, "M": M}

    def branch_index(self, gkmer):
        B = gkmer.numel()
        bits = 8
        while bits < 27 and (1 << bits) < 2 * B:
            bits += 1
        bidx = self.empty(self._bytes("debwt_dev_branch_index_words", bits), torch.int32)
        self._ck(self.L.debwt_dev_branch_index(_p(gkmer), _u64(B), _p(bidx), bits, self._st()))
        return bidx, bits

    def special_scan(self, words, seps, n_rec, sorted_keys, ki):
        info = self.empty(4 * 32 * n_rec)          # 32-byte records
        self._ck(self.L.debwt_dev_special_scan(_p(words), _p(seps), _u64(n_rec), _p(sorted_keys), _u64(sorted_keys.numel()),
                                               _p(ki[0]), ki[1], _p(info), self._st()))
        return info.cpu().numpy()

    def flag_slice(self, words, pos_lo, pos_hi, seps, n_rec, gkmer, gbidx, nbw, cap):
        mo = self.zeros(nbw + 2, torch.int32)
        rec_entry, rec_index, cnt = self.empty(cap), self.empty(cap), self.zeros(1)
        bidx, bits = gbidx
        self._ck(self.L.debwt_dev_flag_slice(_p(words), _u64(pos_lo), _u64(pos_hi), _p(seps), _u64(n_rec), _p(gkmer),
                                             _u64(gkmer.numel()), _p(bidx), bits, _p(mo), _p(rec_entry), _p(rec_index), _p(cnt),
                                             self._st()))
        m = int(cnt.item())
        return mo, rec_entry[:m], rec_index[:m]

    def patch_bits_slice(self, mo, pos_lo, pos_hi, positions):
        self._ck(self.L.debwt_dev_patch_bits_slice(_p(mo), _u64(pos_lo), _u64(pos_hi), _p(positions), _u64(positions.numel()),
                                                   self._st()))

    def scan_popc(self, mo, nbw):
        wp = self.empty(nbw + 2, torch.int32)
        total = ctypes.c_uint64()
        ws = self.empty(self._bytes("debwt_dev_scan_workspace_bytes", _u64(nbw)), torch.uint8)
        self._ck(self.L.debwt_dev_scan_popc(_p(mo), _p(wp), _u64(nbw), ctypes.byref(total), _p(ws), self._st()))
        return wp, total.value

    def emit_codes_slice(self, words, word_lo, nbw, mo, wp, code_base, codes):
        self._ck(self.L.debwt_dev_emit_codes_slice(_p(words), _u64(word_lo), _u64(nbw), _p(mo), _p(wp), _u64(code_base), _p(codes),
                                                   self._st()))

    def mark_sep_slice(self, mo, wp, pos_lo, pos_hi, code_base, tail_pos, sep):
        out = self.zeros(tail_pos.numel())
        self._ck(self.L.debwt_dev_mark_sep_slice(_p(mo), _p(wp), _u64(pos_lo), _u64(pos_hi), _u64(code_base), _p(tail_pos),
                                                 _u64(tail_pos.numel()), _p(sep), _p(out), self._st()))
        return out

    def fix_records(self, rec_entry, mo, wp, pos_lo, code_base):
        self._ck(self.L.debwt_dev_fix_records(_p(rec_entry), _u64(rec_entry.numel()), _p(mo), _p(wp), _u64(pos_lo),
                                              _u64(code_base), self._st()))

    def scatter_blue(self, rec_entry, rec_local, bt):
        blue = self.empty(bt["M"] + 1)
        cursor = self.zeros(bt["B"] + 1, torch.int32)
        self._ck(self.L.debwt_dev_scatter_blue(_p(rec_entry), _p(rec_local), _u64(rec_entry.numel()), _p(bt["kmer"]),
                                               _p(bt["blue"]), _p(cursor), _u64(bt["B"]), _p(blue), self._st()))
        return blue

    def release_cached(self, m):
        """K10 takes its work lists from the driver's stream-ordered pool, not from torch: for large builds hand torch's
        cached (free) blocks back first"""
        if m > (64 << 20):
            torch.cuda.synchronize(self.device)
            torch.cuda.empty_cache()

    def sort_blue(self, blue, bt, codes, sep, dollar_index, n_codes):
        if bt["M"] == 0:
            return
        work = self.zeros(4 * bt["B"] + 16, torch.int32)
        self._ck(self.L.debwt_dev_sort_blue(_p(blue), _p(bt["kmer"]), _p(bt["blue"]), _u64(bt["B"]), _u64(bt["M"]), _p(codes),
                                            _p(sep), _u64(dollar_index), _u64(n_codes), _p(work), self._st()))

    def bwt_segment(self, word_lo, word_hi):
        """zeroed words [word_lo, word_hi) of the BWT: (the segment, a handle the emit kernels index with GLOBAL word numbers)"""
        seg = self.zeros(max(word_hi - word_lo, 0) + 1)
        return seg, _Shifted(seg, 8 * word_lo)

    def fill_range(self, gmask, n_keys, key_base, n_symbols, spec_rows, word_lo, word_hi, bwt):
        self._ck(self.L.debwt_dev_fill_range(_p(gmask), _u64(n_keys), _u64(key_base), _u64(n_symbols), _p(spec_rows),
                                             _u64(spec_rows.numel()), _u64(word_lo), _u64(word_hi), _p(bwt), self._st()))

    def emit_blue(self, blue, bt, key_base, spec_ins, bwt, n_rec):
        sharp = self.zeros(n_rec + 1)
        cnt = self.zeros(4, torch.int32)
        dollar = torch.full((2,), -1, dtype=torch.int64, device=self.device)
        if bt["M"]:
            self._ck(self.L.debwt_dev_emit_blue(_p(blue), _p(bt["kmer"]), _p(bt["head"]), _p(bt["blue"]), _u64(bt["B"]),
                                                _u64(bt["M"]), _u64(key_base), _p(spec_ins), _u64(spec_ins.numel()), _p(bwt),
                                                _p(sharp), _p(cnt), _p(dollar), self._st()))
        k = int(cnt[0].item())
        return sharp[:k], dollar[:1]

    def emit_special(self, spec_rows, spec_chr, bwt):
        self._ck(self.L.debwt_dev_emit_special(_p(spec_rows), _p(spec_chr), _u64(spec_rows.numel()), _p(bwt), self._st()))

    def special_tables(self, info_np, ins_by_t, seps_np, n_rec):
        return special_tables_host(info_np, ins_by_t, seps_np, n_rec)

    def sync(self):
        torch.cuda.synchronize(self.device)

    def free_gib(self):
        return torch.cuda.mem_get_info(self.device)[0] / 2**30


def special_tables_host(info_np, ins_by_t, seps_np, n_rec):
    """host part of the sentinel-window handling (debwt_special_tables in libdebwt_b200.so; no GPU needed)"""
    L = binding.lib()
    m = 32 * n_rec
    info_np = np.ascontiguousarray(info_np)
    ins_by_t = np.ascontiguousarray(ins_by_t, dtype=np.uint64)
    seps_np = np.ascontiguousarray(seps_np, dtype=np.uint64)
    ins, rows, emit, tail = (np.zeros(m, np.uint64), np.zeros(m, np.uint64), np.zeros(m, np.uint64), np.zeros(n_rec, np.uint64))
    chr_ = np.zeros(m, np.uint8)
    n_emit = ctypes.c_uint64()
    vp = ctypes.c_void_p
    L.debwt_special_tables.restype = ctypes.c_int
    binding.check(L.debwt_special_tables(vp(info_np.ctypes.data), vp(ins_by_t.ctypes.data), vp(seps_np.ctypes.data),
                                         ctypes.c_uint64(n_rec), vp(ins.ctypes.data), vp(rows.ctypes.data), vp(chr_.ctypes.data),
                                         vp(emit.ctypes.data), ctypes.byref(n_emit), vp(tail.ctypes.data)))
    return ins, rows, chr_, emit[:n_emit.value].copy(), tail


# --------------------------------------------------------------------------------------------------
# fused bucket + exchange over NVLink peer memory
# --------------------------------------------------------------------------------------------------
class _Shifted:
    """a device buffer addressed from a virtual origin `shift` bytes before its first element"""

    def __init__(self, t: torch.Tensor, shift: int):
        self.t, self.shift = t, shift

    def data_ptr(self):
        return self.t.data_ptr() - self.shift


class _RawCuda:
    """zero-copy view of a raw device pointer for torch.as_tensor"""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 2}


class PeerExchange:
    """All-to-all of 64-bit items without a staging buffer: every rank exports a receive buffer through CUDA
    IPC, the partition kernel stores each item straight into its owner's buffer (coalesced peer stores over
    NVLink / NVSwitch), and a barrier closes the exchange.  Only the G x G count matrix goes through
    torch.distributed.  Used for the key exchange and for the in-edge queries when the backend is NCCL."""

    _cache: dict = {}

    @classmethod
    def get(cls, comm: "Comm", ops, name: str) -> "PeerExchange":
        key = (id(comm), name)
        if key not in cls._cache:
            cls._cache[key] = PeerExchange(comm, ops)
        return cls._cache[key]

    def __init__(self, comm: "Comm", ops):
        self.comm, self.ops, self.cap = comm, ops, 0
        self.ptrs = [0] * comm.size

    def _release(self):
        L = self.ops.L
        for r, p in enumerate(self.ptrs):
            if not p:
                continue
            if r == self.comm.rank:
                L.debwt_dev_ipc_free(ctypes.c_void_p(p))
            else:
                L.debwt_dev_ipc_close(ctypes.c_void_p(p))
        self.ptrs = [0] * self.comm.size
        self.cap = 0

    def _ensure(self, need: int):
        """collective: `need` is the same on every rank"""
        if need <= self.cap:
            return
        torch.cuda.synchronize()
        self.comm.barrier()                      # nobody is still writing into / reading from the old buffers
        self._release()
        cap = int(need * 1.25) + 4096
        L = self.ops.L
        ptr, handle = ctypes.c_void_p(), (ctypes.c_ubyte * 64)()
        binding.check(L.debwt_dev_ipc_alloc(ctypes.c_uint64(cap * 8), ctypes.byref(ptr), handle))
        mine = torch.tensor(list(handle), dtype=torch.uint8)
        allh = self.comm.all_gather_equal(self.comm.to_coll(mine)).cpu().numpy()
        for r in range(self.comm.size):
            if r == self.comm.rank:
                self.ptrs[r] = ptr.value
            else:
                h = (ctypes.c_ubyte * 64)(*allh[r * 64:(r + 1) * 64].tolist())
                p = ctypes.c_void_p()
                binding.check(L.debwt_dev_ipc_open(h, ctypes.byref(p)))
                self.ptrs[r] = p.value
        self.cap = cap

    def exchange(self, items: torch.Tensor, d_split: torch.Tensor, n_split: int, drop_marker: bool) -> torch.Tensor:
        comm, ops, G, me = self.comm, self.ops, self.comm.size, self.comm.rank
        counts = ops.partition_count(items, d_split, n_split, 0xFFFFFFFFFFFFFFFC, drop_marker, G)
        mat = comm.all_gather_equal(comm.to_coll(torch.tensor(counts, dtype=torch.int64))).cpu().view(G, G)   # [src][dst]
        self._ensure(int(mat.sum(0).max()))
        dst = (ctypes.c_void_p * G)(*[self.ptrs[d] + 8 * int(mat[:me, d].sum()) for d in range(G)])
        ops.partition_scatter_p2p(items, d_split, n_split, 0xFFFFFFFFFFFFFFFC, drop_marker, G, dst)
        torch.cuda.synchronize()
        comm.barrier()                            # every peer has finished storing into this rank's buffer
        comm.bytes_sent += int(mat[me].sum() - mat[me, me]) * 8
        n_recv = int(mat[:, me].sum())
        if n_recv == 0:
            return items.new_empty(0)
        return torch.as_tensor(_RawCuda(self.ptrs[me], n_recv), device=items.device)


# --------------------------------------------------------------------------------------------------
# host-side geometry
# --------------------------------------------------------------------------------------------------
def valid_windows_before(x: int, seps: np.ndarray) -> int:
    """number of in-record 32-mer windows that start at a position < x"""
    starts = np.concatenate(([0], seps[:-1].astype(np.int64) + 1))
    last = seps.astype(np.int64) - 32                      # last valid start of each record
    cnt = np.clip(np.minimum(last + 1, x) - starts, 0, None)
    return int(cnt.sum())


def slice_geometry(n_symbols: int, size: int):
    """32-aligned position slices: (words per slice, total words incl. padding and guard)"""
    n_words = (n_symbols + 32 + 31) // 32 + 1
    wp = -(-n_words // size)
    return wp, wp * size


def choose_splitters(sorted_samples: np.ndarray, size: int) -> np.ndarray:
    """G-1 splitters on k-mer boundaries (low 2 bits cleared) from the sorted sample"""
    m = sorted_samples.size
    if size == 1:
        return np.zeros(0, dtype=np.uint64)
    if m == 0:
        return np.full(size - 1, np.uint64(0xFFFFFFFFFFFFFFFC), dtype=np.uint64)
    idx = (np.arange(1, size) * m) // size
    return (sorted_samples[idx] & np.uint64(0xFFFFFFFFFFFFFFFC)).astype(np.uint64)


# --------------------------------------------------------------------------------------------------
# the sharded build
# --------------------------------------------------------------------------------------------------
def my_slice(n_symbols: int, comm: Comm):
    """[pos_lo, pos_hi) of the text this rank uploads and works on"""
    wp, _ = slice_geometry(n_symbols, comm.size)
    lo = 32 * comm.rank * wp
    return lo, max(min(32 * (comm.rank + 1) * wp, n_symbols), lo)


def build_sharded(text: np.ndarray | None, seps: np.ndarray, comm: Comm, ops, stats: dict | None = None,
                  n_symbols: int | None = None, ascii_slice=None, fetch: bool = True):
    """text: the ASCII text T (every rank passes the same array; only its slice is uploaded), or None when
    `ascii_slice` already holds this rank's slice (`my_slice`) on the device and `n_symbols` = len(T).
    Returns (words, sharp_rows, dollar_row) on rank 0 and (None, None, None) elsewhere; with fetch=False
    the packed BWT stays on rank 0's device and is returned as a tensor."""
    G, r = comm.size, comm.rank
    if G > 16:
        raise binding.DebwtError("at most 16 ranks")
    import time as _time
    phases = {}
    _t = [_time.perf_counter()]

    def tick(name):
        if stats is not None and stats.get("profile"):
            ops.sync()
            if hasattr(ops, "free_gib"):
                phases["min_free_gib"] = min(phases.get("min_free_gib", 1e9), ops.free_gib())
            now = _time.perf_counter()
            phases[name] = phases.get(name, 0.0) + (now - _t[0]) * 1e3
            _t[0] = now

    N, R = int(text.size if text is not None else n_symbols), int(seps.size)
    seps = np.ascontiguousarray(seps, dtype=np.uint64)
    NK = N - 32 * R
    wp, wtot = slice_geometry(N, G)
    pos_lo, pos_hi_al = 32 * r * wp, 32 * (r + 1) * wp
    pos_hi = max(min(pos_hi_al, N), pos_lo)                 # a slice may lie entirely in the padding
    d_seps = ops.from_numpy(seps)

    # 1. pack own slice, all-gather the packed text
    n_valid = max(0, pos_hi - pos_lo)
    if ascii_slice is None:
        ascii_slice = ops.from_numpy(text[pos_lo:pos_hi] if n_valid else np.zeros(1, np.uint8))
    my_words = ops.zeros(wp)
    err = ops.zeros(4, torch.int32)
    ops.pack(ascii_slice, n_valid, my_words, wp, err)
    words = torch.cat([comm.all_gather_equal(my_words), ops.zeros(2)])
    err = comm.all_reduce_sum(err)
    if int(err[0].item()):
        raise binding.DebwtError("input contains a symbol other than A, C, G, T (either case)")
    if int(err[1].item()) != R:
        raise binding.DebwtError("input contains '#' or '$' inside a record (they are reserved for the record separators)")
    del ascii_slice

    tick('pack+allgather')
    # 2. keys of own slice, splitters
    idx_base = valid_windows_before(pos_lo, seps)
    cnt = valid_windows_before(pos_hi, seps) - idx_base if n_valid else 0
    keys = ops.empty(cnt)
    if cnt:
        ops.extract(words, pos_lo, pos_hi, d_seps, R, idx_base, keys, n_symbols=N)
    sample = torch.full((SAMPLES_PER_RANK,), I64_ALL_ONES, dtype=torch.int64, device=keys.device)
    ns = min(cnt, SAMPLES_PER_RANK)
    if ns:
        stride = max(cnt // ns, 1)
        sample[:ns] = keys[::stride][:ns]
    all_samples = comm.all_gather_equal(sample)
    ns_all = comm.all_gather_scalar(ns)
    valid = torch.cat([all_samples[i * SAMPLES_PER_RANK:i * SAMPLES_PER_RANK + ns_all[i]] for i in range(G)])
    sorted_samples = ops.sort(valid.contiguous()).cpu().numpy().view(np.uint64)
    splitters_np = choose_splitters(sorted_samples, G)
    d_split = ops.from_numpy(splitters_np) if G > 1 else ops.zeros(1)
    n_split = G - 1

    import os as _os
    use_p2p = (G > 1 and isinstance(ops, CudaOps) and not comm.staged and comm.coll_device.type == "cuda"
               and _os.environ.get("DEBWT_P2P", "1") != "0")

    def exchange(items, drop_marker, name):
        """every item goes to the owner of its k-mer (top 62 bits): fused bucket + peer stores over NVLink when
        the ranks can map each other's memory, else bucket + all-to-all through torch.distributed"""
        if use_p2p:
            return PeerExchange.get(comm, ops, name).exchange(items, d_split, n_split, drop_marker)
        part, counts = ops.partition_by_splitters(items, d_split, n_split, 0xFFFFFFFFFFFFFFFC, drop_marker, G)
        got, _ = comm.all_to_all_v(part, counts)
        return got

    tick('extract+splitters')
    # 3. one all-to-all: every key goes to the owner of its k-mer
    mine = exchange(keys, False, "keys")
    del keys
    tick('partition+alltoall')
    n_loc = int(mine.numel())
    sk = ops.sort(mine, True) if getattr(ops, "timed_main_sort", False) else ops.sort(mine)
    n_all = comm.all_gather_scalar(n_loc)
    if sum(n_all) != NK:
        raise binding.DebwtError("internal: key exchange lost keys")
    key_base = sum(n_all[:r])

    tick('sort')
    # 4. branch k-mer detection on the owned key range
    ki = ops.key_index(sk)
    gmask = ops.zeros(n_loc + 2, torch.int16)
    tick('c.index')
    q = ops.out_edges_queries(sk, gmask) if n_loc else ops.empty(0)
    tick('c.out_edges')
    qrecv = exchange(q, True, "queries")
    tick('c.exchange')
    if n_loc:
        ops.apply_in_queries(sk, ki, gmask, qrecv)
        tick('c.apply')
        ops.heads_tails(words, d_seps, R, sk, ki, gmask)
        ops.propagate(sk, gmask)
    del q, qrecv
    tick('c.propagate')
    bt = ops.branch_table(sk, gmask)
    tick('c.branch')
    gkmer, b_all = comm.all_gather_var(bt["kmer"])
    b_base = np.concatenate(([0], np.cumsum(b_all))).astype(np.uint64)
    m_all = comm.all_gather_scalar(bt["M"])
    gbidx = ops.branch_index(gkmer)

    tick('classify+branch')
    # 5. sentinel-window suffixes (ranked redundantly on every rank; insertion points are summed)
    info = ops.special_scan(words, d_seps, R, sk, ki)
    info_rec = info.view(np.uint64).reshape(-1, 4)
    ins_local = torch.from_numpy(info_rec[:, 2].astype(np.int64).copy())
    ins_global = comm.all_reduce_sum(comm.to_coll(ins_local)).cpu().numpy()
    ins, rows, chr_, emit_pos, tail_pos = ops.special_tables(info, ins_global.astype(np.uint64), seps, R)
    d_rows, d_ins, d_chr = ops.from_numpy(rows), ops.from_numpy(ins), ops.from_numpy(chr_)
    d_emit = ops.from_numpy(emit_pos) if emit_pos.size else ops.empty(0)
    d_tail = ops.from_numpy(tail_pos)

    tick('special')
    # 6. branch codes of own position slice at global code indices
    cap = min(cnt, sum(m_all)) + 1
    mo, rec_entry, rec_index = ops.flag_slice(words, pos_lo, pos_hi, d_seps, R, gkmer, gbidx, wp, cap)
    if d_emit.numel():
        ops.patch_bits_slice(mo, pos_lo, pos_hi_al, d_emit)
    wpfx, s_loc = ops.scan_popc(mo, wp)
    s_all = comm.all_gather_scalar(s_loc)
    code_base, s_tot = sum(s_all[:r]), sum(s_all)
    ncw = s_tot // 32 + 3
    codes, sep = ops.zeros(ncw), ops.zeros(ncw + 1, torch.int32)
    ops.emit_codes_slice(words, r * wp, wp, mo, wpfx, code_base, codes)
    tail_idx = ops.mark_sep_slice(mo, wpfx, pos_lo, pos_hi_al, code_base, d_tail, sep)
    comm.all_reduce_sum(codes)
    comm.all_reduce_sum(sep)
    comm.all_reduce_sum(tail_idx)
    dollar_index = int(tail_idx[R - 1].item())
    if rec_entry.numel():
        ops.fix_records(rec_entry, mo, wpfx, pos_lo, code_base)

    tick('codes')
    # 7. blue entries travel to the owner of their k-mer
    d_bbase = ops.from_numpy(b_base)
    db = ops.owner_of_index(rec_index, d_bbase, G) if rec_index.numel() else ops.empty(0, torch.uint8)
    e_part, i_part, rcounts = ops.partition(rec_entry, rec_index, db, G)
    del rec_entry, rec_index, db, mo, wpfx          # at 30 Gbp every one of these is gigabytes per rank
    e_recv, _ = comm.all_to_all_v(e_part, rcounts)
    del e_part
    i_recv, _ = comm.all_to_all_v(i_part, rcounts)
    del i_part
    if int(e_recv.numel()) != bt["M"]:
        raise binding.DebwtError("internal: blue entry exchange mismatch")
    blue = ops.scatter_blue(e_recv, i_recv, bt)
    del e_recv, i_recv
    ops.release_cached(bt["M"])
    ops.sort_blue(blue, bt, codes, sep, dollar_index, s_tot)

    tick('blue')
    # 8. every rank emits its own contiguous run of BWT rows into a buffer of just that size (SURVEY 8e step 6).
    #    Rank r owns the rows from its first key's row up to the next rank's first key's row; the sentinel-window suffixes
    #    inserted in between belong to the rank whose keys precede them.  Rank 0 stitches: interior words are copied,
    #    the at most one word shared with a neighbour is OR-ed (disjoint 2-bit fields).
    n_out = (N + 31) // 32
    kb = np.concatenate(([0], np.cumsum(n_all))).astype(np.uint64)

    def row_lo(q):
        return 0 if int(kb[q]) == 0 else int(kb[q]) + int(np.searchsorted(ins, kb[q], side="right"))
    r_lo_all = [row_lo(q) for q in range(G)] + [N]
    my_lo, my_hi = r_lo_all[r], r_lo_all[r + 1]
    w_lo, w_hi = my_lo >> 5, (my_hi + 31) >> 5
    seg, bwt_h = ops.bwt_segment(w_lo, w_hi)
    if my_hi > my_lo:
        if n_loc:
            ops.fill_range(gmask, n_loc, key_base, N, d_rows, w_lo, w_hi, bwt_h)
        t_lo, t_hi = int(np.searchsorted(rows, np.uint64(my_lo), side="left")), int(np.searchsorted(rows, np.uint64(my_hi), side="left"))
        if t_hi > t_lo:
            ops.emit_special(d_rows[t_lo:t_hi], d_chr[t_lo:t_hi], bwt_h)
    sharp, dollar = ops.emit_blue(blue, bt, key_base, d_ins, bwt_h, R)
    seg_words = [((r_lo_all[q + 1] + 31) >> 5) - (r_lo_all[q] >> 5) for q in range(G)]
    mx = max(max(seg_words), 1)
    pad = seg if seg.numel() == mx else torch.cat([seg[:min(seg.numel(), mx)], seg.new_zeros(max(mx - seg.numel(), 0))])
    parts = comm.gather_to0(pad[:mx].contiguous())
    bwt = None
    if r == 0:
        bwt = ops.zeros(n_out + 1)
        for q in range(G):
            if seg_words[q] > 0:
                lo_q = r_lo_all[q] >> 5
                bwt[lo_q:lo_q + seg_words[q]] |= parts[q][:seg_words[q]]
    sharp_all, _ = comm.all_gather_var(sharp)
    comm.all_reduce_max(dollar)
    tick('emit+reduce')
    if stats is not None:
        stats["phases_ms"] = phases
        stats.update({"n_symbols": N, "n_keys": NK, "keys_local": n_all, "n_branch": int(sum(b_all)), "n_blue": int(sum(m_all)),
                      "n_codes": int(s_tot), "bytes_sent": comm.bytes_sent, "launches": getattr(ops, "launches", 0)})
    if r != 0:
        return None, None, None
    if not fetch:
        return bwt[:n_out], sharp_all, dollar
    words_np = bwt[:n_out].cpu().numpy().view(np.uint64).copy()
    sharp_np = np.sort(sharp_all.cpu().numpy().view(np.uint64))
    dollar_np = dollar.cpu().numpy().view(np.uint64).copy()
    if sharp_np.size != R - 1 or dollar_np[0] == np.uint64(0xFFFFFFFFFFFFFFFF):
        raise binding.DebwtError("internal: wrong number of separator rows")
    return words_np, sharp_np, dollar_np
