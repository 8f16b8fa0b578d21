/*
 * deBWT-B200 -- device-pointer stage ABI for the sharded (multi-GPU) path.
 *
 * Stateless kernel launchers on raw CUDA device pointers (`void*`) and a CUDA stream passed as
 * `void*` (0 = the legacy default stream).  The host program owns the device buffers and the
 * collectives (torch.distributed / NCCL: debwt_b200/dist.py); the library owns the kernels.  The
 * reference has no distributed code (SURVEY.md section 2.1); these calls are the slice- / key-range-
 * aware forms of the stages declared in debwt_b200.h, plus the bucket-by-owner partition (K12).
 * Every function returns 0 on success, negative on error (debwt_last_error()).
 * All sizes are in elements unless stated; u64 arrays are `uint64_t`, masks `uint16_t`.
 */
#ifndef DEBWT_B200_DEV_H
#define DEBWT_B200_DEV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* once per process and device: keeps the driver's stream-ordered pool from returning memory at every sync
   (K10 takes its round scratch from it) */
int debwt_dev_init(int device);

/* K1 on a text slice: n ASCII symbols -> nwords packed words (T padding for [n, n+32), zeros beyond);
   *d_err (u32, device) is OR-ed with 1 on a non-ACGT symbol (src/collect#$.c:66-90). */
int debwt_dev_pack(const void* d_ascii, uint64_t n, void* d_words, uint64_t nwords, void* d_err, void* stream);
/* K2 on positions [pos_lo, pos_hi): key of window p in record r goes to keys[p - 32 r - idx_base].  Runs the tiled
   kernel of the single-GPU path (packed words staged in shared memory, one record lookup per tile); pos_lo must be a
   multiple of 32, d_words must hold the whole packed text of n_symbols symbols. */
int debwt_dev_extract_slice(const void* d_words, uint64_t n_symbols, uint64_t pos_lo, uint64_t pos_hi, const void* d_seps,
                            uint64_t n_rec, uint64_t idx_base, void* d_keys, void* stream);
/* Workspaces are provided by the caller (device memory, sizes in bytes from the *_workspace_bytes calls):
   no call in this header allocates or frees device memory. */
uint64_t debwt_dev_sort_workspace_bytes(uint64_t n, int cfg);
uint64_t debwt_dev_branch_workspace_bytes(uint64_t n);
uint64_t debwt_dev_scan_workspace_bytes(uint64_t n_words);
/* K3: sorts n keys held in d_a using d_b as scratch; *result_in_b = 1 when the sorted keys end in d_b. */
int debwt_dev_sort(void* d_a, void* d_b, uint64_t n, int cfg, void* d_workspace, int* result_in_b, void* stream);
/* same, synchronous, with device times: whole sort and the scatter passes alone (CUDA events on `stream`) */
int debwt_dev_sort_timed(void* d_a, void* d_b, uint64_t n, int cfg, void* d_workspace, int* result_in_b, float* ms_total,
                         float* ms_sweeps, int* n_sweeps, void* stream);
/* K12: owner rank of each item = number of splitters <= (item & mask); with drop_marker, items equal to ~0
   (the "no query" marker) get owner 255 and are dropped by the partition. */
int debwt_dev_owner_of_keys(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                            int drop_marker, void* d_dest_u8, void* stream);
/* owner of a global table index given the n_ranks+1 ascending bases; idx is rewritten to the owner-local index */
int debwt_dev_owner_of_index(void* d_idx, uint64_t n, const void* d_bases, uint32_t n_ranks, void* d_dest_u8, void* stream);
/* groups a (and b when non-null) by owner; counts_out[r] = items of owner r (host array of n_ranks);
   d_workspace: 128 bytes */
int debwt_dev_partition(const void* d_a, const void* d_b, const void* d_dest_u8, uint64_t n, uint32_t n_ranks,
                        void* d_out_a, void* d_out_b, uint64_t* counts_out, void* d_workspace, void* stream);
/* same for 64-bit items whose owner is the number of splitters <= (item & mask), computed on the fly */
int debwt_dev_partition_by_splitters(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                                     int drop_marker, uint32_t n_ranks, void* d_out, uint64_t* counts_out, void* d_workspace,
                                     void* stream);
/* ---- fused bucket + exchange over NVLink peer memory --------------------------------------------
   Receive buffers are plain cudaMalloc allocations exported through CUDA IPC; every rank opens the
   buffers of its peers once.  A key exchange is then: count (below), all-gather of the counts (host),
   one scatter kernel that stores every item directly into its owner's receive buffer, barrier. */
int debwt_dev_ipc_alloc(uint64_t bytes, void** d_ptr, unsigned char handle_out[64]);
int debwt_dev_ipc_open(const unsigned char handle[64], void** d_ptr);
int debwt_dev_ipc_close(void* d_ptr);
int debwt_dev_ipc_free(void* d_ptr);
/* counts_out[r] = items owned by rank r (host array of n_ranks); d_workspace: 128 bytes */
int debwt_dev_partition_count(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                              int drop_marker, uint32_t n_ranks, uint64_t* counts_out, void* d_workspace, void* stream);
/* dst[r] (host array of n_ranks device pointers): start of this rank's slot in rank r's receive buffer */
int debwt_dev_partition_scatter_p2p(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                                    int drop_marker, uint32_t n_ranks, void* const* dst, void* d_workspace, void* stream);
/* direct index over sorted keys */
int debwt_dev_key_index_bits(uint64_t n);
int debwt_dev_key_index(const void* d_sorted, uint64_t n, void* d_idx_u32, int bits, void* stream);
/* K5/K6 split: out-edges are local; in-edges become queries (X<<2|c, ~0 = none) for the owner of X */
int debwt_dev_out_edges_queries(const void* d_sorted, uint64_t n, void* d_gmask, void* d_queries, void* stream);
int debwt_dev_apply_in_queries(const void* d_sorted, uint64_t n, const void* d_idx_u32, int bits, void* d_gmask,
                               const void* d_queries, uint64_t m, void* stream);
int debwt_dev_heads_tails(const void* d_words, const void* d_seps, uint64_t n_rec, const void* d_sorted, uint64_t n,
                          const void* d_idx_u32, int bits, void* d_gmask, void* stream);
int debwt_dev_propagate(const void* d_sorted, uint64_t n, void* d_gmask, void* stream);
/* K7: two calls sharing one workspace; the first returns B and M */
int debwt_dev_branch_count(const void* d_sorted, uint64_t n, const void* d_gmask, uint64_t* n_branch, uint64_t* n_blue,
                           void* d_workspace, void* stream);
int debwt_dev_branch_write(const void* d_sorted, uint64_t n, const void* d_gmask, void* workspace, void* d_kmer,
                           void* d_head_u32, void* d_blue_u32 /* B+1 */, uint64_t n_branch, uint64_t n_blue, void* stream);
/* d_bidx_u32 holds debwt_dev_branch_index_words(bits) words: the direct index followed by a presence bitmap */
uint64_t debwt_dev_branch_index_words(int bits);
int debwt_dev_branch_index(const void* d_kmer, uint64_t n_branch, void* d_bidx_u32, int bits, void* stream);
/* sentinel-window suffixes: 32 R records of 32 bytes {w0,w1,ins,rank,prev,next} (ins is local to d_sorted) */
int debwt_dev_special_scan(const void* d_words, const void* d_seps, uint64_t n_rec, const void* d_sorted, uint64_t n,
                           const void* d_idx_u32, int bits, void* d_info, void* stream);
/* host-only: from the scan records (ins replaced by the GLOBAL insertion points in `ins_by_t`, indexed
   t = rec*32+j) to the tables the kernels consume, all in suffix order; returns the number of emitting positions */
int debwt_special_tables(const void* info_host, const uint64_t* ins_by_t, const uint64_t* seps, uint64_t n_rec,
                         uint64_t* ins_out, uint64_t* rows_out, uint8_t* chr_out, uint64_t* emit_pos_out,
                         uint64_t* n_emit_out, uint64_t* tail_pos_out);
/* K9 on a position slice */
int debwt_dev_flag_slice(const void* d_words, uint64_t pos_lo, uint64_t pos_hi, const void* d_seps, uint64_t n_rec,
                         const void* d_gkmer, uint64_t n_branch_total, const void* d_bidx_u32, int bits, void* d_mo_bits,
                         void* d_rec_entry, void* d_rec_index, void* d_rec_count, void* stream);
int debwt_dev_patch_bits_slice(void* d_mo_bits, uint64_t pos_lo, uint64_t pos_hi, const void* d_positions, uint64_t m,
                               void* stream);
int debwt_dev_scan_popc(const void* d_mo_bits, void* d_word_prefix, uint64_t nbw, uint64_t* total, void* d_workspace,
                        void* stream);
int debwt_dev_emit_codes_slice(const void* d_words, uint64_t word_lo, uint64_t nbw, const void* d_mo_bits,
                               const void* d_word_prefix, uint64_t code_base, void* d_codes, void* stream);
int debwt_dev_mark_sep_slice(const void* d_mo_bits, const void* d_word_prefix, uint64_t pos_lo, uint64_t pos_hi,
                             uint64_t code_base, const void* d_positions, uint64_t m, void* d_sep, void* d_out_idx,
                             void* stream);
int debwt_dev_fix_records(void* d_rec_entry, uint64_t m, const void* d_mo_bits, const void* d_word_prefix, uint64_t pos_lo,
                          uint64_t code_base, void* stream);
/* K10; d_work_u32: 4 * n_branch + 16 words */
int debwt_dev_scatter_blue(const void* d_rec_entry, const void* d_rec_local, uint64_t m, const void* d_kmer,
                           const void* d_blue_u32, void* d_cursor_u32, uint64_t n_branch, void* d_blue, void* stream);
int debwt_dev_sort_blue(void* d_blue, const void* d_kmer, const void* d_blue_u32, uint64_t n_branch, uint64_t n_blue,
                        const void* d_codes, const void* d_sep, uint64_t dollar_index, uint64_t n_codes, void* d_work_u32,
                        void* stream);
/* K8 / K11 on a key range */
int debwt_dev_fill_range(const void* d_gmask, uint64_t n_keys, uint64_t key_base, uint64_t n_symbols,
                         const void* d_spec_rows, uint64_t m, uint64_t word_lo, uint64_t word_hi, void* d_bwt, void* stream);
int debwt_dev_emit_blue(const void* d_blue, const void* d_kmer, const void* d_head_u32, const void* d_blue_u32,
                        uint64_t n_branch, uint64_t n_blue, uint64_t key_base, const void* d_spec_ins, uint64_t m,
                        void* d_bwt, void* d_sharp_rows, void* d_sharp_count_u32, void* d_dollar_row, void* stream);
int debwt_dev_emit_special(const void* d_spec_rows, const void* d_spec_chr, uint64_t m, void* d_bwt, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DEBWT_B200_DEV_H */
