// include/debwt_b200_dev.h: device-pointer stage ABI for the sharded path (thin wrappers).
#include <string.h>

#include <vector>

#include "../../include/debwt_b200_dev.h"
#include "dist_kernels.cuh"
#include "radix_sort.cuh"
#include "special.cuh"

using namespace debwt;

namespace {
inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline KeyIndex KI(const void* idx, int bits) {
    KeyIndex k;
    k.idx = reinterpret_cast<u32*>(const_cast<void*>(idx));
    k.bits = bits;
    return k;
}
inline BranchTable BT(const void* kmer, const void* head, const void* blue, void* cursor, const void* bidx, int bits,
                      u64 nb, u64 nblue) {
    BranchTable b;
    b.n_branch = nb; b.n_blue = nblue;
    b.kmer = reinterpret_cast<u64*>(const_cast<void*>(kmer));
    b.head = reinterpret_cast<u32*>(const_cast<void*>(head));
    b.blue = reinterpret_cast<u32*>(const_cast<void*>(blue));
    b.cursor = reinterpret_cast<u32*>(cursor);
    b.bidx = reinterpret_cast<u32*>(const_cast<void*>(bidx));
    b.bits = bits;
    return b;
}
#define P64(x) reinterpret_cast<u64*>(const_cast<void*>(static_cast<const void*>(x)))
#define P32(x) reinterpret_cast<u32*>(const_cast<void*>(static_cast<const void*>(x)))
#define P16(x) reinterpret_cast<u16*>(const_cast<void*>(static_cast<const void*>(x)))
#define P8(x) reinterpret_cast<u8*>(const_cast<void*>(static_cast<const void*>(x)))
}  // namespace

extern "C" {

int debwt_dev_init(int device) {
    CUDA_TRY(cudaSetDevice(device));
    cudaMemPool_t mp;
    CUDA_TRY(cudaDeviceGetDefaultMemPool(&mp, device));
    unsigned long long thr = ~0ull;
    CUDA_TRY(cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &thr));
    return 0;
}

int debwt_dev_pack(const void* d_ascii, uint64_t n, void* d_words, uint64_t nwords, void* d_err, void* stream) {
    return k_pack_words(P8(d_ascii), n, P64(d_words), nwords, P32(d_err), S(stream));
}

int debwt_dev_extract_slice(const void* d_words, uint64_t n_symbols, uint64_t pos_lo, uint64_t pos_hi, const void* d_seps,
                            uint64_t n_rec, uint64_t idx_base, void* d_keys, void* stream) {
    return k_extract_slice(P64(d_words), n_symbols, pos_lo, pos_hi, P64(d_seps), n_rec, idx_base, P64(d_keys), S(stream));
}

uint64_t debwt_dev_sort_workspace_bytes(uint64_t n, int cfg) { return sort_workspace_bytes(n, cfg); }
uint64_t debwt_dev_branch_workspace_bytes(uint64_t n) { return branch_workspace_bytes(n) + 64; }
uint64_t debwt_dev_scan_workspace_bytes(uint64_t n_words) { return scan_workspace_bytes(n_words) + 64; }

int debwt_dev_sort(void* d_a, void* d_b, uint64_t n, int cfg, void* d_workspace, int* result_in_b, void* stream) {
    SortWorkspace ws;
    sort_workspace_bind(ws, d_workspace, n, cfg);
    u64* res = nullptr;
    if (radix_sort_u64(P64(d_a), P64(d_b), n, ws, S(stream), &res)) return -1;
    if (result_in_b) *result_in_b = (res == P64(d_b)) ? 1 : 0;
    return 0;
}

int debwt_dev_sort_timed(void* d_a, void* d_b, uint64_t n, int cfg, void* d_workspace, int* result_in_b, float* ms_total,
                         float* ms_sweeps, int* n_sweeps, void* stream) {
    cudaStream_t st = S(stream);
    SortWorkspace ws;
    sort_workspace_bind(ws, d_workspace, n, cfg);
    static cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
    if (!e[0]) for (auto& x : e) CUDA_TRY(cudaEventCreate(&x));
    int sweeps = 0;
    ws.ev_sweep_begin = e[1]; ws.ev_sweep_end = e[2]; ws.sweeps_out = &sweeps;
    CUDA_TRY(cudaEventRecord(e[0], st));
    u64* res = nullptr;
    int rc = radix_sort_u64(P64(d_a), P64(d_b), n, ws, st, &res);
    CUDA_TRY(cudaEventRecord(e[3], st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (!rc) {
        if (ms_total) CUDA_TRY(cudaEventElapsedTime(ms_total, e[0], e[3]));
        if (ms_sweeps) { *ms_sweeps = 0; if (sweeps) CUDA_TRY(cudaEventElapsedTime(ms_sweeps, e[1], e[2])); }
        if (n_sweeps) *n_sweeps = sweeps;
        if (result_in_b) *result_in_b = (res == P64(d_b)) ? 1 : 0;
    }
    return rc;
}

int debwt_dev_owner_of_keys(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                            int drop_marker, void* d_dest_u8, void* stream) {
    return k_owner_of_keys(P64(d_items), n, P64(d_splitters), n_split, mask, drop_marker != 0, P8(d_dest_u8), S(stream));
}

int debwt_dev_owner_of_index(void* d_idx, uint64_t n, const void* d_bases, uint32_t n_ranks, void* d_dest_u8, void* stream) {
    return k_owner_of_index(P64(d_idx), n, P64(d_bases), n_ranks, P8(d_dest_u8), S(stream));
}

namespace {
int partition_impl(const u64* a, const u64* b, const PartitionBy& by, u64 n, u32 n_ranks, u64* out_a, u64* out_b,
                   uint64_t* counts_out, void* d_workspace, cudaStream_t st) {
    if (n_ranks == 0 || n_ranks > 16) { set_error("partition: 1..16 ranks"); return -1; }
    u64* d_counts = P64(d_workspace);
    CUDA_TRY(cudaMemsetAsync(d_counts, 0, 16 * 8, st));
    if (k_partition_count(a, by, n, n_ranks, d_counts, st)) return -1;
    u64 h[16];
    CUDA_TRY(cudaMemcpyAsync(h, d_counts, sizeof h, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    u64 cur[16], run = 0;
    for (int r = 0; r < 16; ++r) { cur[r] = run; run += h[r]; if ((u32)r < n_ranks) counts_out[r] = h[r]; }
    CUDA_TRY(cudaMemcpyAsync(d_counts, cur, sizeof cur, cudaMemcpyHostToDevice, st));
    if (k_partition_scatter(a, b, by, n, n_ranks, d_counts, out_a, out_b, st)) return -1;
    CUDA_TRY(cudaStreamSynchronize(st));     // `cur` lives on this stack frame
    return 0;
}
}  // namespace

int debwt_dev_partition(const void* d_a, const void* d_b, const void* d_dest_u8, uint64_t n, uint32_t n_ranks,
                        void* d_out_a, void* d_out_b, uint64_t* counts_out, void* d_workspace, void* stream) {
    PartitionBy by;
    by.dest = P8(d_dest_u8);
    return partition_impl(P64(d_a), d_b ? P64(d_b) : nullptr, by, n, n_ranks, P64(d_out_a), d_out_b ? P64(d_out_b) : nullptr,
                          counts_out, d_workspace, S(stream));
}

int debwt_dev_partition_by_splitters(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                                     int drop_marker, uint32_t n_ranks, void* d_out, uint64_t* counts_out, void* d_workspace,
                                     void* stream) {
    PartitionBy by;
    by.splitters = P64(d_splitters); by.n_split = n_split; by.mask = mask; by.drop_marker = drop_marker != 0;
    return partition_impl(P64(d_items), nullptr, by, n, n_ranks, P64(d_out), nullptr, counts_out, d_workspace, S(stream));
}

int debwt_dev_ipc_alloc(uint64_t bytes, void** d_ptr, unsigned char handle_out[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size is part of the ABI");
    CUDA_TRY(cudaMalloc(d_ptr, bytes ? bytes : 256));
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, *d_ptr));
    memcpy(handle_out, &h, 64);
    return 0;
}

int debwt_dev_ipc_open(const unsigned char handle[64], void** d_ptr) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CUDA_TRY(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

int debwt_dev_ipc_close(void* d_ptr) {
    CUDA_TRY(cudaIpcCloseMemHandle(d_ptr));
    return 0;
}

int debwt_dev_ipc_free(void* d_ptr) {
    CUDA_TRY(cudaFree(d_ptr));
    return 0;
}

int debwt_dev_partition_count(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                              int drop_marker, uint32_t n_ranks, uint64_t* counts_out, void* d_workspace, void* stream) {
    if (n_ranks == 0 || n_ranks > 16) { set_error("partition: 1..16 ranks"); return -1; }
    cudaStream_t st = S(stream);
    PartitionBy by;
    by.splitters = P64(d_splitters); by.n_split = n_split; by.mask = mask; by.drop_marker = drop_marker != 0;
    u64* d_counts = P64(d_workspace);
    CUDA_TRY(cudaMemsetAsync(d_counts, 0, 16 * 8, st));
    if (k_partition_count(P64(d_items), by, n, n_ranks, d_counts, st)) return -1;
    u64 h[16];
    CUDA_TRY(cudaMemcpyAsync(h, d_counts, sizeof h, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (u32 r = 0; r < n_ranks; ++r) counts_out[r] = h[r];
    return 0;
}

int debwt_dev_partition_scatter_p2p(const void* d_items, uint64_t n, const void* d_splitters, uint32_t n_split, uint64_t mask,
                                    int drop_marker, uint32_t n_ranks, void* const* dst, void* d_workspace, void* stream) {
    if (n_ranks == 0 || n_ranks > 16) { set_error("partition: 1..16 ranks"); return -1; }
    cudaStream_t st = S(stream);
    PartitionBy by;
    by.splitters = P64(d_splitters); by.n_split = n_split; by.mask = mask; by.drop_marker = drop_marker != 0;
    u64* d_cursors = P64(d_workspace);
    CUDA_TRY(cudaMemsetAsync(d_cursors, 0, 16 * 8, st));
    u64* d[16];
    for (u32 r = 0; r < n_ranks; ++r) d[r] = P64(dst[r]);
    return k_partition_scatter_p2p(P64(d_items), by, n, n_ranks, d_cursors, d, st);
}

int debwt_dev_key_index_bits(uint64_t n) { return key_index_bits(n); }

int debwt_dev_key_index(const void* d_sorted, uint64_t n, void* d_idx_u32, int bits, void* stream) {
    return k_build_key_index(P64(d_sorted), n, KI(d_idx_u32, bits), S(stream));
}

int debwt_dev_out_edges_queries(const void* d_sorted, uint64_t n, void* d_gmask, void* d_queries, void* stream) {
    return k_out_edges_queries(P64(d_sorted), n, P16(d_gmask), P64(d_queries), S(stream));
}

int debwt_dev_apply_in_queries(const void* d_sorted, uint64_t n, const void* d_idx_u32, int bits, void* d_gmask,
                               const void* d_queries, uint64_t m, void* stream) {
    return k_apply_in_queries(P64(d_sorted), n, KI(d_idx_u32, bits), P16(d_gmask), P64(d_queries), m, S(stream));
}

int debwt_dev_heads_tails(const void* d_words, const void* d_seps, uint64_t n_rec, const void* d_sorted, uint64_t n,
                          const void* d_idx_u32, int bits, void* d_gmask, void* stream) {
    return k_mark_heads_tails(P64(d_words), P64(d_seps), n_rec, P64(d_sorted), n, KI(d_idx_u32, bits), P16(d_gmask), S(stream));
}

int debwt_dev_propagate(const void* d_sorted, uint64_t n, void* d_gmask, void* stream) {
    return k_propagate(P64(d_sorted), n, P16(d_gmask), S(stream));
}

int debwt_dev_branch_count(const void* d_sorted, uint64_t n, const void* d_gmask, uint64_t* n_branch, uint64_t* n_blue,
                           void* d_workspace, void* stream) {
    cudaStream_t st = S(stream);
    char* ws = reinterpret_cast<char*>(d_workspace);
    u64* d_tot = reinterpret_cast<u64*>(ws);
    if (k_branch_count(P64(d_sorted), n, P16(d_gmask), false, ws + 64, d_tot, st)) return -1;
    u64 h[2];
    CUDA_TRY(cudaMemcpyAsync(h, d_tot, 16, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *n_branch = h[0]; *n_blue = h[1];
    return 0;
}

int debwt_dev_branch_write(const void* d_sorted, uint64_t n, const void* d_gmask, void* workspace, void* d_kmer,
                           void* d_head_u32, void* d_blue_u32, uint64_t n_branch, uint64_t n_blue, void* stream) {
    cudaStream_t st = S(stream);
    BranchTable bt = BT(d_kmer, d_head_u32, d_blue_u32, nullptr, nullptr, 0, n_branch, n_blue);
    if (k_branch_write(P64(d_sorted), n, P16(d_gmask), reinterpret_cast<char*>(workspace) + 64, bt, st)) return -1;
    const u32 m32 = (u32)n_blue;
    CUDA_TRY(cudaMemcpyAsync(P32(d_blue_u32) + n_branch, &m32, 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

uint64_t debwt_dev_branch_index_words(int bits) { return BranchTable::index_words(bits); }

int debwt_dev_branch_index(const void* d_kmer, uint64_t n_branch, void* d_bidx_u32, int bits, void* stream) {
    return k_branch_index(BT(d_kmer, nullptr, nullptr, nullptr, d_bidx_u32, bits, n_branch, 0), S(stream));
}

int debwt_dev_special_scan(const void* d_words, const void* d_seps, uint64_t n_rec, const void* d_sorted, uint64_t n,
                           const void* d_idx_u32, int bits, void* d_info, void* stream) {
    static_assert(sizeof(SpecialInfo) == 32, "SpecialInfo layout is part of the ABI");
    return k_special_scan(P64(d_words), P64(d_seps), n_rec, P64(d_sorted), n, KI(d_idx_u32, bits),
                          reinterpret_cast<SpecialInfo*>(d_info), S(stream));
}

int debwt_dev_flag_slice(const void* d_words, uint64_t pos_lo, uint64_t pos_hi, const void* d_seps, uint64_t n_rec,
                         const void* d_gkmer, uint64_t n_branch_total, const void* d_bidx_u32, int bits, void* d_mo_bits,
                         void* d_rec_entry, void* d_rec_index, void* d_rec_count, void* stream) {
    BranchTable bt = BT(d_gkmer, nullptr, nullptr, nullptr, d_bidx_u32, bits, n_branch_total, 0);
    return k_flag_slice(P64(d_words), pos_lo, pos_hi, P64(d_seps), n_rec, bt, P32(d_mo_bits), P64(d_rec_entry),
                        P64(d_rec_index), P64(d_rec_count), S(stream));
}

int debwt_dev_patch_bits_slice(void* d_mo_bits, uint64_t pos_lo, uint64_t pos_hi, const void* d_positions, uint64_t m,
                               void* stream) {
    return k_patch_bits(P32(d_mo_bits), pos_lo, pos_hi, P64(d_positions), m, S(stream));
}

int debwt_dev_scan_popc(const void* d_mo_bits, void* d_word_prefix, uint64_t nbw, uint64_t* total, void* d_workspace,
                        void* stream) {
    cudaStream_t st = S(stream);
    char* ws = reinterpret_cast<char*>(d_workspace);
    u64* d_tot = reinterpret_cast<u64*>(ws);
    if (scan_exclusive_u32(P32(d_mo_bits), P32(d_word_prefix), nbw, true, ws + 64, d_tot, st)) return -1;
    u64 h = 0;
    CUDA_TRY(cudaMemcpyAsync(&h, d_tot, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *total = h;
    return 0;
}

int debwt_dev_emit_codes_slice(const void* d_words, uint64_t word_lo, uint64_t nbw, const void* d_mo_bits,
                               const void* d_word_prefix, uint64_t code_base, void* d_codes, void* stream) {
    return k_emit_codes(P64(d_words), word_lo, nbw, P32(d_mo_bits), P32(d_word_prefix), code_base, P64(d_codes), S(stream));
}

int debwt_dev_mark_sep_slice(const void* d_mo_bits, const void* d_word_prefix, uint64_t pos_lo, uint64_t pos_hi,
                             uint64_t code_base, const void* d_positions, uint64_t m, void* d_sep, void* d_out_idx,
                             void* stream) {
    return k_mark_sep_codes(P32(d_mo_bits), P32(d_word_prefix), pos_lo, pos_hi, code_base, P64(d_positions), m, P32(d_sep),
                            P64(d_out_idx), S(stream));
}

int debwt_dev_fix_records(void* d_rec_entry, uint64_t m, const void* d_mo_bits, const void* d_word_prefix, uint64_t pos_lo,
                          uint64_t code_base, void* stream) {
    return k_blue_fix(P64(d_rec_entry), m, P32(d_mo_bits), P32(d_word_prefix), pos_lo, code_base, S(stream));
}

int debwt_dev_scatter_blue(const void* d_rec_entry, const void* d_rec_local, uint64_t m, const void* d_kmer,
                           const void* d_blue_u32, void* d_cursor_u32, uint64_t n_branch, void* d_blue, void* stream) {
    BranchTable bt = BT(d_kmer, nullptr, d_blue_u32, d_cursor_u32, nullptr, 0, n_branch, 0);
    return k_scatter_blue(P64(d_rec_entry), P64(d_rec_local), m, bt, P64(d_blue), S(stream));
}

int debwt_dev_sort_blue(void* d_blue, const void* d_kmer, const void* d_blue_u32, uint64_t n_branch, uint64_t n_blue,
                        const void* d_codes, const void* d_sep, uint64_t dollar_index, uint64_t n_codes, void* d_work_u32,
                        void* stream) {
    BranchTable bt = BT(d_kmer, nullptr, d_blue_u32, nullptr, nullptr, 0, n_branch, n_blue);
    SpView sp{P64(d_codes), P32(d_sep), dollar_index, n_codes};
    return k_sort_blue(P64(d_blue), bt, sp, P32(d_work_u32), S(stream));
}

int debwt_dev_fill_range(const void* d_gmask, uint64_t n_keys, uint64_t key_base, uint64_t n_symbols,
                         const void* d_spec_rows, uint64_t m, uint64_t word_lo, uint64_t word_hi, void* d_bwt, void* stream) {
    return k_fill_case2(P16(d_gmask), n_keys, key_base, n_symbols, P64(d_spec_rows), m, word_lo, word_hi, P64(d_bwt), S(stream));
}

int debwt_dev_emit_blue(const void* d_blue, const void* d_kmer, const void* d_head_u32, const void* d_blue_u32,
                        uint64_t n_branch, uint64_t n_blue, uint64_t key_base, const void* d_spec_ins, uint64_t m,
                        void* d_bwt, void* d_sharp_rows, void* d_sharp_count_u32, void* d_dollar_row, void* stream) {
    BranchTable bt = BT(d_kmer, d_head_u32, d_blue_u32, nullptr, nullptr, 0, n_branch, n_blue);
    return k_emit_blue(P64(d_blue), bt, key_base, P64(d_spec_ins), m, P64(d_bwt), P64(d_sharp_rows), P32(d_sharp_count_u32),
                       P64(d_dollar_row), S(stream));
}

int debwt_dev_emit_special(const void* d_spec_rows, const void* d_spec_chr, uint64_t m, void* d_bwt, void* stream) {
    return k_emit_special(P64(d_spec_rows), P8(d_spec_chr), m, P64(d_bwt), S(stream));
}

}  // extern "C"
