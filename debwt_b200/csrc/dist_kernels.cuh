// Sharded (multi-GPU) stage launchers -- see dist_kernels.cu.
#pragma once
#include "stages.cuh"

namespace debwt {

int k_owner_of_keys(const u64* items, u64 n, const u64* d_splitters, u32 n_split, u64 mask, bool drop_marker, u8* dest,
                    cudaStream_t st);
int k_owner_of_index(u64* idx, u64 n, const u64* d_bases, u32 n_ranks, u8* dest, cudaStream_t st);
// how the owner of an item is found: a precomputed byte per item, or on the fly from the splitters
struct PartitionBy {
    const u8* dest = nullptr;
    const u64* splitters = nullptr;
    u32 n_split = 0;
    u64 mask = ~0ull;
    bool drop_marker = false;
};
int k_partition_count(const u64* items, const PartitionBy& by, u64 n, u32 n_ranks, u64* d_counts, cudaStream_t st);
int k_partition_scatter(const u64* a, const u64* b, const PartitionBy& by, u64 n, u32 n_ranks, u64* d_cursors, u64* out_a,
                        u64* out_b, cudaStream_t st);
// fused bucket + exchange: dst[r] = where this rank's items for rank r start (peer memory for r != own rank)
int k_partition_scatter_p2p(const u64* a, const PartitionBy& by, u64 n, u32 n_ranks, u64* d_cursors, u64* const* dst,
                            cudaStream_t st);
int k_out_edges_queries(const u64* sorted, u64 n, u16* gmask, u64* queries, cudaStream_t st);
int k_apply_in_queries(const u64* sorted, u64 n, KeyIndex ki, u16* gmask, const u64* q, u64 m, cudaStream_t st);
int k_flag_slice(const u64* words, u64 pos_lo, u64 pos_hi, const u64* d_seps, u64 n_rec, BranchTable bt, u32* mo_bits,
                 u64* rec_entry, u64* rec_index, u64* d_rec_count, cudaStream_t st);
int k_scatter_blue(const u64* rec_entry, const u64* rec_local, u64 m, BranchTable bt, u64* blue, cudaStream_t st);

}  // namespace debwt
