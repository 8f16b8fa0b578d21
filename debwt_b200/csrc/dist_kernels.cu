// Stages that only the sharded (multi-GPU) build runs -- SURVEY.md section 8e / K12.
//
// The reference has no distributed code; this is new.  The text is split by position into G 32-aligned
// slices, keys are range-partitioned by sampled splitters on k-mer boundaries and exchanged once
// (all-to-all over NVLink), after which every device owns a contiguous key range = a contiguous run of
// BWT rows.  This file holds the owner of an item, the bucket-by-owner partition and the peer-store
// exchange, the in-edge queries that cross key ranges, the K9 flagging of a position slice against the
// global branch table and the scatter of received blue entries into their segments.  The stages that
// both builds run live in stages.cu and take the slice or key range as parameters.
#include "dist_kernels.cuh"

#include "stages_dev.cuh"

namespace debwt {

namespace {

constexpr int TPB = 256;
inline unsigned grid_for(u64 work, int per_block) { return (unsigned)((work + per_block - 1) / per_block); }

// ---- K12 bucket by owner ----------------------------------------------------------------------
// owner of an item = number of splitters <= (item & mask); ~0 items are dropped (dest 255)
__global__ void __launch_bounds__(TPB) owner_of_keys_kernel(const u64* __restrict__ items, u64 n,
                                                           const u64* __restrict__ splitters, u32 n_split, u64 mask,
                                                           bool drop_marker, u8* __restrict__ dest) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;
    const u64 v = items[i];
    if (drop_marker && v == ~0ull) { dest[i] = 255; return; }
    dest[i] = (u8)upper_bound_u64(splitters, 0, n_split, v & mask);
}

// owner of a global table index = last rank whose base is <= index (bases: G+1 ascending values)
__global__ void __launch_bounds__(TPB) owner_of_index_kernel(u64* __restrict__ idx, u64 n, const u64* __restrict__ bases,
                                                            u32 n_ranks, u8* __restrict__ dest) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;
    const u64 g = idx[i];
    const u32 r = (u32)upper_bound_u64(bases, 0, n_ranks, g) - 1u;
    dest[i] = (u8)r;
    idx[i] = g - bases[r];                          // index local to the owner
}

constexpr int PART_ITEMS = 8;
constexpr int PART_TILE = TPB * PART_ITEMS;
constexpr int MAX_RANKS = 16;

// Owner of an item: from a precomputed byte array, or on the fly from the splitters.
struct OwnerFn {
    const u8* dest;            // non-null: precomputed owners
    const u64* splitters;      // else: owner = number of splitters <= (item & mask)
    u32 n_split;
    u64 mask;
    bool drop_marker;          // items equal to ~0 are dropped
    __device__ __forceinline__ u32 operator()(const u64* __restrict__ items, u64 i) const {
        if (dest) return dest[i];
        const u64 v = items[i];
        if (drop_marker && v == ~0ull) return 255u;
        u32 lo = 0;
        for (u32 sidx = 0; sidx < n_split; ++sidx) lo += (splitters[sidx] <= (v & mask)) ? 1u : 0u;   // <= 15 splitters
        return lo;
    }
};

// Warp-aggregated counting: one ballot per destination, lane g keeps the count of destination g.
__global__ void __launch_bounds__(TPB) partition_count_kernel(const u64* __restrict__ items, OwnerFn owner, u64 n, u32 n_ranks,
                                                             u64* __restrict__ counts) {
    __shared__ u32 s[MAX_RANKS];
    if (threadIdx.x < MAX_RANKS) s[threadIdx.x] = 0;
    __syncthreads();
    const u32 lane = threadIdx.x & 31;
    const u64 base = (u64)blockIdx.x * PART_TILE;
    u32 mine = 0;
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const u64 i = base + (u64)j * TPB + threadIdx.x;
        const u32 d = i < n ? owner(items, i) : 255u;
        for (u32 g = 0; g < n_ranks; ++g) {
            const u32 b = __ballot_sync(0xffffffffu, d == g);
            if (lane == g) mine += __popc(b);
        }
    }
    if (lane < n_ranks && mine) atomicAdd(&s[lane], mine);
    __syncthreads();
    if (threadIdx.x < n_ranks && s[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (u64)s[threadIdx.x]);
}

// cursors[d] starts at the exclusive prefix of counts; every block reserves one chunk per owner and keeps
// the items of one (block, owner) pair in their original order
__global__ void __launch_bounds__(TPB) partition_scatter_kernel(const u64* __restrict__ a, const u64* __restrict__ b,
                                                               OwnerFn owner, u64 n, u32 n_ranks,
                                                               u64* __restrict__ cursors, u64* __restrict__ out_a,
                                                               u64* __restrict__ out_b) {
    constexpr int NW = TPB / 32;
    __shared__ u32 s_wcnt[NW][MAX_RANKS];
    __shared__ u64 s_base[MAX_RANKS];
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 lt = lanemask_lt();
    const u64 base = (u64)blockIdx.x * PART_TILE;
    u8 dd[PART_ITEMS];
    u32 mine = 0;
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const u64 i = base + (u64)j * TPB + threadIdx.x;
        const u32 d = i < n ? owner(a, i) : 255u;
        dd[j] = (u8)d;
        for (u32 g = 0; g < n_ranks; ++g) {
            const u32 bal = __ballot_sync(0xffffffffu, d == g);
            if (lane == g) mine += __popc(bal);
        }
    }
    if (lane < MAX_RANKS) s_wcnt[warp][lane] = lane < n_ranks ? mine : 0;
    __syncthreads();
    if (threadIdx.x < n_ranks) {
        u32 run = 0;
        for (int w = 0; w < NW; ++w) { const u32 c = s_wcnt[w][threadIdx.x]; s_wcnt[w][threadIdx.x] = run; run += c; }
        s_base[threadIdx.x] = run ? atomicAdd(&cursors[threadIdx.x], (u64)run) : 0;
    }
    __syncthreads();
    u32 run = lane < n_ranks ? s_wcnt[warp][lane] : 0;      // lane g: next free slot of destination g inside this block
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const u64 i = base + (u64)j * TPB + threadIdx.x;
        const u32 d = dd[j];
        u32 rank = 0, add = 0;
        for (u32 g = 0; g < n_ranks; ++g) {
            const u32 bal = __ballot_sync(0xffffffffu, d == g);
            if (d == g) rank = __popc(bal & lt);
            if (lane == g) add = __popc(bal);
        }
        const u32 start = __shfl_sync(0xffffffffu, run, d < n_ranks ? d : 0);
        if (d < n_ranks) {
            const u64 o = s_base[d] + start + rank;
            out_a[o] = a[i];
            if (b) out_b[o] = b[i];
        }
        run += add;
    }
}

// Fused bucket + exchange: the ordering of partition_scatter_kernel, but every destination has its own base pointer --
// the receive buffer of that rank, mapped into this process (CUDA IPC or peer access) -- so the keys cross NVLink as peer
// stores straight from the partition kernel: no staging buffer in global memory, no separate all-to-all.  dst.ptr[d]
// already points at this rank's slot inside rank d's buffer.
struct PeerDst {
    u64* ptr[MAX_RANKS];
};

// The block's tile is first reordered by destination in shared memory: consecutive threads then store consecutive items
// of one destination's run, so every peer store of a warp is one contiguous 256-byte run instead of G short ones (the
// stores straight from registers, 32-64 bytes per destination and warp row, reached only a fifth of the NVLink bandwidth
// on the 3.1 Gbp build; profiles/r01_c3_3p1gbp_8gpu.log).
// Blocks visit the tiles in a strided order (tile = block * stride mod grid, stride coprime with the grid): when the
// input is sorted -- the in-edge queries are -- consecutive tiles all go to the same owner, every rank walks the owners
// in the same order, and all ranks would store into ONE rank's memory at a time (incast on a single NVLink port: the
// query exchange took twice as long as the key exchange for the same volume, profiles/r02_c3_8gpu_phases.md).
__global__ void __launch_bounds__(TPB) partition_scatter_p2p_staged_kernel(const u64* __restrict__ a, OwnerFn owner, u64 n,
                                                                          u32 n_ranks, u64* __restrict__ cursors, PeerDst dst,
                                                                          u32 stride) {
    constexpr int NW = TPB / 32;
    __shared__ u32 s_wcnt[NW][MAX_RANKS];
    __shared__ u64 s_base[MAX_RANKS];
    __shared__ u32 s_off[MAX_RANKS + 1];
    __shared__ u64 s_items[PART_TILE];
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 lt = lanemask_lt();
    const u64 base = (((u64)blockIdx.x * stride) % gridDim.x) * PART_TILE;
    u8 dd[PART_ITEMS];
    u64 vv[PART_ITEMS];
    u32 mine = 0;
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const u64 i = base + (u64)j * TPB + threadIdx.x;
        const u32 d = i < n ? owner(a, i) : 255u;
        vv[j] = i < n ? a[i] : 0;
        dd[j] = (u8)d;
        for (u32 g = 0; g < n_ranks; ++g) {
            const u32 bal = __ballot_sync(0xffffffffu, d == g);
            if (lane == g) mine += __popc(bal);
        }
    }
    if (lane < MAX_RANKS) s_wcnt[warp][lane] = lane < n_ranks ? mine : 0;
    __syncthreads();
    if (threadIdx.x < n_ranks) {
        u32 run = 0;
        for (int w = 0; w < NW; ++w) { const u32 c = s_wcnt[w][threadIdx.x]; s_wcnt[w][threadIdx.x] = run; run += c; }
        s_base[threadIdx.x] = run ? atomicAdd(&cursors[threadIdx.x], (u64)run) : 0;
        s_off[threadIdx.x + 1] = run;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 run = 0;
        s_off[0] = 0;
        for (u32 g = 0; g < n_ranks; ++g) { const u32 c = s_off[g + 1]; s_off[g + 1] = run + c; run += c; }
    }
    __syncthreads();
    u32 run = lane < n_ranks ? s_wcnt[warp][lane] : 0;
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const u32 d = dd[j];
        u32 rank = 0, add = 0;
        for (u32 g = 0; g < n_ranks; ++g) {
            const u32 bal = __ballot_sync(0xffffffffu, d == g);
            if (d == g) rank = __popc(bal & lt);
            if (lane == g) add = __popc(bal);
        }
        const u32 start = __shfl_sync(0xffffffffu, run, d < n_ranks ? d : 0);
        if (d < n_ranks) s_items[s_off[d] + start + rank] = vv[j];
        run += add;
    }
    __syncthreads();
    const u32 total = s_off[n_ranks];
    for (u32 p = threadIdx.x; p < total; p += TPB) {
        u32 d = 0;
        while (s_off[d + 1] <= p) ++d;
        dst.ptr[d][s_base[d] + (p - s_off[d])] = s_items[p];
    }
}

// ---- K5/K6 split into a local half and an exchanged half --------------------------------------
__global__ void __launch_bounds__(TPB) out_edges_queries_kernel(const u64* __restrict__ k, u64 n, u16* __restrict__ gmask,
                                                               u64* __restrict__ queries) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;
    const u64 key = k[i];
    if (i > 0 && k[i - 1] == key) { queries[i] = ~0ull; return; }   // one representative per distinct (k+1)-mer
    atomic_or_u16(gmask, group_head(k, i), 1u << (GM_OUT_SHIFT + (u32)(key & 3)));
    // in-edge query for the owner of the suffix k-mer X of cX: (X << 2) | c.  X = T..T with c = T would
    // collide with the drop marker, but ~0 << 2 | 3 == ~0 only when the key itself is ~0 (poly-T), whose
    // suffix k-mer is its own prefix k-mer: mark it here.
    const u64 q = (key << 2) | (key >> 62);
    if (q == ~0ull) { atomic_or_u16(gmask, group_head(k, i), 1u << 3); queries[i] = ~0ull; return; }
    queries[i] = q;
}

__global__ void __launch_bounds__(TPB) apply_in_queries_kernel(const u64* __restrict__ k, u64 n, KeyIndex ki,
                                                              u16* __restrict__ gmask, const u64* __restrict__ q, u64 m) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= m) return;
    const u64 x = q[t] & ~3ull;
    const u64 hs = indexed_lower_bound(k, ki, x);
    if (hs < n && (k[hs] & ~3ull) == x) atomic_or_u16(gmask, hs, 1u << (u32)(q[t] & 3ull));
}

// ---- K9 on a position slice -------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) flag_slice_kernel(const u64* __restrict__ words, u64 pos_lo, u64 pos_hi,
                                                        const u64* __restrict__ seps, u64 n_rec, BranchTable bt,
                                                        u32* __restrict__ mo_bits, u64* __restrict__ rec_entry,
                                                        u64* __restrict__ rec_index, u64* __restrict__ rec_count) {
    const u64 p = pos_lo + (u64)blockIdx.x * TPB + threadIdx.x;     // pos_lo is a multiple of 32
    bool mo = false, mi = false;
    u64 entry = 0, index = 0;
    if (p < pos_hi) {
        const u64 r = record_of(seps, n_rec, p);
        if (r < n_rec && p + KMER <= seps[r]) {
            const u64 x = text_window32(words, p) & ~3ull;
            u64 b;
            u32 f;
            if (branch_lookup(bt, x, b, f)) {
                mo = f & 1u;
                if (f & 2u) {
                    const u64 start = r ? seps[r - 1] + 1 : 0;
                    u32 prev;
                    if (p == start) prev = r ? 4u : 5u;
                    else prev = text_symbol(words, p - 1);
                    mi = true;
                    entry = (p << 4) | prev;
                    index = b;                                       // index into the global branch table
                }
            }
        }
    }
    // warp-aggregated append: one atomic per warp instead of one per record
    const u32 lane = threadIdx.x & 31;
    const u32 bmi = __ballot_sync(0xffffffffu, mi);
    if (bmi) {
        u64 base = 0;
        if (lane == (u32)(__ffs(bmi) - 1)) base = atomicAdd(rec_count, (u64)__popc(bmi));
        base = __shfl_sync(0xffffffffu, base, __ffs(bmi) - 1);
        if (mi) {
            const u64 slot = base + __popc(bmi & lanemask_lt());
            rec_entry[slot] = entry;
            rec_index[slot] = index;
        }
    }
    const u32 bal = __ballot_sync(0xffffffffu, mo);
    if (lane == 0) mo_bits[(p - pos_lo) >> 5] = bal;
}

__global__ void __launch_bounds__(TPB) scatter_blue_kernel(const u64* __restrict__ rec_entry, const u64* __restrict__ rec_local,
                                                          u64 m, BranchTable bt, u64* __restrict__ blue) {
    const u64 e = (u64)blockIdx.x * TPB + threadIdx.x;
    if (e >= m) return;
    const u64 b = rec_local[e];
    const u32 slot = atomicAdd(bt.cursor + b, 1u);
    blue[(u64)bt.blue[b] + slot] = rec_entry[e];
}

}  // namespace

#define LAUNCHED(k)                      \
    do {                                 \
        DEBWT_COUNT(k);                  \
        CUDA_TRY(cudaGetLastError());    \
        return 0;                        \
    } while (0)

int k_owner_of_keys(const u64* items, u64 n, const u64* d_splitters, u32 n_split, u64 mask, bool drop_marker, u8* dest,
                    cudaStream_t st) {
    if (n == 0) return 0;
    owner_of_keys_kernel<<<grid_for(n, TPB), TPB, 0, st>>>(items, n, d_splitters, n_split, mask, drop_marker, dest);
    LAUNCHED(1);
}

int k_owner_of_index(u64* idx, u64 n, const u64* d_bases, u32 n_ranks, u8* dest, cudaStream_t st) {
    if (n == 0) return 0;
    owner_of_index_kernel<<<grid_for(n, TPB), TPB, 0, st>>>(idx, n, d_bases, n_ranks, dest);
    LAUNCHED(1);
}

namespace {
OwnerFn make_owner(const PartitionBy& by) {
    OwnerFn f;
    f.dest = by.dest; f.splitters = by.splitters; f.n_split = by.n_split; f.mask = by.mask; f.drop_marker = by.drop_marker;
    return f;
}
}  // namespace

int k_partition_count(const u64* items, const PartitionBy& by, u64 n, u32 n_ranks, u64* d_counts /* MAX_RANKS, zeroed */,
                      cudaStream_t st) {
    if (n == 0) return 0;
    partition_count_kernel<<<grid_for(n, PART_TILE), TPB, 0, st>>>(items, make_owner(by), n, n_ranks, d_counts);
    LAUNCHED(1);
}

int k_partition_scatter(const u64* a, const u64* b, const PartitionBy& by, u64 n, u32 n_ranks, u64* d_cursors, u64* out_a,
                        u64* out_b, cudaStream_t st) {
    if (n == 0) return 0;
    partition_scatter_kernel<<<grid_for(n, PART_TILE), TPB, 0, st>>>(a, b, make_owner(by), n, n_ranks, d_cursors, out_a, out_b);
    LAUNCHED(1);
}

int k_partition_scatter_p2p(const u64* a, const PartitionBy& by, u64 n, u32 n_ranks, u64* d_cursors /* zeroed */,
                            u64* const* dst, cudaStream_t st) {
    if (n == 0) return 0;
    PeerDst pd;
    for (u32 r = 0; r < MAX_RANKS; ++r) pd.ptr[r] = r < n_ranks ? dst[r] : nullptr;
    const unsigned grid = grid_for(n, PART_TILE);
    auto gcd = [](unsigned x, unsigned y) { while (y) { const unsigned t = x % y; x = y; y = t; } return x; };
    unsigned stride = (unsigned)(grid * 0.6180339887) | 1u;                // golden-ratio stride: neighbours in time are far apart in the input
    while (stride > 1 && gcd(stride, grid) != 1) stride -= 2;
    if (grid < 8) stride = 1;
    partition_scatter_p2p_staged_kernel<<<grid, TPB, 0, st>>>(a, make_owner(by), n, n_ranks, d_cursors, pd, stride);
    LAUNCHED(1);
}

int k_out_edges_queries(const u64* sorted, u64 n, u16* gmask, u64* queries, cudaStream_t st) {
    if (n == 0) return 0;
    out_edges_queries_kernel<<<grid_for(n, TPB), TPB, 0, st>>>(sorted, n, gmask, queries);
    LAUNCHED(1);
}

int k_apply_in_queries(const u64* sorted, u64 n, KeyIndex ki, u16* gmask, const u64* q, u64 m, cudaStream_t st) {
    if (m == 0) return 0;
    apply_in_queries_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(sorted, n, ki, gmask, q, m);
    LAUNCHED(1);
}

int k_flag_slice(const u64* words, u64 pos_lo, u64 pos_hi, const u64* d_seps, u64 n_rec, BranchTable bt, u32* mo_bits,
                 u64* rec_entry, u64* rec_index, u64* d_rec_count, cudaStream_t st) {
    if (pos_hi <= pos_lo) return 0;                  // mo_bits stays as the caller zeroed it
    const u64 npos = (pos_hi - pos_lo + 31) & ~31ull;
    flag_slice_kernel<<<grid_for(npos, TPB), TPB, 0, st>>>(words, pos_lo, pos_hi, d_seps, n_rec, bt, mo_bits, rec_entry,
                                                           rec_index, d_rec_count);
    LAUNCHED(1);
}

int k_scatter_blue(const u64* rec_entry, const u64* rec_local, u64 m, BranchTable bt, u64* blue, cudaStream_t st) {
    if (m == 0) return 0;
    scatter_blue_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(rec_entry, rec_local, m, bt, blue);
    LAUNCHED(1);
}

}  // namespace debwt
