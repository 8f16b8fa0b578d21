// The sharded (multi-GPU) build behind the C ABI: one rank per GPU, SPMD -- SURVEY.md section 8e / K12.
//
// The reference has no distributed code; this is the B200 design (DESIGN.md section 6).  A rank is either a process
// (torchrun starts one per GPU: peer buffers are mapped through CUDA IPC) or a thread of one process
// (debwt_build_multi / host/deBWT -g 0,1,...: peer access, plain pointers).  Control data -- counts, handles, splitter
// samples -- travels through a shared-memory communicator (shmcomm.h); every byte of the data path is moved GPU to GPU
// over NVLink by our own kernels and peer copies:
//   1. the text is cut into G 32-aligned position slices; every rank packs its slice and stores it into every peer's copy
//      of the packed text (N/4 bytes, needed everywhere for sentinel windows and branch codes);
//   2. sampled splitters on k-mer boundaries; keys are bucketed and stored straight into their owner's receive buffer
//      (partition_scatter_p2p_staged_kernel: the exchange IS the bucketing kernel); every rank then owns a contiguous key
//      range = a contiguous run of BWT rows, and sorts / classifies it locally;
//   3. in-edges cX -> X travel as a second exchange of queries; branch tables are gathered; branch codes are produced per
//      position slice at global code indices and OR-ed together; blue entries travel to the owner of their k-mer;
//   4. every rank emits its own contiguous BWT segment and stores it into rank 0's result buffer (the one word shared with
//      a neighbour is OR-ed).
// Same kernels as debwt_b200/dist.py (which stays as the CPU-testable harness of this orchestration).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <string>
#include <thread>
#include <vector>

#include "../../include/debwt_b200.h"
#include "ctx.cuh"
#include "dist_kernels.cuh"
#include "radix_sort.cuh"
#include "shmcomm.h"
#include "special.cuh"
#include "stages_dev.cuh"

namespace debwt {

int build_special_tables(const SpecialInfo* info, const u64* seps, u64 R, std::vector<u64>& ins, std::vector<u64>& rows,
                         std::vector<u8>& chr, std::vector<u64>& emit_pos, std::vector<u64>& tail_pos);      // api.cu

namespace {

constexpr int kMaxRanks = 16;
constexpr u64 kSamplesPerRank = 4096;
constexpr u64 kKmerMask = 0xFFFFFFFFFFFFFFFCull;

// a device allocation every rank can address: ptr[r] = rank r's buffer as seen from this rank
struct SharedBuf {
    void* ptr[kMaxRanks] = {};
    size_t cap = 0;                 // of this rank's buffer
    bool mapped = false;
};

__global__ void sample_kernel(const u64* __restrict__ keys, u64 stride, u64 ns, u64* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ns) out[i] = keys[i * stride];
}

// dst[w] |= src[w]: the first and the last word may be shared with another writer
__global__ void or_store_kernel(u64* __restrict__ dst, const u64* __restrict__ src, u64 n) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 v = src[i];
    if (i == 0 || i + 1 == n) { if (v) atomicOr(reinterpret_cast<unsigned long long*>(dst + i), (unsigned long long)v); }
    else dst[i] = v;
}

// copies between ranks are done by the SMs (16-byte loads / stores through the peer mapping, over NVLink): a cudaMemcpy
// between two processes' IPC-mapped buffers may be staged through the host
__global__ void __launch_bounds__(512) peer_copy_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src, u64 n16,
                                                       u8* __restrict__ dst_tail, const u8* __restrict__ src_tail, u32 tail) {
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) dst[i] = src[i];
    if (blockIdx.x == 0 && threadIdx.x < tail) dst_tail[threadIdx.x] = src_tail[threadIdx.x];
}

template <typename T>
__global__ void or_range_kernel(T* __restrict__ dst, const T* __restrict__ src, u64 lo, u64 hi) {
    const u64 i = lo + (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < hi) { const T v = src[i]; if (v) dst[i] |= v; }
}

inline unsigned blocks(u64 n, unsigned tpb = 256) { return (unsigned)((n + tpb - 1) / tpb); }

}  // namespace
}  // namespace debwt

using namespace debwt;

struct debwt_shard {
    int device = 0, rank = 0, world = 1;
    bool same_process = false;
    int sort_cfg = kDefaultSortCfg;
    cudaStream_t st = nullptr;
    ShmComm comm;
    DevPool pool;
    int peer_device[kMaxRanks] = {};
    SharedBuf words, recv_a, recv_b, gkmer, share, out, mail;
    cudaEvent_t ev[8] = {};
    // result (rank 0)
    u64 n = 0, n_rec = 0;
    std::vector<u64> sharp;
    u64 dollar = ~0ull;
    bool built = false;
    debwt_shard_stats stats{};
    std::string err;
};

namespace {

#define SFAIL(msg)                                 \
    do {                                           \
        s->err = (msg);                            \
        debwt::set_error(s->err);                  \
        return -1;                                 \
    } while (0)
#define SCUDA(expr)                                                                              \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            char _b[512];                                                                        \
            snprintf(_b, sizeof _b, "rank %d: %s:%d: %s -> %s", s->rank, __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            s->err = _b;                                                                         \
            debwt::set_error(s->err);                                                            \
            return -1;                                                                           \
        }                                                                                        \
    } while (0)
int barrier(debwt_shard* s) {
    std::string e;
    if (s->comm.barrier(&e)) SFAIL("rank " + std::to_string(s->rank) + ": " + e);
    return 0;
}

template <typename T>
int allgather(debwt_shard* s, const T* mine, size_t count, T* all) {
    std::string e;
    if (s->comm.allgather(mine, count * sizeof(T), all, &e)) SFAIL("rank " + std::to_string(s->rank) + ": " + e);
    return 0;
}

// device-side completion of everything this rank queued, then a barrier: afterwards every peer's stores have landed
int sync_all(debwt_shard* s) {
    SCUDA(cudaStreamSynchronize(s->st));
    return barrier(s);
}

// dst (possibly another rank's memory) <- src (this rank's), both 8-byte aligned
int peer_copy(debwt_shard* s, void* dst, const void* src, size_t bytes) {
    if (bytes == 0) return 0;
    if ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15) {      // 8-byte aligned only: plain words
        SCUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s->st));
        return 0;
    }
    const u64 n16 = bytes / 16;
    const u32 tail = (u32)(bytes % 16);
    unsigned grid = (unsigned)std::min<u64>((n16 + 511) / 512, 148ull * 8);
    if (grid == 0) grid = 1;
    peer_copy_kernel<<<grid, 512, 0, s->st>>>(static_cast<uint4*>(dst), static_cast<const uint4*>(src), n16,
                                              static_cast<u8*>(dst) + n16 * 16, static_cast<const u8*>(src) + n16 * 16, tail);
    DEBWT_COUNT(1);
    SCUDA(cudaGetLastError());
    return 0;
}

void unmap(debwt_shard* s, SharedBuf& b) {
    if (!b.mapped) return;
    for (int r = 0; r < s->world; ++r) {
        if (r == s->rank || !b.ptr[r]) continue;
        if (!s->same_process) cudaIpcCloseMemHandle(b.ptr[r]);
        b.ptr[r] = nullptr;
    }
    b.mapped = false;
}

// Collective: every rank needs `need` bytes of its own (sizes may differ).  Grows (never shrinks) and re-maps when any
// rank has to grow.
int ensure_shared(debwt_shard* s, SharedBuf& b, size_t need) {
    struct Q { u64 need, cap; } mine{(u64)need, (u64)b.cap}, all[kMaxRanks];
    if (allgather(s, &mine, 1, all)) return -1;
    bool grow = !b.mapped;
    for (int r = 0; r < s->world; ++r) grow = grow || all[r].need > all[r].cap;
    if (!grow) return 0;
    SCUDA(cudaStreamSynchronize(s->st));
    if (barrier(s)) return -1;                       // nobody is still using the old mappings
    unmap(s, b);
    if (need > b.cap || !b.ptr[s->rank]) {
        if (b.ptr[s->rank]) SCUDA(cudaFree(b.ptr[s->rank]));
        b.ptr[s->rank] = nullptr;
        size_t cap = need + need / 8 + 4096;
        cap = (cap + 511) & ~(size_t)511;
        SCUDA(cudaMalloc(&b.ptr[s->rank], cap));
        b.cap = cap;
    }
    if (s->world > 1) {
        if (s->same_process) {
            u64 p = reinterpret_cast<u64>(b.ptr[s->rank]), ps[kMaxRanks];
            if (allgather(s, &p, 1, ps)) return -1;
            for (int r = 0; r < s->world; ++r) b.ptr[r] = reinterpret_cast<void*>(ps[r]);
        } else {
            cudaIpcMemHandle_t h, hs[kMaxRanks];
            SCUDA(cudaIpcGetMemHandle(&h, b.ptr[s->rank]));
            if (allgather(s, &h, 1, hs)) return -1;
            for (int r = 0; r < s->world; ++r) {
                if (r == s->rank) continue;
                SCUDA(cudaIpcOpenMemHandle(&b.ptr[r], hs[r], cudaIpcMemLazyEnablePeerAccess));
            }
        }
    }
    b.mapped = true;
    return 0;
}

template <typename T>
int dalloc(debwt_shard* s, T** p, size_t count) {
    if (s->pool.alloc(reinterpret_cast<void**>(p), count * sizeof(T))) { s->err = "out of device memory"; return -1; }
    return 0;
}

u64 windows_before(u64 x, const u64* seps, u64 R) {             // in-record 32-mer windows that start at a position < x
    u64 total = 0, start = 0;
    for (u64 r = 0; r < R; ++r) {
        const u64 last = seps[r] - 32;                          // last valid start of the record (records are > 32 bp)
        const u64 end = last + 1 < x ? last + 1 : x;
        if (end > start) total += end - start;
        start = seps[r] + 1;
        if (start >= x) break;
    }
    return total;
}

// one exchange of 64-bit items to the owners of their k-mers: bucketing kernel == exchange (peer stores)
int exchange_by_splitters(debwt_shard* s, const u64* items, u64 n_items, const u64* d_split, bool drop_marker, SharedBuf& recv,
                          u64* d_small /* 32 u64 */, u64* n_recv_out, u64* n_from_all /* [world] or null */) {
    const int G = s->world, me = s->rank;
    PartitionBy by;
    by.splitters = d_split; by.n_split = (u32)(G - 1); by.mask = kKmerMask; by.drop_marker = drop_marker;
    u64 counts[kMaxRanks] = {}, mat[kMaxRanks * kMaxRanks];
    SCUDA(cudaMemsetAsync(d_small, 0, 32 * 8, s->st));
    if (k_partition_count(items, by, n_items, (u32)G, d_small, s->st)) return -1;
    SCUDA(cudaMemcpyAsync(counts, d_small, kMaxRanks * 8, cudaMemcpyDeviceToHost, s->st));
    SCUDA(cudaStreamSynchronize(s->st));
    if (allgather(s, counts, kMaxRanks, mat)) return -1;                       // mat[src * 16 + dst]
    u64 col = 0;
    for (int src = 0; src < G; ++src) col += mat[src * kMaxRanks + me];
    if (ensure_shared(s, recv, (col + 2) * 8)) return -1;
    u64* dst[kMaxRanks] = {};
    for (int d = 0; d < G; ++d) {
        u64 off = 0;
        for (int src = 0; src < me; ++src) off += mat[src * kMaxRanks + d];
        dst[d] = static_cast<u64*>(recv.ptr[d]) + off;
    }
    if (k_partition_scatter_p2p(items, by, n_items, (u32)G, d_small + 16, dst, s->st)) return -1;
    if (sync_all(s)) return -1;                                                // every peer has finished storing into this rank's buffer
    *n_recv_out = col;
    if (n_from_all)
        for (int d = 0; d < G; ++d) {
            u64 c = 0;
            for (int src = 0; src < G; ++src) c += mat[src * kMaxRanks + d];
            n_from_all[d] = c;
        }
    return 0;
}

struct PhaseClock {                                    // DEBWT_SHARD_PROFILE=1: synchronised per-phase wall times on stderr (rank 0)
    bool on;
    cudaStream_t st;
    double t;
    std::string out;
    static double now() { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; }
    void tick(const char* name) {
        if (!on) return;
        cudaStreamSynchronize(st);
        const double n = now();
        char b[64];
        snprintf(b, sizeof b, " %s %.1f", name, (n - t) * 1e3);
        out += b;
        t = n;
    }
};

int shard_build_impl(debwt_shard* s, const void* slice, int slice_on_device, u64 N, const u64* seps, u64 R) {
    const int G = s->world, me = s->rank;
    cudaStream_t st = s->st;
    PhaseClock pc{getenv("DEBWT_SHARD_PROFILE") != nullptr, st, PhaseClock::now(), ""};
    DevPool& pool = s->pool;
    SCUDA(cudaSetDevice(s->device));
    if (R == 0) SFAIL("no records");
    {
        u64 start = 0;
        for (u64 r = 0; r < R; ++r) {
            if (seps[r] < start || seps[r] - start <= 32) SFAIL("Length <= 32!");      // src/collect#$.c:41-45
            start = seps[r] + 1;
        }
        if (start != N) SFAIL("last separator must be the last symbol");
    }
    pool.release_all();
    s->built = false;
    debwt_shard_stats& S = s->stats;
    S = debwt_shard_stats{};
    const u64 NK = N - 32 * R;
    const u64 n_words = (N + 32 + 31) / 32 + 1;
    const u64 wp = (n_words + G - 1) / G, wtot = wp * G;
    const u64 pos_lo = 32 * (u64)me * wp, pos_hi_al = 32 * (u64)(me + 1) * wp;
    const u64 pos_hi = std::max(std::min(pos_hi_al, N), pos_lo);
    const u64 n_valid = pos_hi - pos_lo;
    S.n_symbols = N; S.n_records = R; S.n_keys = NK;
    pool.hint((NK / G + (1u << 20)) * 30 + wtot * 8 + (512ull << 20));
    SCUDA(cudaEventRecord(s->ev[0], st));

    // ---- small persistent allocations first (the big temporaries are bump-allocated after them and rewound) ----
    u64 *d_seps = nullptr, *d_small = nullptr, *d_split = nullptr, *d_samples = nullptr;
    u32* d_err = nullptr;
    if (dalloc(s, &d_seps, R) || dalloc(s, &d_small, 64) || dalloc(s, &d_split, kMaxRanks) || dalloc(s, &d_samples, kSamplesPerRank) ||
        dalloc(s, &d_err, 4))
        return -1;
    SCUDA(cudaMemcpyAsync(d_seps, seps, R * 8, cudaMemcpyHostToDevice, st));
    SCUDA(cudaMemsetAsync(d_err, 0, 16, st));

    // ---- 1. pack own slice into the shared packed text, store it into every peer's copy ----
    if (ensure_shared(s, s->words, (wtot + 2) * 8)) return -1;
    u64* W = static_cast<u64*>(s->words.ptr[me]);
    {
        const auto mark = pool.mark();
        const u8* d_ascii = static_cast<const u8*>(slice);
        if (!slice_on_device) {
            u8* tmp = nullptr;
            if (dalloc(s, &tmp, n_valid + 64)) return -1;
            if (n_valid) SCUDA(cudaMemcpyAsync(tmp, slice, n_valid, cudaMemcpyHostToDevice, st));
            d_ascii = tmp;
        }
        if (k_pack_words(d_ascii, n_valid, W + (u64)me * wp, wp, d_err, st)) return -1;
        SCUDA(cudaMemsetAsync(W + wtot, 0, 16, st));
        for (int p = 0; p < G; ++p)
            if (p != me)
                if (peer_copy(s, static_cast<u64*>(s->words.ptr[p]) + (u64)me * wp, W + (u64)me * wp, wp * 8)) return -1;
        u32 h_err[4] = {0, 0, 0, 0}, all_err[kMaxRanks * 4];
        SCUDA(cudaMemcpyAsync(h_err, d_err, 16, cudaMemcpyDeviceToHost, st));
        if (sync_all(s)) return -1;
        pool.rewind(mark);
        if (allgather(s, h_err, 4, all_err)) return -1;
        u64 nsep = 0;
        for (int p = 0; p < G; ++p) {
            if (all_err[p * 4]) SFAIL("input contains a symbol other than A, C, G, T (either case)");
            nsep += all_err[p * 4 + 1];
        }
        if (nsep != R) SFAIL("input contains '#' or '$' inside a record (they are reserved for the record separators)");
    }
    pc.tick("pack+gather");
    SCUDA(cudaEventRecord(s->ev[1], st));

    // ---- 2. keys of own slice, sampled splitters ----
    const u64 idx_base = windows_before(pos_lo, seps, R);
    const u64 cnt = n_valid ? windows_before(pos_hi, seps, R) - idx_base : 0;
    u64 n_loc = 0, n_all[kMaxRanks] = {};
    {
        const auto mark = pool.mark();
        u64* keys = nullptr;
        if (dalloc(s, &keys, cnt + 2)) return -1;
        if (cnt && k_extract_slice(W, N, pos_lo, pos_hi, d_seps, R, idx_base, keys, st)) return -1;
        const u64 ns = std::min(cnt, kSamplesPerRank);
        std::vector<u64> h_samp(kSamplesPerRank + 1, ~0ull), all_samp((kSamplesPerRank + 1) * G);
        if (ns) {
            sample_kernel<<<blocks(ns), 256, 0, st>>>(keys, std::max<u64>(cnt / ns, 1), ns, d_samples);
            DEBWT_COUNT(1);
            SCUDA(cudaMemcpyAsync(h_samp.data(), d_samples, ns * 8, cudaMemcpyDeviceToHost, st));
            SCUDA(cudaStreamSynchronize(st));
        }
        h_samp[kSamplesPerRank] = ns;
        if (allgather(s, h_samp.data(), kSamplesPerRank + 1, all_samp.data())) return -1;
        std::vector<u64> valid;
        for (int p = 0; p < G; ++p) {
            const u64* a = all_samp.data() + (size_t)p * (kSamplesPerRank + 1);
            valid.insert(valid.end(), a, a + a[kSamplesPerRank]);
        }
        std::sort(valid.begin(), valid.end());
        u64 h_split[kMaxRanks] = {};
        for (int i = 1; i < G; ++i)
            h_split[i - 1] = valid.empty() ? kKmerMask : (valid[(size_t)i * valid.size() / G] & kKmerMask);   // k-mer boundaries
        SCUDA(cudaMemcpyAsync(d_split, h_split, kMaxRanks * 8, cudaMemcpyHostToDevice, st));

        pc.tick("extract+splitters");
        // ---- 3. one exchange: every key goes to the owner of its k-mer ----
        if (exchange_by_splitters(s, keys, cnt, d_split, false, s->recv_a, d_small, &n_loc, n_all)) return -1;
        pool.rewind(mark);
    }
    u64 key_base = 0, total = 0;
    for (int p = 0; p < G; ++p) { if (p < me) key_base += n_all[p]; total += n_all[p]; }
    if (total != NK) SFAIL("internal: key exchange lost keys");
    if (n_loc >= (1ull << 32) - (1u << 16)) SFAIL("a rank owns 2^32 keys or more: use more GPUs");
    S.n_keys_local = n_loc;
    pc.tick("key_exchange");
    SCUDA(cudaEventRecord(s->ev[2], st));

    // ---- 4. sort the owned key range ----
    u64* sk = nullptr;
    {
        u64* tmp = nullptr;
        void* sortws = nullptr;
        if (dalloc(s, &tmp, n_loc + 2) || pool.alloc(&sortws, sort_workspace_bytes(n_loc, s->sort_cfg))) return -1;
        SortWorkspace ws;
        sort_workspace_bind(ws, sortws, n_loc, s->sort_cfg);
        int sweeps = 0;
        ws.ev_sweep_begin = s->ev[5]; ws.ev_sweep_end = s->ev[6]; ws.sweeps_out = &sweeps;
        if (radix_sort_u64(static_cast<u64*>(s->recv_a.ptr[me]), tmp, n_loc, ws, st, &sk)) return -1;
        S.sort_sweeps = (u32)sweeps;
        pool.adopt(sk == tmp ? nullptr : tmp, sk == tmp ? 0 : (n_loc + 2) * 8);      // the ping-pong half the sort did not end in
        pool.adopt(sortws, sort_workspace_bytes(n_loc, s->sort_cfg));
    }
    SCUDA(cudaEventRecord(s->ev[3], st));
    pc.tick("sort");

    // ---- 5. branch k-mer detection on the owned range ----
    KeyIndex ki;
    ki.bits = key_index_bits(n_loc);
    u16* gmask = nullptr;
    if (dalloc(s, &ki.idx, (1ull << ki.bits) + 2) || dalloc(s, &gmask, n_loc + 2)) return -1;
    SCUDA(cudaMemsetAsync(gmask, 0, (n_loc + 2) * 2, st));
    if (k_build_key_index(sk, n_loc, ki, st)) return -1;
    {
        const auto mark = pool.mark();
        u64* q = nullptr;
        if (dalloc(s, &q, n_loc + 2)) return -1;
        pc.tick("index");
        if (k_out_edges_queries(sk, n_loc, gmask, q, st)) return -1;
        pc.tick("out_edges");
        u64 m_q = 0;                                   // duplicates (marked ~0) are dropped on the way, also on one rank
        if (exchange_by_splitters(s, q, n_loc, d_split, true, s->recv_b, d_small, &m_q, nullptr)) return -1;
        const u64* qr = static_cast<const u64*>(s->recv_b.ptr[me]);
        pc.tick("query_exchange");
        if (n_loc) {
            if (k_apply_in_queries(sk, n_loc, ki, gmask, qr, m_q, st)) return -1;
            if (k_mark_heads_tails(W, d_seps, R, sk, n_loc, ki, gmask, st)) return -1;      // (the masks reach the other members of
        }                                                                                       //  their groups in k_branch_count)
        SCUDA(cudaStreamSynchronize(st));
        pool.rewind(mark);
        pc.tick("apply+propagate");
    }
    BranchTable bt;
    u64 b_base[kMaxRanks + 1] = {}, m_all[kMaxRanks] = {}, B_tot = 0, M_tot = 0;
    {
        void* brws = nullptr;
        u64* d_tot = d_small + 32;
        u64 h_tot[2] = {0, 0};
        if (n_loc) {
            if (pool.alloc(&brws, branch_workspace_bytes(n_loc))) return -1;
            if (k_branch_count(sk, n_loc, gmask, true, brws, d_tot, st)) return -1;
            SCUDA(cudaMemcpyAsync(h_tot, d_tot, 16, cudaMemcpyDeviceToHost, st));
            SCUDA(cudaStreamSynchronize(st));
        }
        bt.n_branch = h_tot[0]; bt.n_blue = h_tot[1];
        if (bt.n_blue >= 0xFFFFFFFFull) SFAIL("a rank owns 2^32 blue entries or more: use more GPUs");
        if (dalloc(s, &bt.kmer, bt.n_branch + 1) || dalloc(s, &bt.head, bt.n_branch + 1) || dalloc(s, &bt.blue, bt.n_branch + 2) ||
            dalloc(s, &bt.cursor, bt.n_branch + 1))
            return -1;
        SCUDA(cudaMemsetAsync(bt.blue, 0, (bt.n_branch + 2) * 4, st));
        if (n_loc && k_branch_write(sk, n_loc, gmask, brws, bt, st)) return -1;
        const u32 m32 = (u32)bt.n_blue;
        SCUDA(cudaMemcpyAsync(bt.blue + bt.n_branch, &m32, 4, cudaMemcpyHostToDevice, st));
        u64 mine[2] = {bt.n_branch, bt.n_blue}, all[kMaxRanks * 2];
        if (allgather(s, mine, 2, all)) return -1;
        for (int p = 0; p < G; ++p) { b_base[p + 1] = b_base[p] + all[p * 2]; m_all[p] = all[p * 2 + 1]; M_tot += m_all[p]; }
        B_tot = b_base[G];
    }
    // the global branch table: every rank stores its k-mers into every peer's copy
    if (ensure_shared(s, s->gkmer, (B_tot + 2) * 8)) return -1;
    for (int p = 0; p < G; ++p)
        if (bt.n_branch)
            if (peer_copy(s, static_cast<u64*>(s->gkmer.ptr[p]) + b_base[me], bt.kmer, bt.n_branch * 8)) return -1;
    if (sync_all(s)) return -1;
    BranchTable gbt;
    gbt.n_branch = B_tot; gbt.kmer = static_cast<u64*>(s->gkmer.ptr[me]);
    {
        int bits = 8;
        while (bits < 27 && (1ull << bits) < 2 * B_tot) ++bits;
        gbt.bits = bits;
        if (dalloc(s, &gbt.bidx, BranchTable::index_words(bits))) return -1;
        if (k_branch_index(gbt, st)) return -1;
        gbt.hbits = BranchTable::hash_bits(B_tot);      // every rank hashes the whole table: one probe per lookup in K9
        while (gbt.hbits > 10 && (16ull << gbt.hbits) > (4ull << 30) && (1ull << (gbt.hbits - 1)) >= B_tot + B_tot / 2) --gbt.hbits;
        if (dalloc(s, &gbt.hslots, 1ull << gbt.hbits) || k_branch_hash(gbt, st)) return -1;
    }
    S.n_branch = B_tot; S.n_blue = M_tot;
    pc.tick("branch_table");
    SCUDA(cudaEventRecord(s->ev[4], st));

    // ---- 6. sentinel-window suffixes: ranked on every rank (same text), insertion points summed over the key ranges ----
    const u64 nspec = 32 * R;
    std::vector<u64> h_ins, h_rows, h_emit_pos, h_tail_pos;
    std::vector<u8> h_chr;
    {
        std::vector<SpecialInfo> info(nspec);
        SpecialInfo* d_info = nullptr;
        if (dalloc(s, &d_info, nspec)) return -1;
        if (k_special_scan(W, d_seps, R, sk, n_loc, ki, d_info, st)) return -1;
        SCUDA(cudaMemcpyAsync(info.data(), d_info, nspec * sizeof(SpecialInfo), cudaMemcpyDeviceToHost, st));
        SCUDA(cudaStreamSynchronize(st));
        if (G > 1) {                                   // sum of the local insertion points = global insertion point
            if (ensure_shared(s, s->mail, (size_t)G * nspec * 8)) return -1;
            std::vector<u64> loc(nspec);
            for (u64 t = 0; t < nspec; ++t) loc[t] = info[t].ins;
            u64* d_loc = nullptr;
            if (dalloc(s, &d_loc, nspec)) return -1;
            SCUDA(cudaMemcpyAsync(d_loc, loc.data(), nspec * 8, cudaMemcpyHostToDevice, st));
            for (int p = 0; p < G; ++p)
                if (peer_copy(s, static_cast<u64*>(s->mail.ptr[p]) + (u64)me * nspec, d_loc, nspec * 8)) return -1;
            if (sync_all(s)) return -1;
            std::vector<u64> all((size_t)G * nspec);
            SCUDA(cudaMemcpyAsync(all.data(), s->mail.ptr[me], all.size() * 8, cudaMemcpyDeviceToHost, st));
            SCUDA(cudaStreamSynchronize(st));
            if (barrier(s)) return -1;                 // the mailbox may be written again
            for (u64 t = 0; t < nspec; ++t) {
                u64 sum = 0;
                for (int p = 0; p < G; ++p) sum += all[(size_t)p * nspec + t];
                info[t].ins = sum;
            }
        }
        if (build_special_tables(info.data(), seps, R, h_ins, h_rows, h_chr, h_emit_pos, h_tail_pos)) { s->err = debwt_last_error(); return -1; }
    }
    u64 *d_rows = nullptr, *d_ins = nullptr, *d_emit = nullptr, *d_tail = nullptr;
    u8* d_chr = nullptr;
    if (dalloc(s, &d_rows, nspec) || dalloc(s, &d_ins, nspec) || dalloc(s, &d_chr, nspec) || dalloc(s, &d_emit, h_emit_pos.size() + 1) ||
        dalloc(s, &d_tail, R))
        return -1;
    SCUDA(cudaMemcpyAsync(d_rows, h_rows.data(), nspec * 8, cudaMemcpyHostToDevice, st));
    SCUDA(cudaMemcpyAsync(d_ins, h_ins.data(), nspec * 8, cudaMemcpyHostToDevice, st));
    SCUDA(cudaMemcpyAsync(d_chr, h_chr.data(), nspec, cudaMemcpyHostToDevice, st));
    SCUDA(cudaMemcpyAsync(d_emit, h_emit_pos.data(), h_emit_pos.size() * 8, cudaMemcpyHostToDevice, st));
    SCUDA(cudaMemcpyAsync(d_tail, h_tail_pos.data(), R * 8, cudaMemcpyHostToDevice, st));

    pc.tick("special");
    // ---- 7. branch codes of own position slice at global code indices ----
    u32 *mo = nullptr, *wpfx = nullptr;
    u64 *rec_entry = nullptr, *rec_index = nullptr;
    const u64 cap = std::min(cnt, M_tot) + 1;
    void* scanws = nullptr;
    if (dalloc(s, &mo, wp + 2) || dalloc(s, &wpfx, wp + 2) || pool.alloc(&scanws, scan_workspace_bytes(wp) + 64)) return -1;
    const auto mark_records = pool.mark();
    if (dalloc(s, &rec_entry, cap) || dalloc(s, &rec_index, cap)) return -1;
    SCUDA(cudaMemsetAsync(mo, 0, (wp + 2) * 4, st));
    SCUDA(cudaMemsetAsync(d_small, 0, 64 * 8, st));
    if (k_flag_slice(W, pos_lo, pos_hi, d_seps, R, gbt, mo, rec_entry, rec_index, d_small, st)) return -1;
    if (k_patch_bits(mo, pos_lo, pos_hi_al, d_emit, h_emit_pos.size(), st)) return -1;
    if (scan_exclusive_u32(mo, wpfx, wp, true, scanws, d_small + 1, st)) return -1;
    u64 h_cnt[2] = {0, 0};
    SCUDA(cudaMemcpyAsync(h_cnt, d_small, 16, cudaMemcpyDeviceToHost, st));
    SCUDA(cudaStreamSynchronize(st));
    const u64 m_rec = h_cnt[0], s_loc = h_cnt[1];
    u64 s_all[kMaxRanks], code_base = 0, s_tot = 0;
    if (allgather(s, &s_loc, 1, s_all)) return -1;
    for (int p = 0; p < G; ++p) { if (p < me) code_base += s_all[p]; s_tot += s_all[p]; }
    const u64 ncw = s_tot / 32 + 3;
    S.n_codes = s_tot;
    // codes | separator bits | code index of every record's tail: one shared block, so that the peers can OR theirs in
    const size_t off_sep = ncw * 8, off_tail = off_sep + (((ncw + 1) * 4 + 7) & ~(size_t)7);
    if (ensure_shared(s, s->share, off_tail + R * 8 + 64)) return -1;
    char* sh = static_cast<char*>(s->share.ptr[me]);
    u64* codes = reinterpret_cast<u64*>(sh);
    u32* sep = reinterpret_cast<u32*>(sh + off_sep);
    u64* tail_idx = reinterpret_cast<u64*>(sh + off_tail);
    SCUDA(cudaMemsetAsync(sh, 0, off_tail + R * 8, st));
    if (k_emit_codes(W, (u64)me * wp, wp, mo, wpfx, code_base, codes, st)) return -1;
    if (k_mark_sep_codes(mo, wpfx, pos_lo, pos_hi_al, code_base, d_tail, R, sep, tail_idx, st)) return -1;
    if (G > 1) {
        if (sync_all(s)) return -1;                    // every rank's share is written
        u64 base_p = 0;
        for (int p = 0; p < G; ++p) {
            if (p != me && s_all[p]) {
                const char* ps = static_cast<const char*>(s->share.ptr[p]);
                const u64 lo = base_p / 32, hi = (base_p + s_all[p] + 31) / 32;
                or_range_kernel<u64><<<blocks(hi - lo), 256, 0, st>>>(codes, reinterpret_cast<const u64*>(ps), lo, hi);
                or_range_kernel<u32><<<blocks(hi - lo + 1), 256, 0, st>>>(sep, reinterpret_cast<const u32*>(ps + off_sep), lo, hi + 1);
                DEBWT_COUNT(2);
            }
            if (p != me) {
                or_range_kernel<u64><<<blocks(R), 256, 0, st>>>(tail_idx, reinterpret_cast<const u64*>(static_cast<const char*>(s->share.ptr[p]) + off_tail), 0, R);
                DEBWT_COUNT(1);
            }
            base_p += s_all[p];
        }
    }
    u64 dollar_index = 0;
    if (G > 1) {
        // peers read each other's ORIGINAL words while OR-ing: a code word is written by at most two ranks (a shared
        // boundary word), each of which only adds its own bits, so reading a word a peer has already OR-ed into is harmless
        if (sync_all(s)) return -1;
    }
    SCUDA(cudaMemcpyAsync(&dollar_index, tail_idx + (R - 1), 8, cudaMemcpyDeviceToHost, st));
    if (k_blue_fix(rec_entry, m_rec, mo, wpfx, pos_lo, code_base, st)) return -1;
    SCUDA(cudaStreamSynchronize(st));
    pc.tick("codes");
    SCUDA(cudaEventRecord(s->ev[7], st));

    // ---- 8. blue entries travel to the owner of their k-mer ----
    u64* blue = nullptr;
    {
        u64 *d_bbase = nullptr;
        if (dalloc(s, &d_bbase, kMaxRanks + 1)) return -1;
        SCUDA(cudaMemcpyAsync(d_bbase, b_base, (kMaxRanks + 1) * 8, cudaMemcpyHostToDevice, st));
        const u64* e_recv = rec_entry;
        const u64* i_recv = rec_index;
        u8* db = nullptr;
        u64 *e_part = nullptr, *i_part = nullptr;
        if (dalloc(s, &db, m_rec + 16)) return -1;
        if (k_owner_of_index(rec_index, m_rec, d_bbase, (u32)G, db, st)) return -1;      // also makes the indices owner-local
        if (G > 1) {
            if (dalloc(s, &e_part, m_rec + 1) || dalloc(s, &i_part, m_rec + 1)) return -1;
            PartitionBy by;
            by.dest = db;
            u64 counts[kMaxRanks] = {}, mat[kMaxRanks * kMaxRanks], curs[kMaxRanks] = {};
            SCUDA(cudaMemsetAsync(d_small, 0, 32 * 8, st));
            if (k_partition_count(rec_entry, by, m_rec, (u32)G, d_small, st)) return -1;
            SCUDA(cudaMemcpyAsync(counts, d_small, kMaxRanks * 8, cudaMemcpyDeviceToHost, st));
            SCUDA(cudaStreamSynchronize(st));
            for (int d = 1; d < G; ++d) curs[d] = curs[d - 1] + counts[d - 1];
            SCUDA(cudaMemcpyAsync(d_small + 16, curs, kMaxRanks * 8, cudaMemcpyHostToDevice, st));
            if (k_partition_scatter(rec_entry, rec_index, by, m_rec, (u32)G, d_small + 16, e_part, i_part, st)) return -1;
            if (allgather(s, counts, kMaxRanks, mat)) return -1;
            u64 max_m = 0;
            for (int p = 0; p < G; ++p) max_m = std::max(max_m, m_all[p]);
            if (ensure_shared(s, s->recv_b, (2 * max_m + 4) * 8)) return -1;
            u64 col = 0;
            for (int src = 0; src < G; ++src) col += mat[src * kMaxRanks + me];
            if (col != bt.n_blue) SFAIL("internal: blue entry exchange mismatch");
            for (int d = 0; d < G; ++d) {
                if (!counts[d]) continue;
                u64 off = 0;
                for (int src = 0; src < me; ++src) off += mat[src * kMaxRanks + d];
                u64* base = static_cast<u64*>(s->recv_b.ptr[d]);
                if (peer_copy(s, base + off, e_part + curs[d], counts[d] * 8)) return -1;
                if (peer_copy(s, base + m_all[d] + 2 + off, i_part + curs[d], counts[d] * 8)) return -1;
            }
            if (sync_all(s)) return -1;
            e_recv = static_cast<const u64*>(s->recv_b.ptr[me]);
            i_recv = e_recv + bt.n_blue + 2;
        } else if (m_rec != bt.n_blue) {
            SFAIL("internal: blue entry count mismatch");
        }
        if (G > 1) pool.rewind(mark_records);          // the flagged records are dead once they have been sent (one rank reads them in place)
        pc.tick("blue_exchange");
        if (dalloc(s, &blue, bt.n_blue + 1)) return -1;
        SCUDA(cudaMemsetAsync(bt.cursor, 0, (bt.n_branch + 1) * 4, st));
        if (k_scatter_blue(e_recv, i_recv, bt.n_blue, bt, blue, st)) return -1;
        u32* d_work = nullptr;
        if (dalloc(s, &d_work, 4 * bt.n_branch + 16)) return -1;
        SCUDA(cudaMemsetAsync(d_work, 0, (4 * bt.n_branch + 16) * 4, st));
        SpView spv{codes, sep, dollar_index, s_tot};
        if (k_sort_blue(blue, bt, spv, d_work, st)) { s->err = debwt_last_error(); return -1; }
    }

    pc.tick("scatter+k10");
    // ---- 9. every rank emits its own contiguous run of BWT rows and stores it into rank 0's result ----
    const u64 n_out = (N + 31) / 32;
    u64 r_lo_all[kMaxRanks + 1];
    {
        u64 kb = 0;
        for (int p = 0; p < G; ++p) {
            r_lo_all[p] = kb == 0 ? 0 : kb + (u64)(std::upper_bound(h_ins.begin(), h_ins.end(), kb) - h_ins.begin());
            kb += n_all[p];
        }
        r_lo_all[G] = N;
    }
    const u64 my_lo = r_lo_all[me], my_hi = r_lo_all[me + 1];
    const u64 w_lo = my_lo >> 5, w_hi = (my_hi + 31) >> 5;
    if (ensure_shared(s, s->out, me == 0 ? (n_out + 2) * 8 : 64)) return -1;
    u64* out0 = static_cast<u64*>(s->out.ptr[0]);
    if (me == 0) SCUDA(cudaMemsetAsync(out0, 0, (n_out + 2) * 8, st));
    u64* seg = nullptr;
    u64* d_sharp = nullptr;
    u32* d_scnt = nullptr;
    u64* d_dollar = nullptr;
    if (dalloc(s, &seg, w_hi - w_lo + 2) || dalloc(s, &d_sharp, R + 1) || dalloc(s, &d_scnt, 4) || dalloc(s, &d_dollar, 2)) return -1;
    SCUDA(cudaMemsetAsync(seg, 0, (w_hi - w_lo + 2) * 8, st));
    SCUDA(cudaMemsetAsync(d_scnt, 0, 16, st));
    SCUDA(cudaMemsetAsync(d_dollar, 0xff, 16, st));
    u64* bwt_v = seg - w_lo;                           // the emit kernels index with global word numbers
    if (my_hi > my_lo) {
        if (n_loc && k_fill_case2(gmask, n_loc, key_base, N, d_rows, nspec, w_lo, w_hi, bwt_v, st)) return -1;
        const u64 t_lo = (u64)(std::lower_bound(h_rows.begin(), h_rows.end(), my_lo) - h_rows.begin());
        const u64 t_hi = (u64)(std::lower_bound(h_rows.begin(), h_rows.end(), my_hi) - h_rows.begin());
        if (t_hi > t_lo && k_emit_special(d_rows + t_lo, d_chr + t_lo, t_hi - t_lo, bwt_v, st)) return -1;
    }
    if (k_emit_blue(blue, bt, key_base, d_ins, nspec, bwt_v, d_sharp, d_scnt, d_dollar, st)) return -1;
    if (G > 1) {
        if (sync_all(s)) return -1;                    // rank 0's result buffer is zeroed
    }
    if (w_hi > w_lo) {
        or_store_kernel<<<blocks(w_hi - w_lo), 256, 0, st>>>(out0 + w_lo, seg, w_hi - w_lo);
        DEBWT_COUNT(1);
    }
    // '#' rows and the '$' row
    u32 scnt = 0;
    u64 dol = ~0ull;
    std::vector<u64> sharp_loc(R + 1);
    SCUDA(cudaMemcpyAsync(&scnt, d_scnt, 4, cudaMemcpyDeviceToHost, st));
    SCUDA(cudaMemcpyAsync(&dol, d_dollar, 8, cudaMemcpyDeviceToHost, st));
    SCUDA(cudaMemcpyAsync(sharp_loc.data(), d_sharp, (R + 1) * 8, cudaMemcpyDeviceToHost, st));
    SCUDA(cudaEventRecord(s->ev[1], st));              // reuse: end of the build on this rank
    if (sync_all(s)) return -1;
    {
        // gather the separator rows on rank 0 through its mailbox
        u64 mine[2] = {scnt, dol}, all[kMaxRanks * 2];
        if (allgather(s, mine, 2, all)) return -1;
        u64 off = 0, tot = 0;
        for (int p = 0; p < G; ++p) { if (p < me) off += all[p * 2]; tot += all[p * 2]; if (all[p * 2 + 1] != ~0ull) s->dollar = all[p * 2 + 1]; }
        if (tot != R - 1) SFAIL("internal: wrong number of '#' rows");
        if (G > 1) {
            if (ensure_shared(s, s->mail, (R + 2) * 8)) return -1;
            if (scnt && peer_copy(s, static_cast<u64*>(s->mail.ptr[0]) + off, d_sharp, scnt * 8)) return -1;
            if (sync_all(s)) return -1;
            if (me == 0) {
                s->sharp.resize(tot);
                if (tot) SCUDA(cudaMemcpyAsync(s->sharp.data(), s->mail.ptr[0], tot * 8, cudaMemcpyDeviceToHost, st));
                SCUDA(cudaStreamSynchronize(st));
            }
            if (barrier(s)) return -1;
        } else {
            s->sharp.assign(sharp_loc.begin(), sharp_loc.begin() + scnt);
        }
        std::sort(s->sharp.begin(), s->sharp.end());
    }
    pc.tick("emit+stitch");
    if (pc.on && me == 0) fprintf(stderr, "[shard phases ms]%s\n", pc.out.c_str());
    float ms = 0;
    SCUDA(cudaEventElapsedTime(&ms, s->ev[0], s->ev[1])); S.ms_total = ms;
    SCUDA(cudaEventElapsedTime(&ms, s->ev[2], s->ev[3])); S.ms_sort = ms;
    if (S.sort_sweeps) { SCUDA(cudaEventElapsedTime(&ms, s->ev[5], s->ev[6])); S.ms_sort_sweeps = ms; }
    S.arena_bytes = pool.reserved_bytes();
    s->n = N; s->n_rec = R;
    s->built = true;
    return 0;
}

}  // namespace

extern "C" {

int debwt_shard_create(debwt_shard** out, int device, int rank, int world, const char* group_tag, int same_process) {
    if (!out || !group_tag) { set_error("null argument"); return -1; }
    if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world) { set_error("1..16 ranks"); return -1; }
    if (debwt_device_count() <= device || device < 0) { set_error("no such CUDA device (this library has no CPU fallback)"); return -1; }
    debwt_shard* s = new debwt_shard();
    s->device = device; s->rank = rank; s->world = world; s->same_process = same_process != 0;
    auto fail = [&](const std::string& m) { set_error(m); delete s; return -1; };
    if (cudaSetDevice(device) != cudaSuccess) return fail("cudaSetDevice failed");
    if (cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking) != cudaSuccess) return fail("cannot create a stream");
    {   // K10 takes its work lists from the stream-ordered pool: keep what it frees cached instead of returning it to the driver
        cudaMemPool_t mp;
        unsigned long long thr = ~0ull;
        if (cudaDeviceGetDefaultMemPool(&mp, device) == cudaSuccess) cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    for (auto& e : s->ev) if (cudaEventCreate(&e) != cudaSuccess) return fail("cannot create an event");
    s->pool.st = s->st;
    std::string err;
    if (s->comm.open(group_tag, rank, world, &err)) return fail(err);
    int devs[kMaxRanks] = {};
    if (s->comm.allgather(&device, sizeof(int), devs, &err)) return fail(err);
    for (int r = 0; r < world; ++r) s->peer_device[r] = devs[r];
    if (s->same_process)
        for (int r = 0; r < world; ++r) {
            if (devs[r] == device) continue;
            const cudaError_t e = cudaDeviceEnablePeerAccess(devs[r], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail("peer access between the GPUs is not available");
            cudaGetLastError();
        }
    *out = s;
    return 0;
}

void debwt_shard_destroy(debwt_shard* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    cudaStreamSynchronize(s->st);
    std::string e;
    s->comm.barrier(&e);                               // nobody unmaps while a peer may still read
    for (SharedBuf* b : {&s->words, &s->recv_a, &s->recv_b, &s->gkmer, &s->share, &s->out, &s->mail}) {
        unmap(s, *b);
    }
    s->comm.barrier(&e);
    for (SharedBuf* b : {&s->words, &s->recv_a, &s->recv_b, &s->gkmer, &s->share, &s->out, &s->mail})
        if (b->ptr[s->rank]) cudaFree(b->ptr[s->rank]);
    s->pool.destroy();
    for (auto& ev : s->ev) if (ev) cudaEventDestroy(ev);
    cudaStreamDestroy(s->st);
    s->comm.close_all();
    delete s;
}

int debwt_shard_set_sort_config(debwt_shard* s, int cfg) {
    const int old = s->sort_cfg;
    s->sort_cfg = cfg > 0 ? cfg : kDefaultSortCfg;
    return old;
}

int debwt_shard_slice(int rank, int world, uint64_t n_symbols, uint64_t* lo, uint64_t* hi) {
    if (world < 1 || rank < 0 || rank >= world || !lo || !hi) { set_error("bad argument"); return -1; }
    const u64 n_words = (n_symbols + 32 + 31) / 32 + 1;
    const u64 wp = (n_words + world - 1) / world;
    const u64 a = std::min<u64>(32 * (u64)rank * wp, n_symbols);
    const u64 b = std::max<u64>(std::min<u64>(32 * (u64)(rank + 1) * wp, n_symbols), a);
    *lo = a;
    *hi = b;
    return 0;
}

int debwt_shard_build(debwt_shard* s, const void* slice, int slice_on_device, uint64_t n_symbols, const uint64_t* seps,
                      uint64_t n_records) {
    if (!s || !seps || (!slice && n_symbols)) { set_error("null argument"); return -1; }
    const int rc = shard_build_impl(s, slice, slice_on_device, n_symbols, reinterpret_cast<const u64*>(seps), n_records);
    if (rc && !s->err.empty()) set_error(s->err);
    return rc;
}

int debwt_shard_result_device(const debwt_shard* s, const uint64_t** d_bwt_words, uint64_t* n_words) {
    if (!s || !s->built) { set_error("no result: call debwt_shard_build first"); return -1; }
    if (d_bwt_words) *d_bwt_words = s->rank == 0 ? reinterpret_cast<const uint64_t*>(s->out.ptr[0]) : nullptr;
    if (n_words) *n_words = (s->n + 31) / 32;
    return 0;
}

int debwt_shard_result_copy(debwt_shard* s, uint64_t* bwt_words, uint64_t* sharp_rows, uint64_t* dollar_row) {
    if (!s || !s->built) { set_error("no result: call debwt_shard_build first"); return -1; }
    if (s->rank != 0) return 0;
    CUDA_TRY(cudaSetDevice(s->device));
    if (bwt_words) {
        CUDA_TRY(cudaMemcpyAsync(bwt_words, s->out.ptr[0], ((s->n + 31) / 32) * 8, cudaMemcpyDeviceToHost, s->st));
        CUDA_TRY(cudaStreamSynchronize(s->st));
    }
    if (sharp_rows) std::copy(s->sharp.begin(), s->sharp.end(), sharp_rows);
    if (dollar_row) *dollar_row = s->dollar;
    return 0;
}

int debwt_shard_get_stats(const debwt_shard* s, debwt_shard_stats* out) {
    if (!s || !out) { set_error("null argument"); return -1; }
    *out = s->stats;
    return 0;
}

// One process, one thread per GPU: what host/deBWT -g 0,1,... calls.
int debwt_build_multi(const int* devices, int n_devices, const char* text, uint64_t n_symbols, const uint64_t* seps, uint64_t n_records,
                      uint64_t* bwt_words, uint64_t* sharp_rows, uint64_t* dollar_row, debwt_shard_stats* stats_out) {
    if (!devices || n_devices < 1 || n_devices > kMaxRanks || !text || !seps) { set_error("bad argument"); return -1; }
    for (int r = 0; r < n_devices; ++r)
        if (devices[r] < 0 || devices[r] >= debwt_device_count()) { set_error("no such CUDA device (this library has no CPU fallback)"); return -1; }
    static unsigned counter = 0;
    const std::string tag = "mt_" + std::to_string((long)getpid()) + "_" + std::to_string(++counter);
    std::vector<int> rc(n_devices, 0);
    std::vector<std::string> errs(n_devices);
    std::vector<std::thread> th;
    for (int r = 0; r < n_devices; ++r)
        th.emplace_back([&, r]() {
            debwt_shard* s = nullptr;
            if (debwt_shard_create(&s, devices[r], r, n_devices, tag.c_str(), 1)) { rc[r] = -1; errs[r] = debwt_last_error(); return; }
            uint64_t lo = 0, hi = 0;
            debwt_shard_slice(r, n_devices, n_symbols, &lo, &hi);
            rc[r] = debwt_shard_build(s, text + lo, 0, n_symbols, seps, n_records);
            if (!rc[r] && r == 0) {
                rc[r] = debwt_shard_result_copy(s, bwt_words, sharp_rows, dollar_row);
                if (stats_out) debwt_shard_get_stats(s, stats_out);
            }
            if (rc[r]) errs[r] = debwt_last_error();
            debwt_shard_destroy(s);
        });
    for (auto& t : th) t.join();
    for (int r = 0; r < n_devices; ++r)
        if (rc[r]) { set_error(errs[r]); return -1; }
    return 0;
}

}  // extern "C"
