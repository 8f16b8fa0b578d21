// Internal: the build context behind the opaque debwt_ctx of include/debwt_b200.h, and its device arena.
#pragma once
#include <vector>

#include "../../include/debwt_b200.h"
#include "common.cuh"

namespace debwt {

constexpr int kDefaultSortCfg = 8;          // 384 threads x 16 keys per tile, 3 CTAs/SM

// ---------------------------------------------------------------------------------------------
// device memory: a per-context arena (grow-only chunks, bump allocation, reset per build).  The driver's
// stream-ordered pool (cudaMallocAsync) showed millisecond-level, step-to-step variance for the
// multi-hundred-MB buffers of a build; an arena makes steady-state builds allocation-free.
// ---------------------------------------------------------------------------------------------
struct DevPool {
    struct Chunk { char* base; size_t cap, used; bool owned; };
    cudaStream_t st = nullptr;
    std::vector<Chunk> chunks;          // adopted (borrowed) regions first, then the chunks this pool cudaMalloc'ed
    size_t next_chunk = 256ull << 20;
    void hint(size_t bytes) { if (bytes > next_chunk) next_chunk = bytes; }
    int alloc(void** p, size_t bytes) {
        bytes = (bytes + 511) & ~(size_t)511;
        if (bytes == 0) bytes = 512;
        for (auto& c : chunks) {
            if (c.cap - c.used >= bytes) { *p = c.base + c.used; c.used += bytes; return 0; }
        }
        Chunk c{nullptr, bytes > next_chunk ? bytes : next_chunk, 0, true};
        CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c.base), c.cap));
        *p = c.base;
        c.used = bytes;
        chunks.push_back(c);
        return 0;
    }
    // A buffer of this pool that the build no longer needs (the ping-pong half the sort did not end in, the ASCII text
    // after packing) becomes a region later allocations are served from first.  It stays reserved in its own chunk,
    // so nothing is handed out twice; adopted regions vanish at the next rewind.
    void adopt(void* p, size_t bytes) {
        char* q = static_cast<char*>(p);
        char* a = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(q) + 511) & ~(uintptr_t)511);
        if (!p || a >= q + bytes) return;
        const size_t cap = (size_t)(q + bytes - a) & ~(size_t)511;
        if (cap) chunks.insert(chunks.begin(), Chunk{a, cap, 0, false});
    }
    // state of the owned chunks (bytes in use), to come back to before a build
    std::vector<size_t> mark() const {
        std::vector<size_t> m;
        for (auto& c : chunks) if (c.owned) m.push_back(c.used);
        return m;
    }
    void rewind(const std::vector<size_t>& m) {
        std::vector<Chunk> keep;
        size_t i = 0;
        for (auto& c : chunks) {
            if (!c.owned) continue;
            c.used = i < m.size() ? m[i] : 0;
            ++i;
            keep.push_back(c);
        }
        chunks.swap(keep);
    }
    void release_all() { rewind({}); }
    size_t reserved_bytes() const {             // HBM this pool holds
        size_t t = 0;
        for (auto& c : chunks) if (c.owned) t += c.cap;
        return t;
    }
    size_t used_bytes() const {                 // high-water marks of the owned chunks (adopted regions live inside them)
        size_t t = 0;
        for (auto& c : chunks) if (c.owned) t += c.used;
        return t;
    }
    void destroy() {
        for (auto& c : chunks) if (c.owned) cudaFree(c.base);
        chunks.clear();
    }
};

}  // namespace debwt

struct debwt_ctx {
    int device = 0;
    int sort_cfg = debwt::kDefaultSortCfg;
    int blue_grouping = 0;              // K9: 0 auto, 1 per-segment cursors, 2 grouping sort (debwt_set_blue_grouping)
    cudaStream_t st = nullptr;
    debwt::DevPool pool;
    // input
    u64 n = 0, n_rec = 0;
    std::vector<u64> seps;
    u8* d_ascii = nullptr;         // owned unless external
    const u8* d_ascii_ext = nullptr;
    // streaming ingest (debwt_ingest_*): the text arrives in chunks through pinned staging and is packed on the fly
    struct Ingest {
        bool active = false;
        u8* h_stage[2] = {nullptr, nullptr};       // pinned host staging (owned by the context, allocated once)
        u8* d_stage[2] = {nullptr, nullptr};       // device staging (arena)
        cudaEvent_t done[2] = {nullptr, nullptr};  // stage i's copy + pack have run
        bool busy[2] = {false, false};
        int cur = 0;
        u64 fill = 0;                              // bytes in the current stage (incl. the < 32 carried over)
        u64 n = 0;                                 // symbols packed so far (a multiple of 32 until the end)
        u64 cap_words = 0;
    } ing;
    // debwt_k_group_masks / debwt_k_branch_kmers / debwt_k_codes: the build copies the K5-K7 masks and the K9 products to
    // the host right before K10 (test entry points only)
    struct Capture {
        bool on = false;
        std::vector<u16> gmask;        // per sorted key: its group's mask, as K7's count pass leaves it (propagated)
        std::vector<u64> codes;        // packed 2-bit SP codes
        std::vector<u32> sep;          // 1 bit per code: '#' / '$'
        u64 dollar_index = 0, n_codes = 0;
        std::vector<u64> blue;         // (spIndex << 4) | prev, grouped by segment, unsorted inside
        std::vector<u32> seg_off;      // n_branch + 1 offsets into blue
        std::vector<u32> seg_head;     // sorted-key index of each branch k-mer's group
        std::vector<u64> seg_kmer;     // (k-mer << 2) | multi_in << 1 | multi_out
    } cap;
    bool resolve_ambiguous = false;   // debwt_set_ambiguity_policy
    u64 ambiguity_seed = 0;
    u64* d_packed = nullptr;          // packed text produced by the ingest (skips K1 in the build)
    u32* d_packed_err = nullptr;
    // result
    u64* d_bwt = nullptr;
    u64* d_sharp = nullptr;
    u32* d_sharp_count = nullptr;
    u64* d_dollar = nullptr;
    u64 n_words = 0;
    bool built = false;
    std::vector<size_t> input_mark;   // pool state right after the input was set: every build starts from here
    debwt_stats stats{};
    cudaEvent_t ev[16]{};
    // FM-index tables over the result (index.cu); own cudaMalloc allocations, dropped with the result
    u64* d_occ = nullptr;             // [(N >> 5) + 1][4]
    u32* d_spec_bits = nullptr;       // one bit per row: the row holds '#' or '$'
    u64* d_sharp_sorted = nullptr;    // n_rec - 1 rows holding '#', ascending
    u64 c_array[6] = {0, 0, 0, 0, 0, 0};
    u64 dollar_row = 0;
    bool indexed = false;
    // sampled suffix array (index.cu, debwt_index_sample_sa); own cudaMalloc allocations, dropped with the index
    u64* d_sa_bits = nullptr;         // [ceil(N / 32)]: sampled-row mask of the word (low half) | sampled rows before it (high)
    u32* d_sa_vals = nullptr;         // SA values of the sampled rows, in row order
    u32 sa_rate = 0;                  // 0 = not sampled
    u64 n_sa_samples = 0;
    u32* d_isa_vals = nullptr;        // [n_sa_samples]: [k] = row of suffix k * rate (the first debwt_index_extract after sampling)
    u64* d_seps_sorted = nullptr;     // [n_rec]: the separator positions, ascending (the first debwt_index_seeds after sampling)
    u32* d_pac = nullptr;             // bwa's pac, 16 forward bases per word, base x at bits 2 (x & 15) (the first debwt_index_regions after sampling)
    bool loaded = false;              // the result came from debwt_set_result, not from a build
};

namespace debwt {
void drop_index(debwt_ctx* c);        // index.cu
void drop_samples(debwt_ctx* c);      // index.cu
}

