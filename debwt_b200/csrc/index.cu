// FM-index tables over the finished BWT and the at-scale verifier built on them (SURVEY.md section 8 f2 / 8c).
//
// The reference builds these in its unreachable "developer mode": occ checkpoints every 32 rows
// (reference src/insertCase3.c:139-208: occ[(N >> 5) + 1][4], rows holding '#'/'$' are stored as T but not counted),
// the C-array of cumulative base counts (src/collect#$.c:92-100), and an LF walk that inverts the BWT
// (src/LFsearch.c:49-166, findSeg :167-235: '#' rows map to the last R rows in rank order, :131).  Here:
//   * occ + C are produced on the device in the reference's layout (one sweep over the packed BWT);
//   * LF(r) for every row in one kernel;
//   * the reference walks the LF permutation one row at a time (N dependent steps); on the GPU the walk is list ranking by
//     pointer jumping (Wyllie): ceil(log2 N) rounds of one random 8-byte gather per row, after which every row knows
//     its distance to the end of the walk, i.e. its text position.  The BWT is the BWT of T iff the permutation is ONE
//     cycle and the symbol of row r equals T[position(r) - 1] for every r -- checked against the caller's ASCII text.
#include <algorithm>
#include <string>
#include <vector>

#include "ctx.cuh"

namespace debwt {

namespace {

constexpr int TPB = 256;
constexpr u32 NIL = 0xFFFFFFFFu;
inline unsigned grid_for(u64 work, u64 per_block = TPB) { return (unsigned)((work + per_block - 1) / per_block); }

// bit j (0..31) of the result set <=> symbol j of the packed word (bits 2*(31-j)) equals `code`
__device__ __forceinline__ u32 symbol_mask(u64 w, u32 code) {
    const u64 x = w ^ (code & 2u ? 0ull : 0xAAAAAAAAAAAAAAAAull) ^ (code & 1u ? 0ull : 0x5555555555555555ull);
    u64 m = x & (x >> 1) & 0x5555555555555555ull;          // bit 2*(31-j) set where both bits match
    // compress the even bits: symbol j sits at bit 2*(31-j) -> bit (31-j); then reverse so that symbol j is bit j
    m = (m | (m >> 1)) & 0x3333333333333333ull;
    m = (m | (m >> 2)) & 0x0F0F0F0F0F0F0F0Full;
    m = (m | (m >> 4)) & 0x00FF00FF00FF00FFull;
    m = (m | (m >> 8)) & 0x0000FFFF0000FFFFull;
    m = (m | (m >> 16)) & 0x00000000FFFFFFFFull;
    return __brev((u32)m);
}
__device__ __forceinline__ u32 valid_rows(u64 n, u64 w) {                 // rows of word w that exist
    const u64 left = n - w * 32;
    return left >= 32 ? 0xFFFFFFFFu : ((1u << left) - 1u);
}

__global__ void __launch_bounds__(TPB) spec_bits_kernel(u32* __restrict__ bits, const u64* __restrict__ rows, u64 m) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t < m) atomicOr(bits + (rows[t] >> 5), 1u << (rows[t] & 31));
}

// per block of TPB words: totals of A, C, G, T (specials excluded)
__global__ void __launch_bounds__(TPB) occ_count_kernel(const u64* __restrict__ bwt, const u32* __restrict__ spec, u64 n, u64 nwords,
                                                       u32* __restrict__ block_tot) {
    __shared__ u32 sm[40];
    const u64 w = (u64)blockIdx.x * TPB + threadIdx.x;
    u32 ac = 0, gt = 0;
    if (w < nwords) {
        const u64 x = bwt[w];
        const u32 ok = valid_rows(n, w) & ~spec[w];
        ac = __popc(symbol_mask(x, 0) & ok) | (__popc(symbol_mask(x, 1) & ok) << 16);
        gt = __popc(symbol_mask(x, 2) & ok) | (__popc(symbol_mask(x, 3) & ok) << 16);
    }
    u32 t_ac, t_gt;
    block_exclusive_scan<TPB>(ac, &t_ac, sm);
    block_exclusive_scan<TPB>(gt, &t_gt, sm);
    if (threadIdx.x == 0) {
        u32* o = block_tot + (u64)blockIdx.x * 4;
        o[0] = t_ac & 0xffffu; o[1] = t_ac >> 16; o[2] = t_gt & 0xffffu; o[3] = t_gt >> 16;
    }
}

// exclusive scan over the block totals (one block, sequential over chunks) -> 64-bit bases; totals[4] at the end
__global__ void __launch_bounds__(1024) occ_scan_kernel(const u32* __restrict__ block_tot, u64 nb, u64* __restrict__ block_base,
                                                       u64* __restrict__ totals) {
    __shared__ u32 sm[40];
    __shared__ u64 carry[4];
    if (threadIdx.x < 4) carry[threadIdx.x] = 0;
    __syncthreads();
    for (u64 base = 0; base < nb; base += 1024) {
        const u64 i = base + threadIdx.x;
        for (int c = 0; c < 4; ++c) {
            const u32 v = i < nb ? block_tot[i * 4 + c] : 0;
            u32 total;
            const u32 ex = block_exclusive_scan<1024>(v, &total, sm);
            if (i < nb) block_base[i * 4 + c] = carry[c] + ex;
            __syncthreads();
            if (threadIdx.x == 0) carry[c] += total;
            __syncthreads();
        }
    }
    if (threadIdx.x < 4) totals[threadIdx.x] = carry[threadIdx.x];
}

// occ[w][c] = number of symbol c in rows [0, 32 w)   (reference layout, src/insertCase3.c:141-142)
__global__ void __launch_bounds__(TPB) occ_write_kernel(const u64* __restrict__ bwt, const u32* __restrict__ spec, u64 n, u64 nwords,
                                                       const u64* __restrict__ block_base, u64* __restrict__ occ, u64 occ_len) {
    __shared__ u32 sm[40];
    const u64 w = (u64)blockIdx.x * TPB + threadIdx.x;
    u32 ac = 0, gt = 0;
    if (w < nwords) {
        const u64 x = bwt[w];
        const u32 ok = valid_rows(n, w) & ~spec[w];
        ac = __popc(symbol_mask(x, 0) & ok) | (__popc(symbol_mask(x, 1) & ok) << 16);
        gt = __popc(symbol_mask(x, 2) & ok) | (__popc(symbol_mask(x, 3) & ok) << 16);
    }
    const u32 e_ac = block_exclusive_scan<TPB>(ac, nullptr, sm);
    const u32 e_gt = block_exclusive_scan<TPB>(gt, nullptr, sm);
    if (w < occ_len) {
        const u64* b = block_base + (u64)blockIdx.x * 4;
        ulonglong2* o = reinterpret_cast<ulonglong2*>(occ + w * 4);
        o[0] = make_ulonglong2(b[0] + (e_ac & 0xffffu), b[1] + (e_ac >> 16));
        o[1] = make_ulonglong2(b[2] + (e_gt & 0xffffu), b[3] + (e_gt >> 16));
    }
    // the checkpoint one past the last word (when N is a multiple of 32 times ... the reference allocates (N >> 5) + 1)
    if (w + 1 == nwords && w + 1 < occ_len) {
        const u64* b = block_base + (u64)blockIdx.x * 4;
        ulonglong2* o = reinterpret_cast<ulonglong2*>(occ + (w + 1) * 4);
        o[0] = make_ulonglong2(b[0] + (e_ac & 0xffffu) + (ac & 0xffffu), b[1] + (e_ac >> 16) + (ac >> 16));
        o[1] = make_ulonglong2(b[2] + (e_gt & 0xffffu) + (gt & 0xffffu), b[3] + (e_gt >> 16) + (gt >> 16));
    }
}

struct FmView {
    const u64* bwt;
    const u32* spec;
    const u64* occ;
    const u64* sharp;      // sorted rows holding '#'
    u64 n_sharp;
    u64 dollar_row;
    u64 n;
    u64 C[6];
};

// number of rows < r holding base c (0..3)   (findSeg, src/LFsearch.c:167-235, without the -1 / +ACGT[type])
__device__ __forceinline__ u64 occ_before(const FmView& f, u32 c, u64 r) {
    const u64 w = r >> 5;
    const u32 below = (1u << (r & 31)) - 1u;
    u64 v = f.occ[w * 4 + c];
    if (below) v += __popc(symbol_mask(f.bwt[w], c) & ~f.spec[w] & below);
    return v;
}

// symbol of row r: 0..3, 4 = '#', 5 = '$'
__device__ __forceinline__ u32 row_symbol(const FmView& f, u64 r) {
    if ((f.spec[r >> 5] >> (r & 31)) & 1u) return r == f.dollar_row ? 5u : 4u;
    return (u32)(f.bwt[r >> 5] >> (2 * (31 - (r & 31)))) & 3u;
}

__device__ __forceinline__ u64 lf_of(const FmView& f, u64 r) {
    const u32 c = row_symbol(f, r);
    if (c == 5u) return f.n - 1;                                                  // '$' is the largest suffix
    if (c == 4u) return f.C[4] + lower_bound_u64(f.sharp, 0, f.n_sharp, r);       // src/LFsearch.c:131
    return f.C[c] + occ_before(f, c, r);
}

// list node of row r: successor (LF) in the high half, distance to it in the low half; the row whose LF is the start
// row (the row of suffix 0, which holds '$') ends the list
__global__ void __launch_bounds__(TPB) lf_init_kernel(FmView f, u64* __restrict__ node) {
    const u64 r = (u64)blockIdx.x * TPB + threadIdx.x;
    if (r >= f.n) return;
    const u64 s = lf_of(f, r);
    node[r] = s == f.dollar_row ? ((u64)NIL << 32) : ((s << 32) | 1ull);
}

__global__ void __launch_bounds__(TPB) jump_kernel(const u64* __restrict__ in, u64* __restrict__ out, u64 n, u32* __restrict__ live) {
    const u64 r = (u64)blockIdx.x * TPB + threadIdx.x;
    if (r >= n) return;
    u64 a = in[r];
    const u32 s = (u32)(a >> 32);
    bool more = false;
    if (s != NIL) {
        const u64 b = in[s];
        a = (b & 0xFFFFFFFF00000000ull) | (u32)((u32)a + (u32)b);
        more = (u32)(b >> 32) != NIL;
    }
    out[r] = a;
    if (__any_sync(0xffffffffu, more) && (threadIdx.x & 31) == 0) *live = 1u;
}

__device__ __forceinline__ u32 ascii_symbol(u8 c) {
    if (c == '#') return 4u;
    if (c == '$') return 5u;
    const u32 u = c & 0xDFu;
    const u32 x = (u >> 1) & 3u;
    return x ^ (x >> 1);
}

// after the jumps: the low half of node[r] is the number of LF steps from r to the end of the walk = position(r) - 1
__global__ void __launch_bounds__(TPB) lf_check_kernel(FmView f, const u64* __restrict__ node, const u8* __restrict__ text,
                                                      unsigned long long* __restrict__ bad) {
    const u64 r = (u64)blockIdx.x * TPB + threadIdx.x;
    if (r >= f.n) return;
    const u64 a = node[r];
    bool ok = (u32)(a >> 32) == NIL;                                              // reached the end: r is on the one cycle
    if (ok) ok = row_symbol(f, r) == ascii_symbol(text[(u32)a]);
    if (!ok) atomicAdd(bad, 1ull);
}

// sequential LF walk from the row of suffix 0 (it holds '$'): step i must show T[N-1-i]; one thread, `steps` dependent
// steps -- the reference's own developer check (src/LFsearch.c:49-166), for texts beyond the list-ranking verifier's 2^32
__global__ void lf_walk_kernel(FmView f, const u8* __restrict__ tail, u64 steps, unsigned long long* __restrict__ bad) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    u64 r = f.dollar_row;
    unsigned long long nb = 0;
    for (u64 i = 0; i < steps; ++i) {
        if (row_symbol(f, r) != ascii_symbol(tail[steps - 1 - i])) ++nb;
        r = lf_of(f, r);
    }
    *bad = nb;
}

// pattern symbol: A, C, G, T in either case -> 0..3, anything else -> 4 (occurs nowhere)
__device__ __forceinline__ u32 pattern_symbol(u8 c) {
    switch (c & 0xDFu) {
        case 'A': return 0u;
        case 'C': return 1u;
        case 'G': return 2u;
        case 'T': return 3u;
        default: return 4u;
    }
}

// backward search of pats[lo .. hi): the rows [sp, ep) whose suffixes start with the pattern (empty when ep <= sp)
__device__ __forceinline__ void fm_range(const FmView& f, const u8* __restrict__ pats, u64 lo, u64 hi, u64& sp_out, u64& ep_out) {
    u64 sp = 0, ep = f.n;
    for (u64 i = hi; i > lo && sp < ep; --i) {
        const u32 c = pattern_symbol(pats[i - 1]);
        if (c > 3u) { sp = ep = 0; break; }
        sp = f.C[c] + occ_before(f, c, sp);
        ep = f.C[c] + (ep == f.n ? f.C[c + 1] - f.C[c] : occ_before(f, c, ep));
    }
    sp_out = sp;
    ep_out = ep > sp ? ep : sp;
}

// backward search of one pattern per thread (count only)
__global__ void __launch_bounds__(TPB) fm_count_kernel(FmView f, const u8* __restrict__ pats, const u64* __restrict__ offs, u64 m,
                                                      u64* __restrict__ counts) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= m) return;
    u64 sp, ep;
    fm_range(f, pats, offs[t], offs[t + 1], sp, ep);
    counts[t] = ep - sp;
}

// ---- sampled suffix array ----------------------------------------------------------------------------------------
// After the list ranking, row r is at text position SA[r] = (d(r) + 1) mod N (d = low half of its node).  Rows with
// SA[r] % rate == 0 are sampled: bits[w] = mask of the sampled rows of word w (low half) | sampled rows in words < w (high
// half), vals[] = their SA values in row order.  The '$' row (SA = 0) is always sampled, so an LF walk from any row reaches
// a sampled row within rate - 1 steps without wrapping around the text.
struct SaView {
    const u64* bits;
    const u32* vals;
    u32 rate;
};

__device__ __forceinline__ u64 block_exclusive_scan_u64(u64 v, u64* total, u64* smem /* 32 u64 */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        u64 w = lane < TPB / 32 ? smem[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u64 t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        smem[lane] = w;
    }
    __syncthreads();
    if (total) *total = smem[TPB / 32 - 1];
    return (warp ? smem[warp - 1] : 0) + inc - v;
}

// the sampled-row mask of word (first word of this warp) + lane; every warp covers 32 words = 1024 rows, one coalesced row
// per lane and step.  `bad` counts rows whose walk did not reach the end (LF is not one N-cycle).
__device__ __forceinline__ u32 sa_word_mask(const u64* __restrict__ node, u64 n, u64 w0, u32 rate, unsigned long long* bad) {
    const u32 lane = threadIdx.x & 31;
    u32 mine = 0, off_cycle = 0;
    for (u32 j = 0; j < 32; ++j) {
        const u64 r = (w0 + j) * 32 + lane;
        bool take = false;
        if (r < n) {
            const u64 a = node[r];
            if ((u32)(a >> 32) != NIL) ++off_cycle;
            const u64 pos = (u64)(u32)a + 1 == n ? 0 : (u64)(u32)a + 1;
            take = (pos & (rate - 1)) == 0;
        }
        const u32 m = __ballot_sync(0xffffffffu, take);
        if (lane == j) mine = m;
    }
    if (bad) {
        off_cycle = __reduce_add_sync(0xffffffffu, off_cycle);
        if (lane == 0 && off_cycle) atomicAdd(bad, (unsigned long long)off_cycle);
    }
    return mine;
}

// per block of TPB words: number of sampled rows; rows off the one cycle into *bad
__global__ void __launch_bounds__(TPB) sa_count_kernel(const u64* __restrict__ node, u64 n, u32 rate, u64* __restrict__ block_tot,
                                                      unsigned long long* __restrict__ bad) {
    __shared__ u64 sm[32];
    const u64 w0 = (u64)blockIdx.x * TPB + (threadIdx.x & ~31u);
    const u32 m = sa_word_mask(node, n, w0, rate, bad);
    u64 tot;
    block_exclusive_scan_u64(__popc(m), &tot, sm);
    if (threadIdx.x == 0) block_tot[blockIdx.x] = tot;
}

// exclusive scan of nb u64 (one block, sequential over chunks); the total goes to base[nb]
__global__ void __launch_bounds__(TPB) scan_u64_kernel(const u64* __restrict__ in, u64 nb, u64* __restrict__ base) {
    __shared__ u64 sm[32];
    u64 carry = 0;
    for (u64 b = 0; b < nb; b += TPB) {
        const u64 i = b + threadIdx.x;
        u64 tot;
        const u64 ex = block_exclusive_scan_u64(i < nb ? in[i] : 0, &tot, sm);
        if (i < nb) base[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) base[nb] = carry;
}

// bits[w] for every word, and the SA value of every sampled row at its rank
__global__ void __launch_bounds__(TPB) sa_write_kernel(const u64* __restrict__ node, u64 n, u64 nwords, u32 rate,
                                                      const u64* __restrict__ block_base, u64* __restrict__ bits,
                                                      u32* __restrict__ vals) {
    __shared__ u64 sm[32];
    const u32 lane = threadIdx.x & 31;
    const u64 w0 = (u64)blockIdx.x * TPB + (threadIdx.x & ~31u);
    const u32 m = sa_word_mask(node, n, w0, rate, nullptr);
    const u64 before = block_base[blockIdx.x] + block_exclusive_scan_u64(__popc(m), nullptr, sm);
    if (w0 + lane < nwords) bits[w0 + lane] = (before << 32) | m;
    for (u32 j = 0; j < 32; ++j) {
        const u32 mj = __shfl_sync(0xffffffffu, m, j);
        const u64 bj = __shfl_sync(0xffffffffu, before, j);
        if ((mj >> lane) & 1u) {
            const u64 a = node[(w0 + j) * 32 + lane];
            vals[bj + __popc(mj & ((1u << lane) - 1u))] = (u64)(u32)a + 1 == n ? 0u : (u32)a + 1u;
        }
    }
}

// SA[r]: LF steps from r until a sampled row, whose value plus the steps taken is the answer (at most rate - 1 steps)
__device__ __forceinline__ u64 sa_of(const FmView& f, const SaView& s, u64 r) {
    for (u32 steps = 0; steps < s.rate; ++steps) {
        const u64 b = s.bits[r >> 5];
        const u32 m = (u32)b, bit = 1u << (r & 31);
        if (m & bit) return (u64)s.vals[(b >> 32) + __popc(m & (bit - 1u))] + steps;
        r = lf_of(f, r);
    }
    return ~0ull;                                                                 // not reached for a sampled BWT
}

__global__ void __launch_bounds__(TPB) sa_lookup_kernel(FmView f, SaView s, const u64* __restrict__ rows, u64 m, u64* __restrict__ out) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t < m) out[t] = sa_of(f, s, rows[t]);
}

// per pattern: first row of its range and its hit count
__global__ void __launch_bounds__(TPB) fm_range_kernel(FmView f, const u8* __restrict__ pats, const u64* __restrict__ offs, u64 m,
                                                      u64* __restrict__ sp_out, u64* __restrict__ counts) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= m) return;
    u64 sp, ep;
    fm_range(f, pats, offs[t], offs[t + 1], sp, ep);
    sp_out[t] = sp;
    counts[t] = ep - sp;
}

// per block of TPB patterns: total hits
__global__ void __launch_bounds__(TPB) hit_count_kernel(const u64* __restrict__ counts, u64 m, u64* __restrict__ block_tot) {
    __shared__ u64 sm[32];
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    u64 tot;
    block_exclusive_scan_u64(t < m ? counts[t] : 0, &tot, sm);
    if (threadIdx.x == 0) block_tot[blockIdx.x] = tot;
}

// hit_offsets[t] = hits of the patterns before t; hit_offsets[m] = all hits
__global__ void __launch_bounds__(TPB) hit_offsets_kernel(const u64* __restrict__ counts, u64 m, const u64* __restrict__ block_base,
                                                         u64* __restrict__ hit_offsets) {
    __shared__ u64 sm[32];
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    const u64 v = t < m ? counts[t] : 0;
    const u64 ex = block_base[blockIdx.x] + block_exclusive_scan_u64(v, nullptr, sm);
    if (t < m) hit_offsets[t] = ex;
    if (t + 1 == m) hit_offsets[m] = ex + v;
}

// one thread per hit: its pattern by binary search over hit_offsets, then SA of row sp + j, in SA order
__global__ void __launch_bounds__(TPB) locate_kernel(FmView f, SaView s, const u64* __restrict__ hit_offsets, const u64* __restrict__ sp,
                                                    u64 m, u64 total, u64* __restrict__ positions) {
    const u64 h = (u64)blockIdx.x * TPB + threadIdx.x;
    if (h >= total) return;
    const u64 i = upper_bound_u64(hit_offsets, 0, m + 1, h) - 1;                 // last pattern whose hits start at or before h
    positions[h] = sa_of(f, s, sp[i] + (h - hit_offsets[i]));
}

FmView view_of(const debwt_ctx* c) {
    FmView f;
    f.bwt = c->d_bwt; f.spec = c->d_spec_bits; f.occ = c->d_occ; f.sharp = c->d_sharp_sorted;
    f.n_sharp = c->n_rec - 1; f.dollar_row = c->dollar_row; f.n = c->n;
    for (int i = 0; i < 6; ++i) f.C[i] = c->c_array[i];
    return f;
}

SaView sa_view_of(const debwt_ctx* c) { return SaView{c->d_sa_bits, c->d_sa_vals, c->sa_rate}; }

}  // namespace

void drop_samples(debwt_ctx* c) {
    if (c->d_sa_bits) cudaFree(c->d_sa_bits);
    if (c->d_sa_vals) cudaFree(c->d_sa_vals);
    c->d_sa_bits = nullptr; c->d_sa_vals = nullptr;
    c->sa_rate = 0;
}

void drop_index(debwt_ctx* c) {
    drop_samples(c);
    if (c->d_occ) cudaFree(c->d_occ);
    if (c->d_spec_bits) cudaFree(c->d_spec_bits);
    if (c->d_sharp_sorted) cudaFree(c->d_sharp_sorted);
    c->d_occ = nullptr; c->d_spec_bits = nullptr; c->d_sharp_sorted = nullptr;
    c->indexed = false;
}

}  // namespace debwt

using namespace debwt;

#define FAIL(msg)              \
    do {                       \
        debwt::set_error(msg); \
        return -1;             \
    } while (0)

extern "C" {

// sharp: the rows holding '#', ascending
static int index_build_with(debwt_ctx* c, std::vector<u64> sharp, u64 dollar_row) {
    cudaStream_t st = c->st;
    const u64 n = c->n, nwords = c->n_words, occ_len = (n >> 5) + 1;
    const u64 cnt = sharp.size();
    c->dollar_row = dollar_row;
    sharp.push_back(dollar_row);                                                  // all special rows: cnt + 1 entries
    drop_index(c);
    const u64 nb = (nwords + TPB - 1) / TPB;
    u32* d_tot = nullptr;
    u64 *d_base = nullptr, *d_totals = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->d_occ), (occ_len + 1) * 32));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->d_spec_bits), (nwords + 1) * 4));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->d_sharp_sorted), (cnt + 1) * 8));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_tot), nb * 16 + 16));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_base), nb * 32 + 64));
    d_totals = d_base + nb * 4;
    CUDA_TRY(cudaMemcpyAsync(c->d_sharp_sorted, sharp.data(), (cnt + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(c->d_spec_bits, 0, (nwords + 1) * 4, st));
    spec_bits_kernel<<<grid_for(cnt + 1), TPB, 0, st>>>(c->d_spec_bits, c->d_sharp_sorted, cnt + 1);
    occ_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(c->d_bwt, c->d_spec_bits, n, nwords, d_tot);
    occ_scan_kernel<<<1, 1024, 0, st>>>(d_tot, nb, d_base, d_totals);
    occ_write_kernel<<<(unsigned)nb, TPB, 0, st>>>(c->d_bwt, c->d_spec_bits, n, nwords, d_base, c->d_occ, occ_len);
    DEBWT_COUNT(4);
    u64 tot[4];
    CUDA_TRY(cudaMemcpyAsync(tot, d_totals, 32, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    cudaFree(d_tot);
    cudaFree(d_base);
    if (tot[0] + tot[1] + tot[2] + tot[3] + c->n_rec != n) FAIL("internal: base counts of the BWT do not add up to N");
    c->c_array[0] = 0;                                                            // src/collect#$.c:92-100
    c->c_array[1] = tot[0];
    c->c_array[2] = tot[0] + tot[1];
    c->c_array[3] = tot[0] + tot[1] + tot[2];
    c->c_array[4] = tot[0] + tot[1] + tot[2] + tot[3];                            // '#' rows
    c->c_array[5] = n - 1;                                                        // '$'
    c->indexed = true;
    return 0;
}

int debwt_index_build(debwt_ctx* c) {
    if (!c || !c->built) FAIL("no result: call debwt_build first");
    if (c->indexed) return 0;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->st;
    // separator rows: '#' rows sorted (src/insertCase3.c:84-95 writes them ascending), '$' row
    std::vector<u64> sharp(c->n_rec + 1);
    u32 cnt = 0;
    u64 dollar = 0;
    CUDA_TRY(cudaMemcpyAsync(&cnt, c->d_sharp_count, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&dollar, c->d_dollar, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(sharp.data(), c->d_sharp, (c->n_rec + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (cnt != c->n_rec - 1) FAIL("internal: wrong number of '#' rows");
    sharp.resize(cnt);
    std::sort(sharp.begin(), sharp.end());
    return index_build_with(c, std::move(sharp), dollar);
}

int debwt_index_sizes(const debwt_ctx* c, uint64_t* occ_rows) {
    if (!c || !c->indexed) FAIL("no index: call debwt_index_build first");
    if (occ_rows) *occ_rows = (c->n >> 5) + 1;
    return 0;
}

int debwt_index_copy(debwt_ctx* c, uint64_t* occ, uint64_t* c_array) {
    if (!c || !c->indexed) FAIL("no index: call debwt_index_build first");
    CUDA_TRY(cudaSetDevice(c->device));
    if (occ) CUDA_TRY(cudaMemcpyAsync(occ, c->d_occ, ((c->n >> 5) + 1) * 32, cudaMemcpyDeviceToHost, c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    if (c_array) for (int i = 0; i < 6; ++i) c_array[i] = c->c_array[i];
    return 0;
}

int debwt_index_count(debwt_ctx* c, const char* patterns, const uint64_t* offsets, uint64_t n_patterns, uint64_t* counts) {
    if (!c || !c->indexed) FAIL("no index: call debwt_index_build first");
    if (n_patterns == 0) return 0;
    CUDA_TRY(cudaSetDevice(c->device));
    u8* d_p = nullptr; u64 *d_o = nullptr, *d_c = nullptr;
    const u64 bytes = offsets[n_patterns];
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_p), bytes + 16));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_o), (n_patterns + 1) * 8));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_c), n_patterns * 8));
    CUDA_TRY(cudaMemcpyAsync(d_p, patterns, bytes, cudaMemcpyHostToDevice, c->st));
    CUDA_TRY(cudaMemcpyAsync(d_o, offsets, (n_patterns + 1) * 8, cudaMemcpyHostToDevice, c->st));
    fm_count_kernel<<<grid_for(n_patterns), TPB, 0, c->st>>>(view_of(c), d_p, d_o, n_patterns, d_c);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(counts, d_c, n_patterns * 8, cudaMemcpyDeviceToHost, c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    CUDA_TRY(cudaGetLastError());
    cudaFree(d_p); cudaFree(d_o); cudaFree(d_c);
    return 0;
}

// List ranking of the LF walk by pointer jumping (Wyllie), shared by the verifier and the SA sampler.  d_a, d_b: N u64 each;
// on return d_a holds the ranked list: for every row r the high half is NIL iff r's walk reached the end of the list, and
// the low half is then the number of LF steps from r to that end.  d_live: one u32 of device scratch.
static int rank_lf(cudaStream_t st, const FmView& f, u64*& d_a, u64*& d_b, u32* d_live) {
    const u64 n = f.n;
    lf_init_kernel<<<grid_for(n), TPB, 0, st>>>(f, d_a);
    DEBWT_COUNT(1);
    for (int rounds = 0; rounds < 34; ++rounds) {
        u32 live = 0;
        CUDA_TRY(cudaMemsetAsync(d_live, 0, 4, st));
        jump_kernel<<<grid_for(n), TPB, 0, st>>>(d_a, d_b, n, d_live);
        DEBWT_COUNT(1);
        CUDA_TRY(cudaMemcpyAsync(&live, d_live, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        std::swap(d_a, d_b);
        if (!live) break;
    }
    return 0;
}

static int verify_indexed(debwt_ctx* c, const void* d_text, uint64_t* n_bad_out, float* ms_out) {
    if (c->n >= 0xFFFFFFFFull) FAIL("verify: N must be below 2^32 - 1");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->st;
    const u64 n = c->n;
    u64 *d_a = nullptr, *d_b = nullptr;
    u32* d_live = nullptr;
    unsigned long long* d_bad = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_a), n * 8) != cudaSuccess || cudaMalloc(reinterpret_cast<void**>(&d_b), n * 8) != cudaSuccess) {
        cudaGetLastError();
        if (d_a) cudaFree(d_a);
        FAIL("verify: not enough device memory for the list-ranking buffers (16 bytes per symbol)");
    }
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_live), 16));
    d_bad = reinterpret_cast<unsigned long long*>(d_live + 2);
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, st));
    const FmView f = view_of(c);
    if (rank_lf(st, f, d_a, d_b, d_live)) return -1;
    CUDA_TRY(cudaMemsetAsync(d_bad, 0, 8, st));
    lf_check_kernel<<<grid_for(n), TPB, 0, st>>>(f, d_a, static_cast<const u8*>(d_text), d_bad);
    DEBWT_COUNT(1);
    unsigned long long bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(e1, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d_a); cudaFree(d_b); cudaFree(d_live);
    if (n_bad_out) *n_bad_out = bad;
    if (ms_out) *ms_out = ms;
    return 0;
}

int debwt_verify_text_device(debwt_ctx* c, const void* d_text, uint64_t n_symbols, uint64_t* n_bad_out, float* ms_out) {
    if (!c || !c->built) FAIL("no result: call debwt_build first");
    if (n_symbols != c->n) FAIL("verify: text length differs from the build's");
    if (debwt_index_build(c)) return -1;
    return verify_indexed(c, d_text, n_bad_out, ms_out);
}

int debwt_verify_bwt_device(int device, const uint64_t* d_bwt_words, uint64_t n_symbols, const uint64_t* sharp_rows, uint64_t n_sharp,
                            uint64_t dollar_row, const void* d_text, uint64_t* n_bad_out, float* ms_out) {
    if (!d_bwt_words || !d_text || (n_sharp && !sharp_rows)) FAIL("null argument");
    if (debwt_device_count() <= device || device < 0) FAIL("no such CUDA device (this library has no CPU fallback)");
    CUDA_TRY(cudaSetDevice(device));
    debwt_ctx tmp;                                        // a view of the caller's buffers, nothing owned but the index
    tmp.device = device;
    CUDA_TRY(cudaStreamCreateWithFlags(&tmp.st, cudaStreamNonBlocking));
    tmp.n = n_symbols; tmp.n_rec = n_sharp + 1; tmp.n_words = (n_symbols + 31) / 32;
    tmp.d_bwt = reinterpret_cast<u64*>(const_cast<uint64_t*>(d_bwt_words));
    tmp.built = true;
    std::vector<u64> sharp(sharp_rows, sharp_rows + n_sharp);
    std::sort(sharp.begin(), sharp.end());
    CUDA_TRY(cudaDeviceSynchronize());                    // the caller's buffers may have been produced on another stream
    int rc = index_build_with(&tmp, std::move(sharp), dollar_row);
    if (!rc) rc = verify_indexed(&tmp, d_text, n_bad_out, ms_out);
    drop_index(&tmp);
    cudaStreamDestroy(tmp.st);
    return rc;
}

int debwt_verify_walk_device(int device, const uint64_t* d_bwt_words, uint64_t n_symbols, const uint64_t* sharp_rows, uint64_t n_sharp,
                             uint64_t dollar_row, const void* d_text_tail, uint64_t steps, uint64_t* n_bad_out, uint64_t* c_array_out) {
    if (!d_bwt_words || !d_text_tail || (n_sharp && !sharp_rows)) FAIL("null argument");
    if (steps > n_symbols) FAIL("verify: more steps than symbols");
    if (debwt_device_count() <= device || device < 0) FAIL("no such CUDA device (this library has no CPU fallback)");
    CUDA_TRY(cudaSetDevice(device));
    debwt_ctx tmp;
    tmp.device = device;
    CUDA_TRY(cudaStreamCreateWithFlags(&tmp.st, cudaStreamNonBlocking));
    tmp.n = n_symbols; tmp.n_rec = n_sharp + 1; tmp.n_words = (n_symbols + 31) / 32;
    tmp.d_bwt = reinterpret_cast<u64*>(const_cast<uint64_t*>(d_bwt_words));
    tmp.built = true;
    std::vector<u64> sharp(sharp_rows, sharp_rows + n_sharp);
    std::sort(sharp.begin(), sharp.end());
    CUDA_TRY(cudaDeviceSynchronize());
    int rc = index_build_with(&tmp, std::move(sharp), dollar_row);           // also checks that the base counts add up to N
    unsigned long long* d_bad = nullptr;
    if (!rc && cudaMalloc(reinterpret_cast<void**>(&d_bad), 8) != cudaSuccess) { cudaGetLastError(); set_error("out of device memory"); rc = -1; }
    if (!rc) {
        lf_walk_kernel<<<1, 32, 0, tmp.st>>>(view_of(&tmp), static_cast<const u8*>(d_text_tail), steps, d_bad);
        DEBWT_COUNT(1);
        unsigned long long bad = 0;
        if (cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, tmp.st) != cudaSuccess || cudaStreamSynchronize(tmp.st) != cudaSuccess) {
            set_error(std::string("verify walk: ") + cudaGetErrorString(cudaGetLastError()));
            rc = -1;
        }
        if (n_bad_out) *n_bad_out = bad;
        if (c_array_out) for (int i = 0; i < 6; ++i) c_array_out[i] = tmp.c_array[i];
    }
    if (d_bad) cudaFree(d_bad);
    drop_index(&tmp);
    cudaStreamDestroy(tmp.st);
    return rc;
}

int debwt_verify_text(debwt_ctx* c, const char* text, uint64_t n_symbols, uint64_t* n_bad_out, float* ms_out) {
    if (!c || !text) FAIL("null argument");
    CUDA_TRY(cudaSetDevice(c->device));
    u8* d_t = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_t), n_symbols + 16));
    CUDA_TRY(cudaMemcpy(d_t, text, n_symbols, cudaMemcpyHostToDevice));
    const int rc = debwt_verify_text_device(c, d_t, n_symbols, n_bad_out, ms_out);
    cudaFree(d_t);
    return rc;
}

int debwt_index_sample_sa(debwt_ctx* c, uint32_t rate, float* ms_out) {
    if (!c || !c->built) FAIL("no result: call debwt_build first");
    if (rate < 1 || rate > 1024 || (rate & (rate - 1))) FAIL("sample_sa: the rate must be a power of two from 1 to 1024");
    if (c->n >= 0xFFFFFFFFull)
        FAIL("sample_sa: N = " + std::to_string(c->n) + " symbols; the list ranking that samples the suffix array needs N below 2^32 - 1");
    if (debwt_index_build(c)) return -1;
    CUDA_TRY(cudaSetDevice(c->device));
    drop_samples(c);
    cudaStream_t st = c->st;
    const u64 n = c->n, nwords = (n + 31) / 32, nb = (nwords + TPB - 1) / TPB;
    u64 *d_a = nullptr, *d_b = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_a), n * 8) != cudaSuccess || cudaMalloc(reinterpret_cast<void**>(&d_b), n * 8) != cudaSuccess) {
        cudaGetLastError();
        if (d_a) cudaFree(d_a);
        FAIL("sample_sa: not enough device memory for the list-ranking buffers (16 bytes per symbol)");
    }
    // scratch: live flag, bad-row count, block totals (nb), their scan (nb + 1)
    u64* d_s = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_s), (2 * nb + 3) * 8) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(d_a); cudaFree(d_b);
        FAIL("sample_sa: out of device memory");
    }
    u32* d_live = reinterpret_cast<u32*>(d_s);
    unsigned long long* d_bad = reinterpret_cast<unsigned long long*>(d_s + 1);
    u64 *d_tot = d_s + 2, *d_base = d_s + 2 + nb;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto fail = [&](const std::string& msg) {
        cudaStreamSynchronize(st);
        cudaGetLastError();
        cudaFree(d_a); cudaFree(d_b); cudaFree(d_s);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        drop_samples(c);
        set_error(msg);
        return -1;
    };
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess || cudaEventRecord(e0, st) != cudaSuccess)
        return fail(std::string("sample_sa: ") + cudaGetErrorString(cudaGetLastError()));
    const FmView f = view_of(c);
    if (rank_lf(st, f, d_a, d_b, d_live)) return fail(debwt_last_error());
    if (cudaMemsetAsync(d_bad, 0, 8, st) != cudaSuccess) return fail(std::string("sample_sa: ") + cudaGetErrorString(cudaGetLastError()));
    sa_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_a, n, rate, d_tot, d_bad);
    scan_u64_kernel<<<1, TPB, 0, st>>>(d_tot, nb, d_base);
    DEBWT_COUNT(2);
    unsigned long long bad = 0;
    u64 n_samples = 0;
    if (cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaMemcpyAsync(&n_samples, d_base + nb, 8, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
        return fail(std::string("sample_sa: ") + cudaGetErrorString(cudaGetLastError()));
    if (bad)
        return fail("sample_sa: the result is not a BWT: " + std::to_string(bad) + " of " + std::to_string(n) +
                    " rows are not on the one N-cycle of its LF mapping");
    if (n_samples != (n + rate - 1) / rate) return fail("internal: wrong number of sampled rows");
    if (cudaMalloc(reinterpret_cast<void**>(&c->d_sa_bits), nwords * 8) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&c->d_sa_vals), n_samples * 4) != cudaSuccess)
        return fail("sample_sa: out of device memory for the samples");
    sa_write_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_a, n, nwords, rate, d_base, c->d_sa_bits, c->d_sa_vals);
    DEBWT_COUNT(1);
    float ms = 0;
    if (cudaEventRecord(e1, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess ||
        cudaEventElapsedTime(&ms, e0, e1) != cudaSuccess)
        return fail(std::string("sample_sa: ") + cudaGetErrorString(cudaGetLastError()));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d_a); cudaFree(d_b); cudaFree(d_s);
    c->sa_rate = rate;
    c->n_sa_samples = n_samples;
    if (ms_out) *ms_out = ms;
    return 0;
}

int debwt_index_sa(debwt_ctx* c, const uint64_t* rows, uint64_t n_rows, uint64_t* positions) {
    if (!c || !c->indexed || !c->sa_rate) FAIL("no sampled suffix array: call debwt_index_sample_sa first");
    if (n_rows == 0) return 0;
    if (!rows || !positions) FAIL("null argument");
    for (u64 i = 0; i < n_rows; ++i)
        if (rows[i] >= c->n) FAIL("index_sa: row " + std::to_string(rows[i]) + " (argument " + std::to_string(i) + ") is not below N = " + std::to_string(c->n));
    CUDA_TRY(cudaSetDevice(c->device));
    u64* d = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d), n_rows * 16));
    CUDA_TRY(cudaMemcpyAsync(d, rows, n_rows * 8, cudaMemcpyHostToDevice, c->st));
    sa_lookup_kernel<<<grid_for(n_rows), TPB, 0, c->st>>>(view_of(c), sa_view_of(c), d, n_rows, d + n_rows);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(positions, d + n_rows, n_rows * 8, cudaMemcpyDeviceToHost, c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    CUDA_TRY(cudaGetLastError());
    cudaFree(d);
    return 0;
}

int debwt_index_locate(debwt_ctx* c, const char* patterns, const uint64_t* offsets, uint64_t n_patterns, uint64_t* hit_offsets,
                       uint64_t* positions, uint64_t positions_cap) {
    if (!c || !c->indexed || !c->sa_rate) FAIL("no sampled suffix array: call debwt_index_sample_sa first");
    if (!offsets || !hit_offsets || (n_patterns && !patterns)) FAIL("null argument");
    hit_offsets[0] = 0;
    if (n_patterns == 0) return 0;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->st;
    const u64 m = n_patterns, bytes = offsets[m], nb = (m + TPB - 1) / TPB;
    // one block: patterns | offsets (m + 1) | sp (m) | counts (m) | hit offsets (m + 1) | block totals (nb) | their scan (nb + 1)
    const u64 words = (bytes + 16 + 7) / 8;
    u64* d = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d), (words + 4 * m + 2 * nb + 3) * 8));
    u8* d_p = reinterpret_cast<u8*>(d);
    u64 *d_o = d + words, *d_sp = d_o + m + 1, *d_cnt = d_sp + m, *d_hit = d_cnt + m, *d_tot = d_hit + m + 1, *d_base = d_tot + nb;
    CUDA_TRY(cudaMemcpyAsync(d_p, patterns, bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_o, offsets, (m + 1) * 8, cudaMemcpyHostToDevice, st));
    const FmView f = view_of(c);
    fm_range_kernel<<<grid_for(m), TPB, 0, st>>>(f, d_p, d_o, m, d_sp, d_cnt);
    hit_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_cnt, m, d_tot);
    scan_u64_kernel<<<1, TPB, 0, st>>>(d_tot, nb, d_base);
    hit_offsets_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_cnt, m, d_base, d_hit);
    DEBWT_COUNT(4);
    CUDA_TRY(cudaMemcpyAsync(hit_offsets, d_hit, (m + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    const u64 total = hit_offsets[m];
    if (!positions || total == 0) { cudaFree(d); return 0; }                  // size query
    if (total > positions_cap) {
        cudaFree(d);
        FAIL("index_locate: the patterns have " + std::to_string(total) + " hits; positions holds " + std::to_string(positions_cap));
    }
    u64* d_pos = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_pos), total * 8) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(d);
        FAIL("index_locate: out of device memory for " + std::to_string(total) + " hits");
    }
    locate_kernel<<<grid_for(total), TPB, 0, st>>>(f, sa_view_of(c), d_hit, d_sp, m, total, d_pos);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(positions, d_pos, total * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    cudaFree(d); cudaFree(d_pos);
    return 0;
}

}  // extern "C"
