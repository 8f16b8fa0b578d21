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
#include <cmath>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "ctx.cuh"
#include "radix_sort.cuh"

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

// LF(r) for a row r whose symbol c = row_symbol(f, r) is already known
__device__ __forceinline__ u64 lf_with(const FmView& f, u64 r, u32 c) {
    if (c == 5u) return f.n - 1;                                                  // '$' is the largest suffix
    if (c == 4u) return f.C[4] + lower_bound_u64(f.sharp, 0, f.n_sharp, r);       // src/LFsearch.c:131
    return f.C[c] + occ_before(f, c, r);
}

__device__ __forceinline__ u64 lf_of(const FmView& f, u64 r) { return lf_with(f, r, row_symbol(f, r)); }

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

// ---- extract ------------------------------------------------------------------------------------------------------
// Inverse samples: isa[v / rate] = r for every sampled row r with SA[r] = v.  The samples are exactly the multiples of
// the rate below N, so every slot is written once; isa[0] is the '$' row.
__global__ void __launch_bounds__(TPB) isa_from_sa_kernel(SaView s, u64 n, u32* __restrict__ isa) {
    const u64 r = (u64)blockIdx.x * TPB + threadIdx.x;
    if (r >= n) return;
    const u64 b = s.bits[r >> 5];
    const u32 m = (u32)b, bit = 1u << (r & 31);
    if (m & bit) isa[s.vals[(b >> 32) + __popc(m & (bit - 1u))] >> (__ffs(s.rate) - 1)] = (u32)r;
}

// One thread per rate-aligned block q of interval i = [a, b): it writes T[lo, hi) with lo = max(a, q rate),
// hi = min(b, (q + 1) rate).  It starts in the row of suffix s = min((q + 1) rate, N) -- the sampled row isa[s / rate], or
// the '$' row when s = N (suffix N is suffix 0 cyclically) -- and each LF step reads the symbol before the current
// suffix, so it reads s - lo <= rate symbols to reach lo.  out_off[i] is where T[a] goes; b = a + out_off[i + 1] - out_off[i].
__global__ void __launch_bounds__(TPB) extract_kernel(FmView f, SaView s, const u32* __restrict__ isa, const u64* __restrict__ starts,
                                                     const u64* __restrict__ blk_off, const u64* __restrict__ out_off, u64 m,
                                                     u64 n_blocks, u8* __restrict__ out) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= n_blocks) return;
    const u64 i = upper_bound_u64(blk_off, 0, m + 1, t) - 1;                     // last interval whose blocks start at or before t
    const u32 sh = __ffs(s.rate) - 1;
    const u64 a = starts[i], b = a + (out_off[i + 1] - out_off[i]);
    const u64 q = (a >> sh) + (t - blk_off[i]);
    const u64 lo = max(a, q << sh), hi = min(b, (q + 1) << sh), top = min((q + 1) << sh, f.n);
    u8* o = out + out_off[i];                                                     // o[p - a] receives T[p]
    u64 r = top == f.n ? f.dollar_row : isa[top >> sh];
    for (u64 p = top - 1;; --p) {                                                 // r is the row of suffix p + 1
        const u32 c = row_symbol(f, r);
        if (p < hi) o[p - a] = (u8)"ACGT#$"[c];
        if (p == lo) break;
        r = lf_with(f, r, c);
    }
}

// ---- SMEM search (FMD-index, Li 2012) ----------------------------------------------------------------------------
// Over a text closed under reverse complement the rows of rc(P) are the reverse interval of P: a bi-interval (k, l, s)
// holds the rows [k, k + s) of P and [l, l + s) of rc(P).  Here '#' and '$' sort after T, so inside [l, l + s) the suffixes
// rc(P)T, rc(P)G, rc(P)C, rc(P)A come first, in that order, and rc(P)# / rc(P)$ last: the reverse starts need no sentinel
// term (BWA's bwt_extend has its sentinel first and does not carry over).

// counts of A, C, G, T in the rows < r: one 32-byte occ checkpoint, the BWT word and the '#'/'$' mask word
__device__ __forceinline__ void occ4_before(const FmView& f, u64 r, u64 o[4]) {
    const u64 w = r >> 5;
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(f.occ + w * 4);
    const ulonglong2 a = p[0], b = p[1];
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
    const u32 below = (1u << (r & 31)) - 1u;
    if (below) {                                                                  // r = N on a word edge reads no word
        const u64 x = f.bwt[w];
        const u32 ok = ~f.spec[w] & below;
#pragma unroll
        for (u32 c = 0; c < 4; ++c) o[c] += __popc(symbol_mask(x, c) & ok);
    }
}

__device__ __forceinline__ u64 pick4(const u64 v[4], u32 c) { return c == 0 ? v[0] : c == 1 ? v[1] : c == 2 ? v[2] : v[3]; }

struct BiIv {
    u64 k, l, s;   // rows [k, k + s) start with P, [l, l + s) with rc(P)
    u64 end;       // read position one past P
};

// P -> aP: k_a = C[a] + occ(a, k), s_a = occ(a, k + s) - occ(a, k); l_T = l, l_G = l_T + s_T, l_C = l_G + s_G, l_A = l_C + s_C
__device__ __forceinline__ BiIv backward_ext(const FmView& f, const BiIv& p, u32 a) {
    u64 lo[4], hi[4];
    occ4_before(f, p.k, lo);
    occ4_before(f, p.k + p.s, hi);
    u64 l = p.l;
#pragma unroll
    for (u32 c = 3; c > 0; --c)
        if (c > a) l += hi[c] - lo[c];
    const u64 k_a = (a == 0 ? f.C[0] : a == 1 ? f.C[1] : a == 2 ? f.C[2] : f.C[3]) + pick4(lo, a);
    return BiIv{k_a, l, pick4(hi, a) - pick4(lo, a), p.end};
}

// P -> Pa: backward extension of rc(P) by comp(a), starts swapped back
__device__ __forceinline__ BiIv forward_ext(const FmView& f, const BiIv& p, u32 a) {
    const BiIv r = backward_ext(f, BiIv{p.l, p.k, p.s, p.end}, 3u - a);
    return BiIv{r.l, r.k, r.s, p.end};
}

__device__ __forceinline__ u64 base_count(const FmView& f, u32 a) {                  // occurrences of base a (0 past T)
    return a > 3u ? 0 : (a == 0 ? f.C[1] - f.C[0] : a == 1 ? f.C[2] - f.C[1] : a == 2 ? f.C[3] - f.C[2] : f.C[4] - f.C[3]);
}

// the bi-interval of the one base a (count ca) at read position x
__device__ __forceinline__ BiIv single_base(const FmView& f, u32 a, u64 ca, u32 x) {
    return BiIv{a == 0 ? f.C[0] : a == 1 ? f.C[1] : a == 2 ? f.C[2] : f.C[3],
                a == 3 ? f.C[0] : a == 2 ? f.C[1] : a == 1 ? f.C[2] : f.C[3], ca, (u64)x + 1};
}

// Li's smem1 from q[x], a base a that occurs ca >= 1 times in T: BWA's bwt_smem1a(x, min_intv = t, max_intv = 0).  Every
// SMEM it finds goes to emit(interval, qbeg) by descending qbeg (qend = interval.end); returns the end of the longest match
// from x.  list0 / list1: the slot's two interval lists of list_cap entries, entry j at [j n_slots].
template <class Emit>
__device__ __forceinline__ u32 smem1(const FmView& f, const u8* __restrict__ q, u32 m, u32 x, u32 a, u64 ca, u64 t, BiIv* list0,
                                     BiIv* list1, u64 n_slots, u64 list_cap, Emit&& emit) {
    // forward from x: push the interval before each change of size, at the end of the read or before a non-ACGT;
    // pushed at descending entries of list 1 so that they read back longest-match first
    BiIv ik = single_base(f, a, ca, x);
    u64 top = list_cap;
    u32 i = x + 1;
    for (; i < m; ++i) {
        const u32 c = pattern_symbol(q[i]);
        if (c > 3u) { list1[--top * n_slots] = ik; break; }
        BiIv ok = forward_ext(f, ik, c);
        if (ok.s != ik.s) {
            list1[--top * n_slots] = ik;
            if (ok.s < t) break;
        }
        ik = ok;
        ik.end = (u64)i + 1;
    }
    if (i == m) list1[--top * n_slots] = ik;
    const BiIv* prev = list1 + top * n_slots;
    u64 n_prev = list_cap - top;
    const u32 ret = (u32)prev[0].end;
    // backward: extend every interval by q[i]; the first that falls below t ends an SMEM at i + 1 unless a longer one
    // ended there; equal sizes are kept once
    u32 last_beg = 0xFFFFFFFFu;
    BiIv* curr = list0;
    for (long long i2 = (long long)x - 1; i2 >= -1; --i2) {
        const u32 c = i2 < 0 ? 4u : pattern_symbol(q[i2]);
        u64 n_curr = 0, last_s = 0;
        for (u64 j = 0; j < n_prev; ++j) {
            const BiIv p = prev[j * n_slots];
            BiIv ok{0, 0, 0, 0};
            if (c < 4u) ok = backward_ext(f, p, c);
            if (ok.s < t) {
                const u32 beg = (u32)(i2 + 1);
                if (n_curr == 0 && beg < last_beg) {
                    last_beg = beg;
                    emit(p, beg);
                }
            } else if (n_curr == 0 || ok.s != last_s) {
                curr[n_curr++ * n_slots] = ok;
                last_s = ok.s;
            }
        }
        if (n_curr == 0) break;
        prev = curr;
        n_prev = n_curr;
        curr = curr == list0 ? list1 : list0;
    }
    return ret;
}

// One thread per scratch slot; slots take reads from the work counter `next`.  Slot t owns two interval lists of
// `list_cap` entries (the longest read + 1), entry j of list h at scratch[(h list_cap + j) n_slots + t], so that the
// threads of a warp that stand at the same entry touch neighbouring 32-byte entries.  Li's outer loop: x = 0; x = smem1(x)
// at A/C/G/T that occurs in T, x + 1 past any other symbol.  The count pass (out == nullptr) writes the number of SMEMs
// of at least min_len per read; the write pass writes them at out_off.
__global__ void __launch_bounds__(TPB) smem_kernel(FmView f, const u8* __restrict__ reads, const u64* __restrict__ offs, u64 n_reads,
                                                  u32 min_len, BiIv* __restrict__ scratch, u64 n_slots, u64 list_cap,
                                                  unsigned long long* __restrict__ next, u64* __restrict__ counts,
                                                  const u64* __restrict__ out_off, debwt_smem* __restrict__ out) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= n_slots) return;
    BiIv* const list0 = scratch + t;
    BiIv* const list1 = scratch + list_cap * n_slots + t;
    for (;;) {
        const u64 rd = atomicAdd(next, 1ull);
        if (rd >= n_reads) break;
        const u8* q = reads + offs[rd];
        const u32 m = (u32)(offs[rd + 1] - offs[rd]);
        debwt_smem* o = out ? out + out_off[rd] : nullptr;
        u64 n_out = 0;
        u32 x = 0;
        while (x < m) {
            const u32 a = pattern_symbol(q[x]);
            const u64 ca = base_count(f, a);
            if (ca == 0) { ++x; continue; }                                       // no match covers x
            const u64 first = n_out;
            x = smem1(f, q, m, x, a, ca, 1, list0, list1, n_slots, list_cap, [&](const BiIv& p, u32 beg) {
                if (p.end - beg >= min_len) {
                    if (o) o[n_out] = debwt_smem{p.k, p.l, p.s, beg, (u32)p.end};
                    ++n_out;
                }
            });
            if (o)                                                                // one smem1 call finds them by descending qbeg
                for (u64 lo = first, hi = n_out; lo + 1 < hi; ++lo, --hi) {
                    const debwt_smem tmp = o[lo];
                    o[lo] = o[hi - 1];
                    o[hi - 1] = tmp;
                }
        }
        if (!o) counts[rd] = n_out;
    }
}

// ---- BWA-MEM seed collection (mem_collect_intv) -----------------------------------------------------------------------
struct SeedParams {
    u32 min_len, max_occ;
    u64 split_len, split_width, max_mem_intv;
};

__device__ __forceinline__ bool seed_less(const debwt_seed& a, const debwt_seed& b) {
    return a.qbeg != b.qbeg ? a.qbeg < b.qbeg : a.qend != b.qend ? a.qend < b.qend : a.round < b.round;
}

// heapsort of one read's seeds into (qbeg, qend, round): O(n log n) in place; seeds with the same key are the same piece
// and bi-interval, so the order between them does not show
__device__ void sort_seeds(debwt_seed* a, u64 n) {
    auto sift = [&](u64 r, u64 end) {
        for (u64 ch; (ch = 2 * r + 1) < end; r = ch) {
            if (ch + 1 < end && seed_less(a[ch], a[ch + 1])) ++ch;
            if (!seed_less(a[r], a[ch])) return;
            const debwt_seed tmp = a[r]; a[r] = a[ch]; a[ch] = tmp;
        }
    };
    for (u64 r = n / 2; r-- > 0;) sift(r, n);
    for (u64 end = n; end-- > 1;) {
        const debwt_seed tmp = a[0]; a[0] = a[end]; a[end] = tmp;
        sift(0, end);
    }
}

// The three rounds of BWA-MEM's seeding per read, with the slots, lists and work counter of smem_kernel.  Round 1: Li's
// outer loop with t = 1, seeds of at least min_len; each one of at least split_len bases and at most split_width
// occurrences leaves (its middle << 32 | count) in the slot's `mids` list (entry j at [j n_slots]; one per qbeg, so at
// most the read's length).  Round 2: smem1(middle, count + 1) for each, seeds of at least min_len.  Round 3 (max_mem_intv
// > 0): from x, forward extension until the first piece [x, i + 1) of more than min_len bases with fewer than
// max_mem_intv occurrences, a seed if it occurs; on at i + 1 (also after a non-ACGT at i).  The count pass (out ==
// nullptr) writes the seeds and hits per read; the write pass writes the seeds at out_off, sorts them and gives each its
// first hit, also into seed_hit.
__global__ void __launch_bounds__(TPB) seed_kernel(FmView f, const u8* __restrict__ reads, const u64* __restrict__ offs, u64 n_reads,
                                                  SeedParams o, BiIv* __restrict__ scratch, u64* __restrict__ mids, u64 n_slots,
                                                  u64 list_cap, unsigned long long* __restrict__ next, u64* __restrict__ counts,
                                                  u64* __restrict__ hit_counts, const u64* __restrict__ out_off,
                                                  const u64* __restrict__ hit_off, debwt_seed* __restrict__ out,
                                                  u64* __restrict__ seed_hit) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= n_slots) return;
    BiIv* const list0 = scratch + t;
    BiIv* const list1 = scratch + list_cap * n_slots + t;
    u64* const mid = mids + t;
    for (;;) {
        const u64 rd = atomicAdd(next, 1ull);
        if (rd >= n_reads) break;
        const u8* q = reads + offs[rd];
        const u32 m = (u32)(offs[rd + 1] - offs[rd]);
        debwt_seed* w = out ? out + out_off[rd] : nullptr;
        u64 n = 0, hits = 0, n_mid = 0;
        auto put = [&](const BiIv& p, u32 beg, u32 end, u32 round) {
            const u32 nh = (u32)min(p.s, (u64)o.max_occ);
            if (w) w[n] = debwt_seed{p.k, p.l, p.s, beg, end, 0, nh, round};
            ++n;
            hits += nh;
        };
        for (u32 x = 0; x < m;) {                                                 // round 1
            const u32 a = pattern_symbol(q[x]);
            const u64 ca = base_count(f, a);
            if (ca == 0) { ++x; continue; }
            x = smem1(f, q, m, x, a, ca, 1, list0, list1, n_slots, list_cap, [&](const BiIv& p, u32 beg) {
                const u32 len = (u32)p.end - beg;
                if (len < o.min_len) return;
                put(p, beg, (u32)p.end, 1);
                if (len >= o.split_len && p.s <= o.split_width) mid[n_mid++ * n_slots] = ((u64)((beg + (u32)p.end) >> 1) << 32) | p.s;
            });
        }
        for (u64 j = 0; j < n_mid; ++j) {                                         // round 2
            const u64 v = mid[j * n_slots];
            const u32 x = (u32)(v >> 32), a = pattern_symbol(q[x]);
            smem1(f, q, m, x, a, base_count(f, a), (u64)(u32)v + 1, list0, list1, n_slots, list_cap, [&](const BiIv& p, u32 beg) {
                if ((u32)p.end - beg >= o.min_len) put(p, beg, (u32)p.end, 2);
            });
        }
        if (o.max_mem_intv > 0)                                                   // round 3
            for (u32 x = 0; x < m;) {
                const u32 a = pattern_symbol(q[x]);
                const u64 ca = base_count(f, a);
                if (ca == 0) { ++x; continue; }
                BiIv ik = single_base(f, a, ca, x);
                u32 next_x = m;
                for (u32 i = x + 1; i < m; ++i) {
                    const u32 c = pattern_symbol(q[i]);
                    if (c > 3u) { next_x = i + 1; break; }
                    if (ik.s) ik = forward_ext(f, ik, c);                         // an empty interval stays empty
                    if (ik.s < o.max_mem_intv && i - x >= o.min_len) {
                        if (ik.s) put(ik, x, i + 1, 3);
                        next_x = i + 1;
                        break;
                    }
                }
                x = next_x;
            }
        if (w) {
            sort_seeds(w, n);
            u64 h = hit_off[rd];
            for (u64 j = 0; j < n; ++j) {
                w[j].hit_begin = h;
                seed_hit[out_off[rd] + j] = h;
                h += w[j].n_hits;
            }
        } else {
            counts[rd] = n;
            hit_counts[rd] = hits;
        }
    }
}

// One thread per hit: its seed by binary search over seed_hit (n_seeds + 1 entries), then SA of row + j step (BWA's
// mem_chain sampling: step = count / max_occ when count > max_occ), then record, strand and forward offset from the R
// ascending separator positions `seps` of the both-strands text (records R / 2 .. R - 1 are the reverse copies).
__global__ void __launch_bounds__(TPB) seed_hits_kernel(FmView f, SaView s, const debwt_seed* __restrict__ seeds,
                                                       const u64* __restrict__ seed_hit, u64 n_seeds, u64 total, u32 max_occ,
                                                       const u64* __restrict__ seps, u64 R, debwt_seed_hit* __restrict__ out) {
    const u64 h = (u64)blockIdx.x * TPB + threadIdx.x;
    if (h >= total) return;
    const u64 i = upper_bound_u64(seed_hit, 0, n_seeds + 1, h) - 1;
    const debwt_seed sd = seeds[i];
    const u64 step = sd.count > max_occ ? sd.count / max_occ : 1;
    const u64 pos = sa_of(f, s, sd.row + (h - seed_hit[i]) * step);
    const u64 rec = lower_bound_u64(seps, 0, R, pos);                            // records that end before pos
    const u64 start = rec ? seps[rec - 1] + 1 : 0, off = pos - start, half = R / 2;
    const bool rev = rec >= half;
    out[h] = debwt_seed_hit{pos, rev ? seps[rec] - start - off - (sd.qend - sd.qbeg) : off, (u32)(rev ? rec - half : rec), rev ? 1u : 0u};
}

// ---- BWA-MEM seed chaining (mem_chain, mem_chain_flt) ----------------------------------------------------------------
struct ChainParams {
    long long w, max_chain_gap, max_chain_extend, min_seed_len;
    u32 min_chain_weight, max_occ;
    float mask_level, drop_ratio;
    u64 l_pac;
};

// One chain after the weight pass, at its ordinal in chain-set order: query span, weight, seeds, slot, bwa's first and kept
struct ChainRec {
    u32 beg, end, w, n, slot;
    int first;
    u32 kept;
};

// Per-hit scratch; a read with hits [hb, hb + H) owns entries [hb, hb + H) of each array (indices inside are read-local
// u32: a read's hits stay below 2^32, whose 24-byte hits alone would not fit the device) and bitmap words from
// hb / 64 + read, summary words from hb / 4096 + read.
struct ChainScratch {
    debwt_chain_seed* cs;   // hit h as a chain seed, in hit order
    u64* key;               // slot p: the p-th smallest (rbeg, hit) pair's rbeg; after chaining the filter's sort keys
    u32* idx;               // slot p: that pair's hit, the hit that creates the chain of slot p
    u32* nxt;               // hit h: the next seed of its chain (NIL at the end)
    u32* tail;              // slot p: the last seed of its chain
    u32* list;              // the filter's kept list
    ChainRec* rec;          // chains in chain-set order
    u64* bits;              // bit p: slot p holds a chain
    u64* summary;           // bit w: bitmap word w is not zero
};

// bwa's coordinate of a hit of `len` bases: F[r] + o forward, 2 l_pac - (F[r] + o + len) reverse (F[r] = seps[r-1] + 1 - r)
__device__ __forceinline__ u64 bwa_rbeg(const debwt_seed_hit& h, u32 len, const u64* __restrict__ seps, u64 l_pac) {
    const u64 f = (h.record ? seps[h.record - 1] + 1 - h.record : 0) + h.offset;
    return h.strand ? 2 * l_pac - (f + len) : f;
}

// heapsort of (key, idx) pairs by (key, idx); the pairs are distinct
__device__ void sort_pairs(u64* key, u32* idx, u64 n) {
    auto less = [&](u64 a, u64 b) { return key[a] != key[b] ? key[a] < key[b] : idx[a] < idx[b]; };
    auto swap = [&](u64 a, u64 b) {
        const u64 k = key[a]; key[a] = key[b]; key[b] = k;
        const u32 i = idx[a]; idx[a] = idx[b]; idx[b] = i;
    };
    auto sift = [&](u64 r, u64 end) {
        for (u64 ch; (ch = 2 * r + 1) < end; r = ch) {
            if (ch + 1 < end && less(ch, ch + 1)) ++ch;
            if (!less(r, ch)) return;
            swap(r, ch);
        }
    };
    for (u64 r = n / 2; r-- > 0;) sift(r, n);
    for (u64 end = n; end-- > 1;) {
        swap(0, end);
        sift(0, end);
    }
}

// heapsort of distinct u64 keys
__device__ void sort_keys(u64* a, u64 n) {
    auto sift = [&](u64 r, u64 end) {
        for (u64 ch; (ch = 2 * r + 1) < end; r = ch) {
            if (ch + 1 < end && a[ch] < a[ch + 1]) ++ch;
            if (a[r] >= a[ch]) return;
            const u64 t = a[r]; a[r] = a[ch]; a[ch] = t;
        }
    };
    for (u64 r = n / 2; r-- > 0;) sift(r, n);
    for (u64 end = n; end-- > 1;) {
        const u64 t = a[0]; a[0] = a[end]; a[end] = t;
        sift(0, end);
    }
}

__device__ __forceinline__ int top_bit(u64 x) { return 63 - __clzll((long long)x); }
__device__ __forceinline__ int low_bit(u64 x) { return __ffsll((long long)x) - 1; }

// the greatest occupied slot below x, or -1; bits / summary are the read's words
__device__ long long slot_before(const u64* __restrict__ bits, const u64* __restrict__ summary, u64 x) {
    if (x == 0) return -1;
    const u64 q = x - 1, w = q >> 6;
    const u64 m = bits[w] & (~0ull >> (63 - (q & 63)));
    if (m) return (long long)(w * 64 + top_bit(m));
    for (long long sw = (long long)(w >> 6), below = (long long)(w & 63); sw >= 0; --sw, below = 64) {
        const u64 s = summary[sw] & (below == 64 ? ~0ull : (1ull << below) - 1);
        if (s) {
            const u64 w2 = (u64)sw * 64 + top_bit(s);
            return (long long)(w2 * 64 + top_bit(bits[w2]));
        }
    }
    return -1;
}

// the least occupied slot at or above x (one exists)
__device__ u64 slot_from(const u64* __restrict__ bits, const u64* __restrict__ summary, u64 x) {
    const u64 w = x >> 6;
    const u64 m = bits[w] & (~0ull << (x & 63));
    if (m) return w * 64 + low_bit(m);
    for (u64 sw = w >> 6, from = (w & 63) + 1;; ++sw, from = 0) {
        const u64 s = from == 64 ? 0 : summary[sw] & (~0ull << from);
        if (s) {
            const u64 w2 = sw * 64 + low_bit(s);
            return w2 * 64 + low_bit(bits[w2]);
        }
    }
}

// One thread per read in flight, reads from the work counter `next`: the read's hits become chain seeds, its (rbeg, hit)
// pairs are sorted once, and a chain lives in the slot of the hit that created it, so `lower` is the chain of the first
// occupied slot of the rbeg group of the greatest occupied slot below upper_bound(rbeg).  Then the weights, the sort and
// bwa's filter.  Writes per read the kept chains and their seeds (for the scans), the chains after the weight pass and
// frac_rep; the chains and the filter's order stay in the scratch for chain_write_kernel.
__global__ void __launch_bounds__(TPB) chain_kernel(const u64* __restrict__ offs, u64 n_reads, const debwt_seed* __restrict__ seeds,
                                                   const u64* __restrict__ seed_off, const debwt_seed_hit* __restrict__ hits,
                                                   const u64* __restrict__ hit_off, const u64* __restrict__ seps, ChainParams o,
                                                   ChainScratch s, unsigned long long* __restrict__ next, u64* __restrict__ chain_cnt,
                                                   u64* __restrict__ seed_cnt, u32* __restrict__ n_sorted, float* __restrict__ frac) {
    for (;;) {
        const u64 rd = atomicAdd(next, 1ull);
        if (rd >= n_reads) break;
        const u64 hb = hit_off[rd], H = hit_off[rd + 1] - hb, len = offs[rd + 1] - offs[rd];
        const debwt_seed* sd = seeds + seed_off[rd];
        const u64 n_sd = seed_off[rd + 1] - seed_off[rd];
        // frac_rep: bwa's sweep over the seeds above max_occ
        u64 b = 0, e = 0, l_rep = 0;
        for (u64 j = 0; j < n_sd; ++j) {
            if (sd[j].count <= o.max_occ) continue;
            if (sd[j].qbeg > e) { l_rep += e - b; b = sd[j].qbeg; e = sd[j].qend; }
            else e = max(e, (u64)sd[j].qend);
        }
        l_rep += e - b;
        frac[rd] = len ? (float)l_rep / (float)len : 0.f;
        debwt_chain_seed* cs = s.cs + hb;
        u64* key = s.key + hb;
        u32 *idx = s.idx + hb, *nxt = s.nxt + hb, *tail = s.tail + hb;
        const debwt_seed_hit* ht = hits + hb;
        for (u64 j = 0, h = 0; j < n_sd; ++j) {
            const u32 l = sd[j].qend - sd[j].qbeg;
            for (u32 k = 0; k < sd[j].n_hits; ++k, ++h) {
                const u64 r = bwa_rbeg(ht[h], l, seps, o.l_pac);
                cs[h] = debwt_chain_seed{r, sd[j].qbeg, l};
                key[h] = r;
                idx[h] = (u32)h;
            }
        }
        sort_pairs(key, idx, H);
        const u64 nw = (H + 63) / 64;
        u64* bits = s.bits + hb / 64 + rd;
        u64* summary = s.summary + hb / 4096 + rd;
        for (u64 w = 0; w < nw; ++w) bits[w] = 0;
        for (u64 w = 0; w < (nw + 63) / 64; ++w) summary[w] = 0;
        // mem_chain
        for (u32 h = 0; h < H; ++h) {
            const debwt_chain_seed p = cs[h];
            const u64 lb = lower_bound_u64(key, 0, H, p.rbeg), ub = upper_bound_u64(key, lb, H, p.rbeg);
            const long long pred = slot_before(bits, summary, ub);
            bool merged = false;
            if (pred >= 0) {
                const u64 pk = key[pred];
                const u64 c = slot_from(bits, summary, pk == p.rbeg ? lb : lower_bound_u64(key, 0, (u64)pred, pk));
                const debwt_chain_seed first = cs[idx[c]], last = cs[tail[c]];
                if (ht[h].record == ht[idx[c]].record) {
                    if (p.qbeg >= first.qbeg && p.qbeg + p.len <= last.qbeg + last.len && p.rbeg >= first.rbeg &&
                        p.rbeg + p.len <= last.rbeg + last.len) {
                        merged = true;                                            // contained: not added
                    } else if (!((last.rbeg < o.l_pac || first.rbeg < o.l_pac) && p.rbeg >= o.l_pac)) {
                        const long long x = (long long)p.qbeg - (long long)last.qbeg, y = (long long)(p.rbeg - last.rbeg);
                        if (y >= 0 && x - y <= o.w && y - x <= o.w && x - (long long)last.len < o.max_chain_gap &&
                            y - (long long)last.len < o.max_chain_gap) {
                            nxt[tail[c]] = h;
                            nxt[h] = NIL;
                            tail[c] = h;
                            merged = true;
                        }
                    }
                }
            }
            if (!merged) {                                                        // a new chain in the slot of (rbeg, h)
                u64 lo = lb, hi = ub;
                while (lo < hi) {
                    const u64 mid = lo + ((hi - lo) >> 1);
                    if (idx[mid] < h) lo = mid + 1; else hi = mid;
                }
                bits[lo >> 6] |= 1ull << (lo & 63);
                summary[lo >> 12] |= 1ull << ((lo >> 6) & 63);
                tail[lo] = h;
                nxt[h] = NIL;
            }
        }
        // mem_chain_weight in chain-set order; chains below min_chain_weight are dropped
        ChainRec* rec = s.rec + hb;
        u32 nc = 0;
        for (u64 w = 0; w < nw; ++w)
            for (u64 m = bits[w]; m; m &= m - 1) {
                const u32 p = (u32)(w * 64 + low_bit(m));
                u64 qe = 0, re = 0, wq = 0, wr = 0;
                u32 n = 0;
                for (u32 h = idx[p]; h != NIL; h = nxt[h], ++n) {
                    const debwt_chain_seed q = cs[h];
                    wq += q.qbeg >= qe ? q.len : (q.qbeg + (u64)q.len > qe ? q.qbeg + (u64)q.len - qe : 0);
                    qe = max(qe, q.qbeg + (u64)q.len);
                    wr += q.rbeg >= re ? q.len : (q.rbeg + q.len > re ? q.rbeg + q.len - re : 0);
                    re = max(re, (u64)(q.rbeg + q.len));
                }
                const u32 wt = (u32)min(wq, wr);
                if (wt < o.min_chain_weight) continue;
                const debwt_chain_seed f = cs[idx[p]], l = cs[tail[p]];
                rec[nc] = ChainRec{f.qbeg, l.qbeg + l.len, wt, n, p, -1, 0};
                key[nc] = (u64)(0xFFFFFFFFu - wt) << 32 | nc;                   // weight descending, then chain-set order
                ++nc;
            }
        sort_keys(key, nc);
        // mem_chain_flt
        u32* list = s.list + hb;
        u64 n_list = 0;
        if (nc) {
            rec[(u32)key[0]].kept = 3;
            list[n_list++] = 0;
        }
        for (u32 i = 1; i < nc; ++i) {
            ChainRec& a = rec[(u32)key[i]];
            bool large = false;
            u64 k = 0;
            for (; k < n_list; ++k) {
                const u32 j = list[k];
                ChainRec& c = rec[(u32)key[j]];
                const u32 bm = max(a.beg, c.beg), em = min(a.end, c.end);
                if (em <= bm) continue;
                const long long min_l = min(a.end - a.beg, c.end - c.beg);
                if ((float)(em - bm) >= (float)min_l * o.mask_level && min_l < o.max_chain_gap) {
                    large = true;
                    if (c.first < 0) c.first = (int)i;
                    if ((float)a.w < (float)c.w * o.drop_ratio && (long long)c.w - (long long)a.w >= 2 * o.min_seed_len) break;
                }
            }
            if (k == n_list) {
                list[n_list++] = i;
                a.kept = large ? 2 : 3;
            }
        }
        for (u64 k = 0; k < n_list; ++k) {
            const int f = rec[(u32)key[list[k]]].first;
            if (f >= 0) rec[(u32)key[f]].kept = 1;
        }
        u32 i = 0;
        for (long long cnt = 0; i < nc; ++i) {
            const u32 kp = rec[(u32)key[i]].kept;
            if (kp == 0 || kp == 3) continue;
            if (++cnt >= o.max_chain_extend) break;
        }
        for (; i < nc; ++i)
            if (rec[(u32)key[i]].kept < 3) rec[(u32)key[i]].kept = 0;
        u64 kept = 0, kept_seeds = 0;
        for (u32 j = 0; j < nc; ++j) {
            const ChainRec& a = rec[(u32)key[j]];
            if (a.kept) { ++kept; kept_seeds += a.n; }
        }
        chain_cnt[rd] = kept;
        seed_cnt[rd] = kept_seeds;
        n_sorted[rd] = nc;
    }
}

// One thread per read: its kept chains in filter order at chain_off, their seeds (list order) at cseed_off
__global__ void __launch_bounds__(TPB) chain_write_kernel(u64 n_reads, const debwt_seed_hit* __restrict__ hits, const u64* __restrict__ hit_off,
                                                         ChainScratch s, const u32* __restrict__ n_sorted, const float* __restrict__ frac,
                                                         const u64* __restrict__ chain_off, const u64* __restrict__ cseed_off,
                                                         debwt_chain* __restrict__ chains, debwt_chain_seed* __restrict__ chain_seeds) {
    const u64 rd = (u64)blockIdx.x * TPB + threadIdx.x;
    if (rd >= n_reads) return;
    const u64 hb = hit_off[rd];
    const debwt_chain_seed* cs = s.cs + hb;
    const u64* key = s.key + hb;
    const u32 *idx = s.idx + hb, *nxt = s.nxt + hb;
    const ChainRec* rec = s.rec + hb;
    u64 o = chain_off[rd], so = cseed_off[rd];
    for (u32 i = 0; i < n_sorted[rd]; ++i) {
        const ChainRec a = rec[(u32)key[i]];
        if (!a.kept) continue;
        const u32 h0 = idx[a.slot];
        const debwt_seed_hit& ht = hits[hb + h0];
        chains[o++] = debwt_chain{cs[h0].rbeg, so, a.n, a.w, ht.record, ht.strand, a.kept, frac[rd]};
        for (u32 h = h0; h != NIL; h = nxt[h]) chain_seeds[so++] = cs[h];
    }
}

// ---- BWA-MEM seed extension (mem_flt_chained_seeds, mem_chain2aln) ------------------------------------------------
// bwa's pac from the index: one thread per rate-aligned block of the forward half T[0, fwd_end) (records 0 .. R/2 - 1),
// walking LF from a sampled row as extract_kernel does.  Base T[p] goes to pac index p - (separators before p); `below`
// counts the separators at or before the current p.  Blocks share boundary words, so words are merged with atomicOr.
__global__ void __launch_bounds__(TPB) pac_kernel(FmView f, SaView s, const u32* __restrict__ isa, const u64* __restrict__ seps, u64 R,
                                                 u64 fwd_end, u64 n_blocks, u32* __restrict__ pac) {
    const u64 q = (u64)blockIdx.x * TPB + threadIdx.x;
    if (q >= n_blocks) return;
    const u32 sh = __ffs(s.rate) - 1;
    const u64 lo = q << sh, hi = min(fwd_end, (q + 1) << sh), top = min((q + 1) << sh, f.n);
    u64 r = top == f.n ? f.dollar_row : isa[top >> sh];
    u64 below = upper_bound_u64(seps, 0, R, top - 1);
    u64 word = ~0ull;
    u32 acc = 0;
    for (u64 p = top - 1;; --p) {                                                 // r is the row of suffix p + 1
        const u32 c = row_symbol(f, r);
        if (c >= 4) {
            --below;
        } else if (p < hi) {
            const u64 x = p - below;
            if (x >> 4 != word) {
                if (acc) atomicOr(pac + word, acc);
                word = x >> 4;
                acc = 0;
            }
            acc |= c << (2 * (x & 15));
        }
        if (p == lo) break;
        r = lf_with(f, r, c);
    }
    if (acc) atomicOr(pac + word, acc);
}

struct ExtParams {
    int a, b, o_del, e_del, o_ins, e_ins, pen_clip5, pen_clip3, zdrop, w, min_chain_weight;
    u32 ring;               // int2 entries per warp: the DP window of the widest band, and seed SW's 199 columns
    u64 l_pac;
};

// Per chain seed (indexed as chain_seeds): the seeds a chain keeps after mem_flt_chained_seeds with their scores, bwa's
// srt, and the read's region slots (a read has at most as many regions as chain seeds); per chain: its kept seeds.
struct ExtScratch {
    debwt_chain_seed* fs;
    int* sc;
    u64* srt;
    debwt_region* reg;
    u32* fn;
};

struct ExtOut {
    int score, qle, tle, gtle, gscore, max_off;
};

constexpr int EXT_WARPS = 4;
constexpr int kMaxExtW = 1024;          // widest w: a retry's band w << 1 needs 2 (w << 1) + 3 ring entries per warp
constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr long long NEG = -(1ll << 62);

__device__ __forceinline__ u32 nt4(u8 c) {
    const u32 l = c | 0x20u;
    return l == 'a' ? 0u : l == 'c' ? 1u : l == 'g' ? 2u : l == 't' ? 3u : 4u;
}

__device__ __forceinline__ u32 ref_base(const u32* __restrict__ pac, u64 l_pac, u64 x) {
    const u64 y = x < l_pac ? x : 2 * l_pac - 1 - x;
    const u32 v = (pac[y >> 4] >> (2 * (y & 15))) & 3u;
    return x < l_pac ? v : 3u - v;
}

__device__ __forceinline__ int cal_max_gap(const ExtParams& o, int qlen) {
    const int l_del = (int)((double)(qlen * o.a - o.o_del) / o.e_del + 1.);
    const int l_ins = (int)((double)(qlen * o.a - o.o_ins) / o.e_ins + 1.);
    const int l = max(max(l_del, l_ins), 1);
    return min(l, o.w << 1);
}

__device__ __forceinline__ long long warp_incl_max(long long v, u32 lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long u = __shfl_up_sync(FULL, v, d);
        if ((int)lane >= d) v = max(v, u);
    }
    return v;
}

// ksw_extend2 for one warp: rows i over the target, lanes over 32 columns j of the query at a time.  In a row, M and E
// of a column need only that column, and F is a max-plus prefix scan: F(j) = max over beg <= k < j of
// max(M_k - oe_ins, 0) - (j - 1 - k) e_ins.  Every column row i touches lies in [i - w, i + w + 1] and beg never
// decreases, so `ring` (2 w + 3 entries or more) holds bwa's eh array; a column above `top` was never written and still
// has its row-0 value.
template <class Q, class T>
__device__ ExtOut warp_extend(const ExtParams& o, int qlen, Q qsym, int tlen, T tsym, int w, int end_bonus, int h0, int2* ring, u32 lane) {
    const int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins, RS = (int)o.ring;
    const int max_ins = max((int)((double)(qlen * o.a + end_bonus - o.o_ins) / o.e_ins + 1.), 1);
    const int max_del = max((int)((double)(qlen * o.a + end_bonus - o.o_del) / o.e_del + 1.), 1);
    w = min(w, min(max_ins, max_del));
    auto row0 = [&](int j) -> int {
        if (j == 0) return h0;
        if (h0 <= oe_ins) return 0;
        const long long v = (long long)h0 - oe_ins - (long long)(j - 1) * o.e_ins;
        return v > 0 ? (int)v : 0;
    };
    int beg = 0, end = qlen, mx = h0, max_i = -1, max_j = -1, max_ie = -1, gscore = -1, max_off = 0, top = -1;
    for (int i = 0; i < tlen; ++i) {
        beg = max(beg, i - w);
        end = min(min(end, i + w + 1), qlen);
        int h1 = 0;
        if (beg == 0) {
            const long long v = (long long)h0 - (o.o_del + (long long)o.e_del * (i + 1));
            h1 = v > 0 ? (int)v : 0;
        }
        const u32 tb = tsym(i);
        long long P = NEG;                                                        // max of M'_k + k e_ins over earlier chunks
        int hc = h1;                                                              // H(i, c - 1)
        unsigned long long best = 0;                                              // (m, mj) with the last j reaching m
        bool any = false;
        int first_nz = -1, last_nz = -1;
        for (int c = beg; c < end; c += 32) {
            const int j = c + (int)lane;
            const bool act = j < end;
            int ho = 0, eo = 0;
            u32 qs = 4;
            if (act) {
                if (j > top) ho = row0(j);
                else { const int2 v = ring[j % RS]; ho = v.x; eo = v.y; }
                qs = qsym(j);
            }
            const int M = ho ? ho + (qs > 3 ? -1 : qs == tb ? o.a : -o.b) : 0;
            const long long v = warp_incl_max(act ? (long long)max(M - oe_ins, 0) + (long long)j * o.e_ins : NEG, lane);
            long long ex = __shfl_up_sync(FULL, v, 1);
            ex = max(lane ? ex : NEG, P);
            const int f = j == beg ? 0 : (int)(ex - (long long)(j - 1) * o.e_ins);
            const int h = max(max(M, eo), f);
            int hp = __shfl_up_sync(FULL, h, 1);
            if (lane == 0) hp = hc;
            const int en = max(eo - o.e_del, max(M - oe_del, 0));
            const u32 nz = __ballot_sync(FULL, act && (hp || en));
            if (nz) {
                if (first_nz < 0) first_nz = c + __ffs(nz) - 1;
                last_nz = c + 31 - __clz(nz);
            }
            unsigned long long key = act ? ((unsigned long long)(u32)h << 32 | (u32)j) : 0ull;
#pragma unroll
            for (int d = 16; d; d >>= 1) key = max(key, __shfl_xor_sync(FULL, key, d));
            best = max(best, key);
            any = true;
            if (act) ring[j % RS] = make_int2(hp, en);
            const int last = min(end - c, 32) - 1;
            hc = __shfl_sync(FULL, h, last);
            P = max(P, __shfl_sync(FULL, v, last));
            __syncwarp();
        }
        if (lane == 0) ring[end % RS] = make_int2(hc, 0);
        __syncwarp();
        top = max(top, end);
        if (max(beg, end) == qlen) {
            max_ie = gscore > hc ? max_ie : i;
            gscore = max(gscore, hc);
        }
        const int m = any ? (int)(best >> 32) : 0, mj = any ? (int)(u32)best : -1;
        if (m == 0) break;
        if (m > mx) {
            mx = m; max_i = i; max_j = mj;
            max_off = max(max_off, abs(mj - i));
        } else if (o.zdrop > 0) {
            const long long di = i - max_i, dj = mj - max_j;
            if (di > dj) {
                if (mx - m - (di - dj) * o.e_del > o.zdrop) break;
            } else if (mx - m - (dj - di) * o.e_ins > o.zdrop) break;
        }
        const int nb = first_nz >= 0 ? first_nz : end;
        const int lj = hc ? end : last_nz >= 0 ? last_nz : nb - 1;
        beg = nb;
        end = min(lj + 2, qlen);
    }
    return ExtOut{mx, max_j + 1, max_i + 1, max_ie + 1, gscore, max_off};
}

// ksw_align2's score for one warp: Gotoh local alignment, rows over the target, lanes over the query.  buf[j] holds
// (H(i - 1, j), E(i, j)).  Opening a gap from an H that came from F is never better than extending F, so F is again a
// prefix scan, over G = max(M, E, 0): F(j) = max(0, max over k < j of G_k - oe_ins - (j - 1 - k) e_ins).
template <class Q, class T>
__device__ int warp_seed_sw(const ExtParams& o, int qlen, Q qsym, int tlen, T tsym, int2* buf, u32 lane) {
    const int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins;
    for (int j = (int)lane; j < qlen; j += 32) buf[j] = make_int2(0, 0);
    __syncwarp();
    int best = 0;
    for (int i = 0; i < tlen; ++i) {
        const u32 tb = tsym(i);
        int hd = 0;
        long long P = NEG;
        for (int c = 0; c < qlen; c += 32) {
            const int j = c + (int)lane;
            const bool act = j < qlen;
            const int2 v = act ? buf[j] : make_int2(0, 0);
            const u32 qs = act ? qsym(j) : 4;
            int hdiag = __shfl_up_sync(FULL, v.x, 1);
            if (lane == 0) hdiag = hd;
            const int G = max(max(hdiag + (qs > 3 ? -1 : qs == tb ? o.a : -o.b), v.y), 0);
            const long long u = warp_incl_max(act ? (long long)G - oe_ins + (long long)j * o.e_ins : NEG, lane);
            long long ex = __shfl_up_sync(FULL, u, 1);
            ex = max(lane ? ex : NEG, P);
            const int H = max(G, (int)max(0ll, ex - (long long)(j - 1) * o.e_ins));
            if (act) {
                best = max(best, H);
                buf[j] = make_int2(H, max(max(v.y - o.e_del, H - oe_del), 0));
            }
            const int last = min(qlen - c, 32) - 1;
            hd = __shfl_sync(FULL, v.x, last);
            P = max(P, __shfl_sync(FULL, u, last));
            __syncwarp();
        }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) best = max(best, __shfl_xor_sync(FULL, best, d));
    return best;
}

// bns_fetch_seq's clip of [beg, end) to the record `rec` on the strand of mid; F(r) = seps[r - 1] + 1 - r
__device__ __forceinline__ void clip_to_record(const u64* __restrict__ seps, u64 l_pac, u32 rec, long long mid, long long& beg, long long& end) {
    const long long start = rec ? (long long)seps[rec - 1] + 1 : 0;
    long long fb = start - rec, fe = fb + ((long long)seps[rec] - start);
    if (mid >= (long long)l_pac) {
        const long long t = fb;
        fb = 2 * (long long)l_pac - fe;
        fe = 2 * (long long)l_pac - t;
    }
    beg = max(beg, fb);
    end = min(end, fe);
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    return v;
}

// One warp per read in flight, reads from the work counter `next`: mem_flt_chained_seeds over the read's kept chains,
// then mem_chain2aln chain by chain.  Every lane runs the read's control flow (it depends only on values all lanes
// read alike); lanes split the DP rows, the containment and overlap tests and seedcov; lane 0 writes.  The regions go
// to the read's slots from its first chain seed on; reg_cnt[rd] receives their number.
__global__ void __launch_bounds__(EXT_WARPS * 32) ext_kernel(const u8* __restrict__ reads, const u64* __restrict__ offs, u64 n_reads,
                                                            const debwt_chain* __restrict__ chains, const u64* __restrict__ chain_off,
                                                            const debwt_chain_seed* __restrict__ cseeds, const u64* __restrict__ cseed_off,
                                                            const u32* __restrict__ pac, const u64* __restrict__ seps, ExtParams o,
                                                            ExtScratch s, unsigned long long* __restrict__ next, u64* __restrict__ reg_cnt) {
    extern __shared__ int2 ext_smem[];
    const u32 lane = threadIdx.x & 31;
    int2* ring = ext_smem + (threadIdx.x >> 5) * o.ring;
    const long long l_pac = (long long)o.l_pac;
    for (;;) {
        unsigned long long rd = 0;
        if (lane == 0) rd = atomicAdd(next, 1ull);
        rd = __shfl_sync(FULL, rd, 0);
        if (rd >= n_reads) break;
        const u8* q = reads + offs[rd];
        const int L = (int)(offs[rd + 1] - offs[rd]);
        const u64 c0 = chain_off[rd], c1 = chain_off[rd + 1], sb = cseed_off[rd];
        // mem_flt_chained_seeds
        const double min_l = o.min_chain_weight ? (double)(1.1f * (float)o.min_chain_weight) : (double)5.5f * log((double)L);
        const int min_hsp = (int)(o.a * min_l + .499);
        const bool flt = !(min_l > (double)(0.05f * (float)L));
        for (u64 ci = c0; ci < c1; ++ci) {
            const debwt_chain ch = chains[ci];
            const debwt_chain_seed* sd = cseeds + ch.seed_begin;
            u32 k = 0;
            for (u32 j = 0; j < ch.n_seeds; ++j) {
                const debwt_chain_seed t = sd[j];
                int sc = (int)t.len;
                if (flt) {
                    sc = -1;
                    if (t.len < 200) {
                        const long long rbeg = (long long)t.rbeg;
                        const long long qb = max((long long)t.qbeg - 50, 0ll), qe = min((long long)t.qbeg + t.len + 50, (long long)L);
                        long long rb = max(rbeg - 50, 0ll), re = min(rbeg + t.len + 50, 2 * l_pac);
                        const long long mid = (rbeg + rbeg + t.len) >> 1;
                        if (rb < l_pac && l_pac < re) {
                            if (mid < l_pac) re = l_pac;
                            else rb = l_pac;
                        }
                        if (qe - qb < 200 && re - rb < 200) {
                            clip_to_record(seps, o.l_pac, ch.record, mid, rb, re);
                            sc = warp_seed_sw(o, (int)(qe - qb), [&](int x) { return nt4(q[qb + x]); }, (int)(re - rb),
                                              [&](int y) { return ref_base(pac, o.l_pac, (u64)(rb + y)); }, ring, lane);
                        }
                    }
                    if (sc >= 0 && sc < min_hsp) continue;
                    if (sc < 0) sc = (int)t.len * o.a;
                }
                if (lane == 0) {
                    s.fs[ch.seed_begin + k] = t;
                    s.sc[ch.seed_begin + k] = sc;
                }
                ++k;
            }
            if (lane == 0) s.fn[ci] = k;
        }
        __syncwarp();
        // mem_chain2aln
        u32 n_reg = 0;
        debwt_region* reg = s.reg + sb;
        for (u64 ci = c0; ci < c1; ++ci) {
            const debwt_chain ch = chains[ci];
            const u32 n = s.fn[ci];
            if (n == 0) continue;
            const debwt_chain_seed* S = s.fs + ch.seed_begin;
            u64* srt = s.srt + ch.seed_begin;
            long long rmax0 = 2 * l_pac, rmax1 = 0;
            for (u32 i = 0; i < n; ++i) {
                const debwt_chain_seed t = S[i];
                const int r = L - (int)(t.qbeg + t.len);
                rmax0 = min(rmax0, (long long)t.rbeg - (t.qbeg + cal_max_gap(o, (int)t.qbeg)));
                rmax1 = max(rmax1, (long long)t.rbeg + t.len + (r + cal_max_gap(o, r)));
            }
            rmax0 = max(rmax0, 0ll);
            rmax1 = min(rmax1, 2 * l_pac);
            if (rmax0 < l_pac && l_pac < rmax1) {
                if ((long long)S[0].rbeg < l_pac) rmax1 = l_pac;
                else rmax0 = l_pac;
            }
            clip_to_record(seps, o.l_pac, ch.record, (long long)S[0].rbeg, rmax0, rmax1);
            if (lane == 0) {
                for (u32 i = 0; i < n; ++i) srt[i] = (u64)(u32)s.sc[ch.seed_begin + i] << 32 | i;
                sort_keys(srt, n);
            }
            __syncwarp();
            for (int k = (int)n - 1; k >= 0; --k) {
                const debwt_chain_seed sd = S[(u32)srt[k]];
                const long long srb = (long long)sd.rbeg;
                const int sq = (int)sd.qbeg, sl = (int)sd.len;
                bool covered = false;
                for (u32 i0 = 0; i0 < n_reg && !covered; i0 += 32) {
                    bool hit = false;
                    if (i0 + lane < n_reg) {
                        const debwt_region p = reg[i0 + lane];
                        const long long prb = (long long)p.rb, pre = (long long)p.re;
                        const int pqb = (int)p.qb, pqe = (int)p.qe, pw = (int)p.w;
                        if (!(srb < prb || srb + sl > pre || sq < pqb || sq + sl > pqe) && !(sl - (int)p.seedlen0 > .1 * L)) {
                            int qd = sq - pqb;
                            long long rd2 = srb - prb;
                            int wd = min(cal_max_gap(o, (int)min((long long)qd, rd2)), pw);
                            hit = qd - rd2 < wd && rd2 - qd < wd;
                            if (!hit) {
                                qd = pqe - (sq + sl);
                                rd2 = pre - (srb + sl);
                                wd = min(cal_max_gap(o, (int)min((long long)qd, rd2)), pw);
                                hit = qd - rd2 < wd && rd2 - qd < wd;
                            }
                        }
                    }
                    covered = __any_sync(FULL, hit);
                }
                if (covered) {
                    bool ov = false;
                    for (u32 i0 = (u32)k + 1; i0 < n && !ov; i0 += 32) {
                        bool hit = false;
                        const u32 i = i0 + lane;
                        if (i < n && srt[i] != 0) {
                            const debwt_chain_seed t = S[(u32)srt[i]];
                            const int tq = (int)t.qbeg, tl = (int)t.len;
                            const long long trb = (long long)t.rbeg;
                            if (!(tl < sl * .95))
                                hit = (sq <= tq && sq + sl - tq >= (sl >> 2) && (long long)(tq - sq) != trb - srb) ||
                                      (tq <= sq && tq + tl - sq >= (sl >> 2) && (long long)(sq - tq) != srb - trb);
                        }
                        ov = __any_sync(FULL, hit);
                    }
                    if (!ov) {
                        if (lane == 0) srt[k] = 0;
                        __syncwarp();
                        continue;
                    }
                }
                int aw0 = o.w, aw1 = o.w, score, truesc;
                long long qb, rb, qe, re;
                if (sq) {
                    ExtOut x{};
                    score = -1;
                    for (int t = 0; t < 2; ++t) {
                        const int prev = score;
                        aw0 = o.w << t;
                        x = warp_extend(o, sq, [&](int j) { return nt4(q[sq - 1 - j]); }, (int)(srb - rmax0),
                                        [&](int i) { return ref_base(pac, o.l_pac, (u64)(srb - 1 - i)); }, aw0, o.pen_clip5, sl * o.a, ring, lane);
                        score = x.score;
                        if (score == prev || x.max_off < (aw0 >> 1) + (aw0 >> 2)) break;
                    }
                    if (x.gscore <= 0 || x.gscore <= score - o.pen_clip5) {
                        qb = sq - x.qle; rb = srb - x.tle; truesc = score;
                    } else {
                        qb = 0; rb = srb - x.gtle; truesc = x.gscore;
                    }
                } else {
                    score = truesc = sl * o.a;
                    qb = 0; rb = srb;
                }
                if (sq + sl != L) {
                    const int sc0 = score, qe0 = sq + sl;
                    const long long re0 = srb + sl - rmax0;
                    ExtOut x{};
                    for (int t = 0; t < 2; ++t) {
                        const int prev = score;
                        aw1 = o.w << t;
                        x = warp_extend(o, L - qe0, [&](int j) { return nt4(q[qe0 + j]); }, (int)(rmax1 - rmax0 - re0),
                                        [&](int i) { return ref_base(pac, o.l_pac, (u64)(rmax0 + re0 + i)); }, aw1, o.pen_clip3, sc0, ring, lane);
                        score = x.score;
                        if (score == prev || x.max_off < (aw1 >> 1) + (aw1 >> 2)) break;
                    }
                    if (x.gscore <= 0 || x.gscore <= score - o.pen_clip3) {
                        qe = qe0 + x.qle; re = rmax0 + re0 + x.tle; truesc += score - sc0;
                    } else {
                        qe = L; re = rmax0 + re0 + x.gtle; truesc += x.gscore - sc0;
                    }
                } else {
                    qe = L; re = srb + sl;
                }
                int cov = 0;
                for (u32 i = lane; i < n; i += 32) {
                    const debwt_chain_seed t = S[i];
                    if ((long long)t.qbeg >= qb && (long long)t.qbeg + t.len <= qe && (long long)t.rbeg >= rb && (long long)t.rbeg + t.len <= re)
                        cov += (int)t.len;
                }
                cov = warp_sum(cov);
                if (lane == 0)
                    reg[n_reg] = debwt_region{(u64)rb, (u64)re, (u32)qb, (u32)qe, score, truesc, (u32)max(aw0, aw1), (u32)cov, (u32)sl,
                                              (u32)(ci - c0), ch.record, ch.strand, ch.frac_rep, 0};
                __syncwarp();
                ++n_reg;
            }
        }
        if (lane == 0) reg_cnt[rd] = n_reg;
    }
}

// One thread per read: its regions from its slots to reg_off
__global__ void __launch_bounds__(TPB) region_write_kernel(u64 n_reads, const u64* __restrict__ cseed_off, const debwt_region* __restrict__ slots,
                                                          const u64* __restrict__ reg_off, debwt_region* __restrict__ out) {
    const u64 rd = (u64)blockIdx.x * TPB + threadIdx.x;
    if (rd >= n_reads) return;
    const debwt_region* a = slots + cseed_off[rd];
    debwt_region* b = out + reg_off[rd];
    for (u64 i = 0, n = reg_off[rd + 1] - reg_off[rd]; i < n; ++i) b[i] = a[i];
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
    if (c->d_isa_vals) cudaFree(c->d_isa_vals);
    if (c->d_seps_sorted) cudaFree(c->d_seps_sorted);
    if (c->d_pac) cudaFree(c->d_pac);
    c->d_sa_bits = nullptr; c->d_sa_vals = nullptr; c->d_isa_vals = nullptr; c->d_seps_sorted = nullptr; c->d_pac = nullptr;
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

// The inverse samples, built from the SA samples the first time after sampling and kept with them
static int inverse_samples(debwt_ctx* c, const char* name) {
    if (c->d_isa_vals) return 0;
    if (cudaMalloc(reinterpret_cast<void**>(&c->d_isa_vals), c->n_sa_samples * 4) != cudaSuccess) {
        cudaGetLastError();
        c->d_isa_vals = nullptr;
        FAIL(std::string(name) + ": out of device memory for the inverse samples");
    }
    isa_from_sa_kernel<<<grid_for(c->n), TPB, 0, c->st>>>(sa_view_of(c), c->n, c->d_isa_vals);
    DEBWT_COUNT(1);
    return 0;
}

int debwt_index_extract(debwt_ctx* c, const uint64_t* starts, const uint64_t* ends, uint64_t n_intervals, char* out, uint64_t out_cap) {
    if (!c || !c->indexed || !c->sa_rate) FAIL("no sampled suffix array: call debwt_index_sample_sa first");
    if (n_intervals == 0) return 0;
    if (!starts || !ends) FAIL("null argument");
    const u64 m = n_intervals, n = c->n, rate = c->sa_rate;
    // what the device reads: starts (m) | block offsets (m + 1) | output offsets (m + 1)
    std::vector<u64> h(3 * m + 2);
    u64 *blk = h.data() + m, *off = blk + m + 1;
    blk[0] = off[0] = 0;
    for (u64 i = 0; i < m; ++i) {
        const u64 a = starts[i], b = ends[i];
        if (a > b || b > n)
            FAIL("index_extract: interval " + std::to_string(i) + " = [" + std::to_string(a) + ", " + std::to_string(b) +
                 ") does not satisfy 0 <= start <= end <= N = " + std::to_string(n));
        h[i] = a;
        blk[i + 1] = blk[i] + (b > a ? (b + rate - 1) / rate - a / rate : 0);
        off[i + 1] = off[i] + (b - a);
    }
    const u64 total = off[m], n_blocks = blk[m];
    if (total > out_cap)
        FAIL("index_extract: the intervals hold " + std::to_string(total) + " symbols; out holds " + std::to_string(out_cap));
    if (total == 0) return 0;
    if (!out) FAIL("null argument");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->st;
    if (inverse_samples(c, "index_extract")) return -1;
    u64* d = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d), h.size() * 8 + total) != cudaSuccess) {
        cudaGetLastError();
        FAIL("index_extract: out of device memory for " + std::to_string(total) + " symbols");
    }
    u64 *d_starts = d, *d_blk = d + m, *d_off = d_blk + m + 1;
    u8* d_out = reinterpret_cast<u8*>(d + h.size());
    CUDA_TRY(cudaMemcpyAsync(d, h.data(), h.size() * 8, cudaMemcpyHostToDevice, st));
    extract_kernel<<<grid_for(n_blocks), TPB, 0, st>>>(view_of(c), sa_view_of(c), c->d_isa_vals, d_starts, d_blk, d_off, m, n_blocks,
                                                       d_out);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(out, d_out, total, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    cudaFree(d);
    return 0;
}

static_assert(sizeof(debwt_smem) == 32, "debwt_smem is 3 u64 + 2 u32");
static_assert(sizeof(BiIv) == 32, "one scratch entry is one 32-byte sector");

// Scratch of the SMEM lists: each read in flight holds two lists of (longest read + 1) entries of 32 bytes
constexpr u64 kSmemScratchBytes = 1ull << 30;

int debwt_index_smem(debwt_ctx* c, const char* reads, const uint64_t* offsets, uint64_t n_reads, uint32_t min_len,
                     uint64_t* smem_offsets, debwt_smem* smems, uint64_t smems_cap) {
    if (!c || !c->indexed) FAIL("no index: call debwt_index_build first");
    if (!offsets || !smem_offsets || (n_reads && !reads)) FAIL("null argument");
    if (min_len == 0) FAIL("index_smem: min_len must be at least 1");
    const u64* C = c->c_array;
    const u64 nA = C[1] - C[0], nC = C[2] - C[1], nG = C[3] - C[2], nT = C[4] - C[3];
    if (nA != nT || nC != nG)
        FAIL("index_smem: the text is not closed under reverse complement: it holds A = " + std::to_string(nA) + ", C = " +
             std::to_string(nC) + ", G = " + std::to_string(nG) + ", T = " + std::to_string(nT) +
             " bases; build it from every record and its reverse complement (api.both_strands)");
    const u64 m = n_reads;
    u64 max_len = 0, longest = 0;
    for (u64 i = 0; i < m; ++i) {
        if (offsets[i + 1] < offsets[i]) FAIL("index_smem: offsets decrease at read " + std::to_string(i));
        if (offsets[i + 1] - offsets[i] > max_len) { max_len = offsets[i + 1] - offsets[i]; longest = i; }
    }
    const u64 list_cap = max_len + 1, slot_bytes = 2 * list_cap * sizeof(BiIv);
    if (slot_bytes > kSmemScratchBytes)
        FAIL("index_smem: read " + std::to_string(longest) + " has " + std::to_string(max_len) + " symbols; its interval lists need " +
             std::to_string(slot_bytes) + " bytes, more than the " + std::to_string(kSmemScratchBytes) + " bytes of scratch (reads up to " +
             std::to_string(kSmemScratchBytes / (2 * sizeof(BiIv)) - 1) + " symbols)");
    smem_offsets[0] = 0;
    if (m == 0) return 0;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->st;
    int sms = 0, per_sm = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    CUDA_TRY(cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxThreadsPerMultiProcessor, c->device));
    const u64 n_slots = std::min<u64>({(u64)sms * (u64)per_sm, kSmemScratchBytes / slot_bytes, m});
    const u64 bytes = offsets[m], nb = (m + TPB - 1) / TPB, words = (bytes + 16 + 7) / 8;
    // one block: reads | offsets (m + 1) | counts (m) | SMEM offsets (m + 1) | block totals (nb) | their scan (nb + 1) | counter
    u64* d = nullptr;
    BiIv* d_scratch = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d), (words + 3 * m + 2 * nb + 4) * 8));
    if (cudaMalloc(reinterpret_cast<void**>(&d_scratch), n_slots * slot_bytes) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(d);
        FAIL("index_smem: out of device memory for " + std::to_string(n_slots * slot_bytes) + " bytes of scratch");
    }
    u8* d_r = reinterpret_cast<u8*>(d);
    u64 *d_o = d + words, *d_cnt = d_o + m + 1, *d_off = d_cnt + m, *d_tot = d_off + m + 1, *d_base = d_tot + nb;
    unsigned long long* d_next = reinterpret_cast<unsigned long long*>(d_base + nb + 1);
    CUDA_TRY(cudaMemcpyAsync(d_r, reads, bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_o, offsets, (m + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(d_next, 0, 8, st));
    const FmView f = view_of(c);
    const unsigned grid = grid_for(n_slots);
    smem_kernel<<<grid, TPB, 0, st>>>(f, d_r, d_o, m, min_len, d_scratch, n_slots, list_cap, d_next, d_cnt, nullptr, nullptr);
    hit_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_cnt, m, d_tot);
    scan_u64_kernel<<<1, TPB, 0, st>>>(d_tot, nb, d_base);
    hit_offsets_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_cnt, m, d_base, d_off);
    DEBWT_COUNT(4);
    CUDA_TRY(cudaMemcpyAsync(smem_offsets, d_off, (m + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    const u64 total = smem_offsets[m];
    if (!smems || total == 0) { cudaFree(d); cudaFree(d_scratch); return 0; }   // size query
    if (total > smems_cap) {
        cudaFree(d); cudaFree(d_scratch);
        FAIL("index_smem: the reads have " + std::to_string(total) + " SMEMs; smems holds " + std::to_string(smems_cap));
    }
    debwt_smem* d_out = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_out), total * sizeof(debwt_smem)) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(d); cudaFree(d_scratch);
        FAIL("index_smem: out of device memory for " + std::to_string(total) + " SMEMs");
    }
    CUDA_TRY(cudaMemsetAsync(d_next, 0, 8, st));
    smem_kernel<<<grid, TPB, 0, st>>>(f, d_r, d_o, m, min_len, d_scratch, n_slots, list_cap, d_next, nullptr, d_off, d_out);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(smems, d_out, total * sizeof(debwt_smem), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    cudaFree(d); cudaFree(d_scratch); cudaFree(d_out);
    return 0;
}

static_assert(sizeof(debwt_seed) == 48, "debwt_seed is 3 u64 + 2 u32 + u64 + 2 u32");
static_assert(sizeof(debwt_seed_hit) == 24, "debwt_seed_hit is 2 u64 + 2 u32");

// The R separator positions of T, ascending, kept with the SA samples: SA of the rows [N - R, N), which hold the suffixes
// that start with '#' or '$', sorted on the device.
static int sorted_separators(debwt_ctx* c, const char* name) {
    if (c->d_seps_sorted) return 0;
    cudaStream_t st = c->st;
    const u64 R = c->n_rec, n = c->n;
    std::vector<u64> rows(R);
    for (u64 i = 0; i < R; ++i) rows[i] = n - R + i;
    u64 *d_a = nullptr, *d_b = nullptr;
    void* d_ws = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_a), (R + 2) * 8) != cudaSuccess || cudaMalloc(reinterpret_cast<void**>(&d_b), (R + 2) * 8) != cudaSuccess ||
        cudaMalloc(&d_ws, sort_workspace_bytes(R, c->sort_cfg)) != cudaSuccess) {
        cudaGetLastError();
        if (d_a) cudaFree(d_a);
        if (d_b) cudaFree(d_b);
        FAIL(std::string(name) + ": out of device memory for the separator positions");
    }
    SortWorkspace ws;
    sort_workspace_bind(ws, d_ws, R, c->sort_cfg);
    CUDA_TRY(cudaMemcpyAsync(d_b, rows.data(), R * 8, cudaMemcpyHostToDevice, st));
    sa_lookup_kernel<<<grid_for(R), TPB, 0, st>>>(view_of(c), sa_view_of(c), d_b, R, d_a);
    DEBWT_COUNT(1);
    u64* res = nullptr;
    const int rc = radix_sort_u64(d_a, d_b, R, ws, st, &res);
    if (!rc) CUDA_TRY(cudaStreamSynchronize(st));
    cudaFree(d_ws);
    cudaFree(res == d_a ? d_b : d_a);
    if (rc) { cudaFree(res ? res : d_a); return -1; }
    c->d_seps_sorted = res;
    return 0;
}

}  // extern "C"

// The device buffers of one seeding run, freed with it
struct SeedRun {
    u64* d = nullptr;                 // reads | offsets | seed counts | seed offsets | hit counts | hit offsets | block sums
    BiIv* scratch = nullptr;
    char* out = nullptr;              // the seeds | their first hits (total + 1) | the hits
    u64 *d_o = nullptr, *d_off = nullptr, *d_hoff = nullptr, *d_tot = nullptr, *d_base = nullptr;
    unsigned long long* d_next = nullptr;
    debwt_seed* seeds = nullptr;
    debwt_seed_hit* hits = nullptr;
    u64 total = 0, total_hits = 0;
    SeedRun() = default;
    SeedRun(const SeedRun&) = delete;
    ~SeedRun() {
        if (d) cudaFree(d);
        if (scratch) cudaFree(scratch);
        if (out) cudaFree(out);
    }
};

// The input checks of debwt_index_seeds after its NULL checks; `name` starts the messages.  max_len: the longest read.
static int check_seed_input(const debwt_ctx* c, const char* name, const uint64_t* offsets, u64 m, const debwt_seed_opts& op,
                            u64& max_len) {
    const std::string nm(name);
    if (op.min_seed_len == 0) FAIL(nm + ": min_seed_len must be at least 1");
    if (op.max_occ == 0) FAIL(nm + ": max_occ must be at least 1");
    if (!std::isfinite(op.split_factor) || op.split_factor < 0)
        FAIL(nm + ": split_factor must be finite and not negative, not " + std::to_string(op.split_factor));
    const u64* C = c->c_array;
    const u64 nA = C[1] - C[0], nC = C[2] - C[1], nG = C[3] - C[2], nT = C[4] - C[3];
    if (nA != nT || nC != nG)
        FAIL(nm + ": the text is not closed under reverse complement: it holds A = " + std::to_string(nA) + ", C = " +
             std::to_string(nC) + ", G = " + std::to_string(nG) + ", T = " + std::to_string(nT) +
             " bases; build it from every record and its reverse complement (api.both_strands)");
    if (c->n_rec % 2)
        FAIL(nm + ": the text holds " + std::to_string(c->n_rec) +
             " records; one built from every record and its reverse complement (api.both_strands) holds an even number");
    u64 longest = 0;
    max_len = 0;
    for (u64 i = 0; i < m; ++i) {
        if (offsets[i + 1] < offsets[i]) FAIL(nm + ": offsets decrease at read " + std::to_string(i));
        if (offsets[i + 1] - offsets[i] > max_len) { max_len = offsets[i + 1] - offsets[i]; longest = i; }
    }
    // per read in flight: two interval lists of len + 1 entries and the middles of the round-1 seeds to split (one per qbeg)
    const u64 slot_bytes = 2 * (max_len + 1) * sizeof(BiIv) + max_len * 8;
    if (slot_bytes > kSmemScratchBytes)
        FAIL(nm + ": read " + std::to_string(longest) + " has " + std::to_string(max_len) + " symbols; its interval lists need " +
             std::to_string(slot_bytes) + " bytes, more than the " + std::to_string(kSmemScratchBytes) + " bytes of scratch (reads up to " +
             std::to_string((kSmemScratchBytes - 2 * sizeof(BiIv)) / (2 * sizeof(BiIv) + 8)) + " symbols)");
    return 0;
}

// The seeding of debwt_index_seeds for m >= 1 checked reads, leaving everything in r: the count pass and the two scans
// (seed_offsets, when given, receives the seed offsets), then proceed(total seeds, total hits): 1 goes on to the write
// pass and the hit lookups, 0 stops there, -1 fails the call.
template <class Proceed>
static int run_seeds(debwt_ctx* c, const char* name, const char* reads, const uint64_t* offsets, u64 m, const debwt_seed_opts& op,
                     u64 max_len, uint64_t* seed_offsets, SeedRun& r, Proceed&& proceed) {
    const std::string nm(name);
    const u64 list_cap = max_len + 1, slot_bytes = 2 * list_cap * sizeof(BiIv) + max_len * 8;
    SeedParams prm;
    prm.min_len = op.min_seed_len;
    prm.max_occ = op.max_occ;
    const double split = (double)(op.min_seed_len * op.split_factor) + .499;    // bwa: (int)(min_seed_len * split_factor + .499)
    prm.split_len = split >= 18446744073709551615.0 ? ~0ull : (u64)split;
    prm.split_width = op.split_width;
    prm.max_mem_intv = op.max_mem_intv;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->st;
    int sms = 0, per_sm = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    CUDA_TRY(cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxThreadsPerMultiProcessor, c->device));
    const u64 n_slots = std::min<u64>({(u64)sms * (u64)per_sm, kSmemScratchBytes / slot_bytes, m});
    const u64 bytes = offsets[m], nb = (m + TPB - 1) / TPB, words = (bytes + 16 + 7) / 8;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&r.d), (words + 5 * m + 2 * nb + 5) * 8));
    if (cudaMalloc(reinterpret_cast<void**>(&r.scratch), n_slots * slot_bytes) != cudaSuccess) {
        cudaGetLastError();
        r.scratch = nullptr;
        FAIL(nm + ": out of device memory for " + std::to_string(n_slots * slot_bytes) + " bytes of scratch");
    }
    u64* d_mids = reinterpret_cast<u64*>(r.scratch + 2 * list_cap * n_slots);
    u8* d_r = reinterpret_cast<u8*>(r.d);
    r.d_o = r.d + words;
    u64 *d_cnt = r.d_o + m + 1, *d_hcnt;
    r.d_off = d_cnt + m;
    d_hcnt = r.d_off + m + 1;
    r.d_hoff = d_hcnt + m;
    r.d_tot = r.d_hoff + m + 1;
    r.d_base = r.d_tot + nb;
    r.d_next = reinterpret_cast<unsigned long long*>(r.d_base + nb + 1);
    CUDA_TRY(cudaMemcpyAsync(d_r, reads, bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(r.d_o, offsets, (m + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(r.d_next, 0, 8, st));
    const FmView f = view_of(c);
    const unsigned grid = grid_for(n_slots);
    seed_kernel<<<grid, TPB, 0, st>>>(f, d_r, r.d_o, m, prm, r.scratch, d_mids, n_slots, list_cap, r.d_next, d_cnt, d_hcnt, nullptr,
                                      nullptr, nullptr, nullptr);
    hit_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_cnt, m, r.d_tot);
    scan_u64_kernel<<<1, TPB, 0, st>>>(r.d_tot, nb, r.d_base);
    hit_offsets_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_cnt, m, r.d_base, r.d_off);
    hit_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_hcnt, m, r.d_tot);
    scan_u64_kernel<<<1, TPB, 0, st>>>(r.d_tot, nb, r.d_base);
    hit_offsets_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_hcnt, m, r.d_base, r.d_hoff);
    DEBWT_COUNT(7);
    if (seed_offsets) CUDA_TRY(cudaMemcpyAsync(seed_offsets, r.d_off, (m + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&r.total, r.d_off + m, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&r.total_hits, r.d_hoff + m, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    const int go = proceed(r.total, r.total_hits);
    if (go <= 0) return go;
    if (sorted_separators(c, name)) return -1;
    const u64 total = r.total, total_hits = r.total_hits;
    const u64 out_bytes = total * sizeof(debwt_seed) + (total + 1) * 8 + total_hits * sizeof(debwt_seed_hit);
    if (cudaMalloc(reinterpret_cast<void**>(&r.out), out_bytes) != cudaSuccess) {
        cudaGetLastError();
        r.out = nullptr;
        FAIL(nm + ": out of device memory for " + std::to_string(total) + " seeds and " + std::to_string(total_hits) + " hits");
    }
    r.seeds = reinterpret_cast<debwt_seed*>(r.out);
    u64* d_seed_hit = reinterpret_cast<u64*>(r.seeds + total);
    r.hits = reinterpret_cast<debwt_seed_hit*>(d_seed_hit + total + 1);
    CUDA_TRY(cudaMemcpyAsync(d_seed_hit + total, r.d_hoff + m, 8, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemsetAsync(r.d_next, 0, 8, st));
    seed_kernel<<<grid, TPB, 0, st>>>(f, d_r, r.d_o, m, prm, r.scratch, d_mids, n_slots, list_cap, r.d_next, nullptr, nullptr, r.d_off,
                                      r.d_hoff, r.seeds, d_seed_hit);
    seed_hits_kernel<<<grid_for(total_hits), TPB, 0, st>>>(f, sa_view_of(c), r.seeds, d_seed_hit, total, total_hits, op.max_occ,
                                                           c->d_seps_sorted, c->n_rec, r.hits);
    DEBWT_COUNT(2);
    return 1;
}

extern "C" {

int debwt_index_seeds(debwt_ctx* c, const char* reads, const uint64_t* offsets, uint64_t n_reads, const debwt_seed_opts* opts,
                      uint64_t* seed_offsets, uint64_t* n_hits_out, debwt_seed* seeds, uint64_t seeds_cap, debwt_seed_hit* hits,
                      uint64_t hits_cap) {
    if (!c || !c->indexed || !c->sa_rate) FAIL("no sampled suffix array: call debwt_index_sample_sa first");
    if (!offsets || !seed_offsets || !n_hits_out || !opts || (n_reads && !reads) || (seeds && !hits)) FAIL("null argument");
    const debwt_seed_opts op = *opts;
    const u64 m = n_reads;
    u64 max_len = 0;
    if (check_seed_input(c, "index_seeds", offsets, m, op, max_len)) return -1;
    seed_offsets[0] = 0;
    *n_hits_out = 0;
    if (m == 0) return 0;
    SeedRun r;
    const int rc = run_seeds(c, "index_seeds", reads, offsets, m, op, max_len, seed_offsets, r, [&](u64 total, u64 total_hits) -> int {
        *n_hits_out = total_hits;
        if (!seeds || total == 0) return 0;                                     // size query
        if (total > seeds_cap || total_hits > hits_cap)
            FAIL("index_seeds: the reads have " + std::to_string(total) + " seeds and " + std::to_string(total_hits) + " hits; seeds holds " +
                 std::to_string(seeds_cap) + " and hits " + std::to_string(hits_cap));
        return 1;
    });
    if (rc <= 0) return rc;
    cudaStream_t st = c->st;
    CUDA_TRY(cudaMemcpyAsync(seeds, r.seeds, r.total * sizeof(debwt_seed), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(hits, r.hits, r.total_hits * sizeof(debwt_seed_hit), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static_assert(sizeof(debwt_chain) == 40, "debwt_chain is 2 u64 + 5 u32 + float");
static_assert(sizeof(debwt_chain_seed) == 16, "debwt_chain_seed is u64 + 2 u32");

}  // extern "C"

// The checks of debwt_chain_opts; `name` starts the messages
static int check_chain_opts(const char* name, const debwt_chain_opts& co) {
    const std::pair<int32_t, const char*> ints[] = {{co.w, "w"}, {co.max_chain_gap, "max_chain_gap"}, {co.min_chain_weight, "min_chain_weight"},
                                                     {co.max_chain_extend, "max_chain_extend"}};
    for (const auto& [v, nm] : ints)
        if (v < 0) FAIL(std::string(name) + ": " + nm + " must not be negative, not " + std::to_string(v));
    const std::pair<float, const char*> reals[] = {{co.mask_level, "mask_level"}, {co.drop_ratio, "drop_ratio"}};
    for (const auto& [v, nm] : reals)
        if (!std::isfinite(v) || v < 0) FAIL(std::string(name) + ": " + nm + " must be finite and not negative, not " + std::to_string(v));
    return 0;
}

// The device buffers of one chaining run (its seeding run included), freed with it
struct ChainRun {
    SeedRun seeds;
    char* scratch = nullptr;          // ChainScratch | chain counts | seed counts | chain offsets | seed offsets | n_sorted | frac_rep
    char* out = nullptr;              // the kept chains | their seeds
    u64 *d_coff = nullptr, *d_soff = nullptr;
    debwt_chain* chains = nullptr;
    debwt_chain_seed* cseeds = nullptr;
    u64 total = 0, total_seeds = 0;
    ChainRun() = default;
    ChainRun(const ChainRun&) = delete;
    ~ChainRun() {
        if (scratch) cudaFree(scratch);
        if (out) cudaFree(out);
    }
};

// The seeding and chaining of debwt_index_chains for m >= 1 checked reads, leaving everything in r: chain_kernel and the
// two scans (chain_offsets, when given, receives the chain offsets; all zero when the reads have no hits), then
// proceed(total chains, total chain seeds): 1 goes on to write the kept chains and their seeds on the device, 0 stops
// there, -1 fails the call.  Returns 0 also when there are no hits.
template <class Proceed>
static int run_chains(debwt_ctx* c, const char* name, const char* reads, const uint64_t* offsets, u64 m, const debwt_seed_opts& op,
                      const debwt_chain_opts& co, u64 max_len, uint64_t* chain_offsets, ChainRun& cr, Proceed&& proceed) {
    const std::string nm(name);
    SeedRun& r = cr.seeds;
    const int rc = run_seeds(c, name, reads, offsets, m, op, max_len, nullptr, r, [](u64, u64 total_hits) { return total_hits ? 1 : 0; });
    if (rc < 0) return -1;
    if (rc == 0) {                                                                // no hits: no chains
        if (chain_offsets) std::fill(chain_offsets, chain_offsets + m + 1, 0ull);
        return proceed(0, 0) < 0 ? -1 : 0;
    }
    cudaStream_t st = c->st;
    const u64 H = r.total_hits, nb = (m + TPB - 1) / TPB;
    ChainParams prm;
    prm.w = co.w;
    prm.max_chain_gap = co.max_chain_gap;
    prm.max_chain_extend = co.max_chain_extend;
    prm.min_seed_len = op.min_seed_len;
    prm.min_chain_weight = (u32)co.min_chain_weight;
    prm.max_occ = op.max_occ;
    prm.mask_level = co.mask_level;
    prm.drop_ratio = co.drop_ratio;
    prm.l_pac = (c->n - c->n_rec) / 2;
    // per hit: chain seed, sort key, ChainRec, slot hit, next, tail, kept list (68 bytes); per read: kept chains and their
    // seeds, the offsets of both, chains after the weight pass, frac_rep; the slot bitmap and its summary
    const u64 n_bits = H / 64 + m + 1, n_summary = H / 4096 + m + 1;
    ChainScratch s;
    u64 *d_ccnt, *d_scnt;
    u32* d_nsorted;
    float* d_frac;
    char* p = nullptr;
    auto take = [&](auto*& dst, u64 n) {
        dst = reinterpret_cast<std::remove_reference_t<decltype(dst)>>(p);
        p += (n * sizeof(*dst) + 15) / 16 * 16;
    };
    auto lay_out = [&]() {
        take(s.cs, H); take(s.key, H); take(s.rec, H); take(s.idx, H); take(s.nxt, H); take(s.tail, H); take(s.list, H);
        take(s.bits, n_bits); take(s.summary, n_summary);
        take(d_ccnt, m); take(d_scnt, m); take(cr.d_coff, m + 1); take(cr.d_soff, m + 1); take(d_nsorted, m); take(d_frac, m);
    };
    lay_out();
    const u64 scratch_bytes = (u64)reinterpret_cast<uintptr_t>(p);
    if (cudaMalloc(reinterpret_cast<void**>(&cr.scratch), scratch_bytes) != cudaSuccess) {
        cudaGetLastError();
        cr.scratch = nullptr;
        FAIL(nm + ": out of device memory for " + std::to_string(scratch_bytes) + " bytes of chaining scratch (" + std::to_string(H) + " hits)");
    }
    p = cr.scratch;
    lay_out();
    int sms = 0, per_sm = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    CUDA_TRY(cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxThreadsPerMultiProcessor, c->device));
    const u64 n_threads = std::min<u64>((u64)sms * (u64)per_sm, m);
    CUDA_TRY(cudaMemsetAsync(r.d_next, 0, 8, st));
    chain_kernel<<<grid_for(n_threads), TPB, 0, st>>>(r.d_o, m, r.seeds, r.d_off, r.hits, r.d_hoff, c->d_seps_sorted, prm, s, r.d_next,
                                                      d_ccnt, d_scnt, d_nsorted, d_frac);
    hit_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_ccnt, m, r.d_tot);
    scan_u64_kernel<<<1, TPB, 0, st>>>(r.d_tot, nb, r.d_base);
    hit_offsets_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_ccnt, m, r.d_base, cr.d_coff);
    hit_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_scnt, m, r.d_tot);
    scan_u64_kernel<<<1, TPB, 0, st>>>(r.d_tot, nb, r.d_base);
    hit_offsets_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_scnt, m, r.d_base, cr.d_soff);
    DEBWT_COUNT(7);
    if (chain_offsets) CUDA_TRY(cudaMemcpyAsync(chain_offsets, cr.d_coff, (m + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&cr.total, cr.d_coff + m, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&cr.total_seeds, cr.d_soff + m, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    const int go = proceed(cr.total, cr.total_seeds);
    if (go <= 0) return go;
    const u64 total = cr.total, total_seeds = cr.total_seeds;
    if (cudaMalloc(reinterpret_cast<void**>(&cr.out), total * sizeof(debwt_chain) + total_seeds * sizeof(debwt_chain_seed)) != cudaSuccess) {
        cudaGetLastError();
        cr.out = nullptr;
        FAIL(nm + ": out of device memory for " + std::to_string(total) + " chains and " + std::to_string(total_seeds) + " chain seeds");
    }
    cr.chains = reinterpret_cast<debwt_chain*>(cr.out);
    cr.cseeds = reinterpret_cast<debwt_chain_seed*>(cr.chains + total);
    chain_write_kernel<<<grid_for(m), TPB, 0, st>>>(m, r.hits, r.d_hoff, s, d_nsorted, d_frac, cr.d_coff, cr.d_soff, cr.chains, cr.cseeds);
    DEBWT_COUNT(1);
    return 1;
}

extern "C" {

int debwt_index_chains(debwt_ctx* c, const char* reads, const uint64_t* offsets, uint64_t n_reads, const debwt_seed_opts* seed_opts,
                       const debwt_chain_opts* chain_opts, uint64_t* chain_offsets, uint64_t* n_chain_seeds_out, debwt_chain* chains,
                       uint64_t chains_cap, debwt_chain_seed* chain_seeds, uint64_t chain_seeds_cap) {
    if (!c || !c->indexed || !c->sa_rate) FAIL("no sampled suffix array: call debwt_index_sample_sa first");
    if (!offsets || !chain_offsets || !n_chain_seeds_out || !seed_opts || !chain_opts || (n_reads && !reads) || (chains && !chain_seeds))
        FAIL("null argument");
    const debwt_seed_opts op = *seed_opts;
    const debwt_chain_opts co = *chain_opts;
    if (check_chain_opts("index_chains", co)) return -1;
    const u64 m = n_reads;
    u64 max_len = 0;
    if (check_seed_input(c, "index_chains", offsets, m, op, max_len)) return -1;
    if (m == 0) {
        chain_offsets[0] = 0;
        *n_chain_seeds_out = 0;
        return 0;
    }
    ChainRun cr;
    const int rc = run_chains(c, "index_chains", reads, offsets, m, op, co, max_len, chain_offsets, cr, [&](u64 total, u64 total_seeds) -> int {
        *n_chain_seeds_out = total_seeds;
        if (!chains || total == 0) return 0;                                      // size query
        if (total > chains_cap || total_seeds > chain_seeds_cap)
            FAIL("index_chains: the reads have " + std::to_string(total) + " chains and " + std::to_string(total_seeds) + " chain seeds; chains holds " +
                 std::to_string(chains_cap) + " and chain_seeds " + std::to_string(chain_seeds_cap));
        return 1;
    });
    if (rc <= 0) return rc;
    cudaStream_t st = c->st;
    CUDA_TRY(cudaMemcpyAsync(chains, cr.chains, cr.total * sizeof(debwt_chain), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(chain_seeds, cr.cseeds, cr.total_seeds * sizeof(debwt_chain_seed), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    return 0;
}

}  // extern "C"

static_assert(sizeof(debwt_region) == 64, "debwt_region is 2 u64 + 11 u32 + float");

// bwa's pac, derived from the index the first time after sampling: the forward records' bases by the LF walks of
// extract_kernel (inverse samples built here if extract has not built them), 2 bits each.
static int build_pac(debwt_ctx* c, const char* name) {
    if (c->d_pac) return 0;
    const std::string nm(name);
    if (sorted_separators(c, name) || inverse_samples(c, name)) return -1;
    cudaStream_t st = c->st;
    const u64 R = c->n_rec, l_pac = (c->n - R) / 2, words = l_pac / 16 + 1;
    u64 fwd_end = 0;
    CUDA_TRY(cudaMemcpyAsync(&fwd_end, c->d_seps_sorted + R / 2 - 1, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (fwd_end - (R / 2 - 1) != l_pac) FAIL("internal: the forward records do not hold (N - R) / 2 bases");
    if (cudaMalloc(reinterpret_cast<void**>(&c->d_pac), words * 4) != cudaSuccess) {
        cudaGetLastError();
        c->d_pac = nullptr;
        FAIL(nm + ": out of device memory for the " + std::to_string(words * 4) + "-byte reference (pac)");
    }
    CUDA_TRY(cudaMemsetAsync(c->d_pac, 0, words * 4, st));
    const u64 n_blocks = (fwd_end + c->sa_rate - 1) / c->sa_rate;
    if (n_blocks) {
        pac_kernel<<<grid_for(n_blocks), TPB, 0, st>>>(view_of(c), sa_view_of(c), c->d_isa_vals, c->d_seps_sorted, R, fwd_end, n_blocks, c->d_pac);
        DEBWT_COUNT(1);
    }
    return 0;
}

extern "C" {

int debwt_index_regions(debwt_ctx* c, const char* reads, const uint64_t* offsets, uint64_t n_reads, const debwt_seed_opts* seed_opts,
                        const debwt_chain_opts* chain_opts, const debwt_ext_opts* ext_opts, uint64_t* region_offsets, debwt_region* regions,
                        uint64_t regions_cap) {
    if (!c || !c->indexed || !c->sa_rate) FAIL("no sampled suffix array: call debwt_index_sample_sa first");
    if (!offsets || !region_offsets || !seed_opts || !chain_opts || !ext_opts || (n_reads && !reads)) FAIL("null argument");
    const debwt_seed_opts op = *seed_opts;
    const debwt_chain_opts co = *chain_opts;
    const debwt_ext_opts eo = *ext_opts;
    if (check_chain_opts("index_regions", co)) return -1;
    const std::pair<int32_t, const char*> pos[] = {{eo.a, "a"}, {eo.e_del, "e_del"}, {eo.e_ins, "e_ins"}};
    for (const auto& [v, nm] : pos)
        if (v < 1) FAIL(std::string("index_regions: ") + nm + " must be at least 1, not " + std::to_string(v));
    const std::pair<int32_t, const char*> nonneg[] = {{eo.b, "b"}, {eo.o_del, "o_del"}, {eo.o_ins, "o_ins"}, {eo.pen_clip5, "pen_clip5"},
                                                       {eo.pen_clip3, "pen_clip3"}, {eo.zdrop, "zdrop"}};
    for (const auto& [v, nm] : nonneg)
        if (v < 0) FAIL(std::string("index_regions: ") + nm + " must not be negative, not " + std::to_string(v));
    for (const auto& [v, nm] : {std::pair<int32_t, const char*>{eo.a, "a"}, {eo.b, "b"}})
        if (v > 127) FAIL(std::string("index_regions: ") + nm + " = " + std::to_string(v) + " does not fit bwa's int8_t scoring matrix (at most 127)");
    if (co.w > kMaxExtW)
        FAIL("index_regions: w = " + std::to_string(co.w) + " is too wide: the band w << 1 of a retry must fit the DP window of " +
             std::to_string(2 * (kMaxExtW << 1) + 3) + " columns (w at most " + std::to_string(kMaxExtW) + ")");
    const u64 m = n_reads;
    u64 max_len = 0;
    if (check_seed_input(c, "index_regions", offsets, m, op, max_len)) return -1;
    {
        const long long mul = std::max({eo.a, eo.b, eo.e_del, eo.e_ins}), add = std::max({eo.o_del, eo.o_ins, eo.pen_clip5, eo.pen_clip3, eo.zdrop});
        const long double bound = (long double)(2 * max_len + 4 * (u64)co.w + 2) * mul + add;
        if (bound >= 2147483648.0L)
            FAIL("index_regions: the options can overflow a 32-bit score: (2 x " + std::to_string(max_len) + " (the longest read) + 4 w + 2) x " +
                 "max(a, b, e_del, e_ins) + max(o_del, o_ins, pen_clip5, pen_clip3, zdrop) = " + std::to_string((double)bound) + " is not below 2^31");
    }
    region_offsets[0] = 0;
    if (m == 0) return 0;
    ChainRun cr;
    const int rc = run_chains(c, "index_regions", reads, offsets, m, op, co, max_len, nullptr, cr, [](u64 total, u64) { return total ? 1 : 0; });
    if (rc < 0) return -1;
    if (rc == 0) {                                                                // no chains: no regions
        std::fill(region_offsets, region_offsets + m + 1, 0ull);
        return 0;
    }
    if (build_pac(c, "index_regions")) return -1;
    cudaStream_t st = c->st;
    SeedRun& r = cr.seeds;
    const u64 S = cr.total_seeds, nc = cr.total, nb = (m + TPB - 1) / TPB;
    // per chain seed: kept seed, its score, srt, a region slot (92 bytes); per chain: kept seeds; per read: regions, offsets
    ExtScratch xs;
    u64 *d_rcnt, *d_roff;
    char* p = nullptr;
    auto take = [&](auto*& dst, u64 n) {
        dst = reinterpret_cast<std::remove_reference_t<decltype(dst)>>(p);
        p += (n * sizeof(*dst) + 15) / 16 * 16;
    };
    auto lay_out = [&]() {
        take(xs.reg, S); take(xs.fs, S); take(xs.srt, S); take(xs.sc, S); take(xs.fn, nc); take(d_rcnt, m); take(d_roff, m + 1);
    };
    lay_out();
    const u64 scratch_bytes = (u64)reinterpret_cast<uintptr_t>(p);
    char* d_x = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_x), scratch_bytes) != cudaSuccess) {
        cudaGetLastError();
        FAIL("index_regions: out of device memory for " + std::to_string(scratch_bytes) + " bytes of extension scratch (" + std::to_string(S) +
             " chain seeds)");
    }
    struct Free { char* p; ~Free() { cudaFree(p); } } free_x{d_x};
    p = d_x;
    lay_out();
    ExtParams prm;
    prm.a = eo.a; prm.b = eo.b; prm.o_del = eo.o_del; prm.e_del = eo.e_del; prm.o_ins = eo.o_ins; prm.e_ins = eo.e_ins;
    prm.pen_clip5 = eo.pen_clip5; prm.pen_clip3 = eo.pen_clip3; prm.zdrop = eo.zdrop; prm.w = co.w; prm.min_chain_weight = co.min_chain_weight;
    prm.ring = std::max<u32>(2 * ((u32)co.w << 1) + 3, 200);
    prm.l_pac = (c->n - c->n_rec) / 2;
    const size_t smem = (size_t)EXT_WARPS * prm.ring * sizeof(int2);
    CUDA_TRY(cudaFuncSetAttribute(ext_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int sms = 0, per_sm = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    CUDA_TRY(cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxThreadsPerMultiProcessor, c->device));
    const u64 n_warps = std::min<u64>((u64)sms * (u64)per_sm / 32, m);
    CUDA_TRY(cudaMemsetAsync(r.d_next, 0, 8, st));
    ext_kernel<<<(unsigned)((n_warps + EXT_WARPS - 1) / EXT_WARPS), EXT_WARPS * 32, smem, st>>>(
        reinterpret_cast<const u8*>(r.d), r.d_o, m, cr.chains, cr.d_coff, cr.cseeds, cr.d_soff, c->d_pac, c->d_seps_sorted, prm, xs, r.d_next, d_rcnt);
    hit_count_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_rcnt, m, r.d_tot);
    scan_u64_kernel<<<1, TPB, 0, st>>>(r.d_tot, nb, r.d_base);
    hit_offsets_kernel<<<(unsigned)nb, TPB, 0, st>>>(d_rcnt, m, r.d_base, d_roff);
    DEBWT_COUNT(4);
    CUDA_TRY(cudaMemcpyAsync(region_offsets, d_roff, (m + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    const u64 total = region_offsets[m];
    if (!regions || total == 0) return 0;                                         // size query
    if (total > regions_cap)
        FAIL("index_regions: the reads have " + std::to_string(total) + " regions; regions holds " + std::to_string(regions_cap));
    debwt_region* d_out = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&d_out), total * sizeof(debwt_region)) != cudaSuccess) {
        cudaGetLastError();
        FAIL("index_regions: out of device memory for " + std::to_string(total) + " regions");
    }
    Free free_out{reinterpret_cast<char*>(d_out)};
    region_write_kernel<<<grid_for(m), TPB, 0, st>>>(m, cr.d_soff, xs.reg, d_roff, d_out);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(regions, d_out, total * sizeof(debwt_region), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    return 0;
}

}  // extern "C"
