// Device stages around the radix sort: packing, extraction, count-by-sort, branch k-mer detection,
// branch codes, emission.  Each kernel cites the reference loop it replaces (SURVEY.md section 2.2).
#include "stages.cuh"

#include <cstdlib>
#include "special.cuh"
#include "stages_dev.cuh"

namespace debwt {

namespace {

constexpr int TPB = 256;
inline unsigned grid_for(u64 work, int per_block) { return (unsigned)((work + per_block - 1) / per_block); }

// =============================================================================================
// generic exclusive scan (reduce -> scan partials -> rescan)
// =============================================================================================
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = TPB * SCAN_ITEMS;

template <bool POPC>
__device__ __forceinline__ u32 scan_f(u32 v) { return POPC ? (u32)__popc(v) : v; }

template <bool POPC>
__global__ void __launch_bounds__(TPB) scan_reduce_kernel(const u32* __restrict__ in, u64 m, u32* __restrict__ part) {
    __shared__ u32 sm[40];
    const u64 base = (u64)blockIdx.x * SCAN_TILE;
    u32 s = 0;
#pragma unroll 4
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        u64 i = base + (u64)j * TPB + threadIdx.x;
        if (i < m) s += scan_f<POPC>(in[i]);
    }
    u32 total;
    block_exclusive_scan<TPB>(s, &total, sm);
    if (threadIdx.x == 0) part[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) scan_partials_kernel(u32* __restrict__ part, u64 nb, u64* __restrict__ d_total) {
    __shared__ u32 sm[40];
    __shared__ u64 carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (u64 base = 0; base < nb; base += 1024) {
        u64 i = base + threadIdx.x;
        u32 v = i < nb ? part[i] : 0;
        u32 total;
        u32 ex = block_exclusive_scan<1024>(v, &total, sm);
        u64 carry = carry_s;
        if (i < nb) part[i] = (u32)(carry + ex);
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + total;
        __syncthreads();
    }
    if (threadIdx.x == 0 && d_total) *d_total = carry_s;
}

template <bool POPC>
__global__ void __launch_bounds__(TPB) scan_final_kernel(const u32* __restrict__ in, u32* __restrict__ out, u64 m,
                                                        const u32* __restrict__ part) {
    __shared__ u32 sm[40];
    const u64 base = (u64)blockIdx.x * SCAN_TILE + (u64)threadIdx.x * SCAN_ITEMS;
    u32 v[SCAN_ITEMS];
    u32 s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        u64 i = base + j;
        v[j] = i < m ? scan_f<POPC>(in[i]) : 0;
        s += v[j];
    }
    u32 ex = block_exclusive_scan<TPB>(s, nullptr, sm) + part[blockIdx.x];
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        u64 i = base + j;
        if (i < m) out[i] = ex;
        ex += v[j];
    }
}

}  // namespace

size_t scan_workspace_bytes(u64 m) { return ((m + SCAN_TILE - 1) / SCAN_TILE + 1) * 4 + 64; }

int scan_exclusive_u32(const u32* in, u32* out, u64 m, bool popc, void* workspace, u64* d_total, cudaStream_t st) {
    if (m == 0) {
        if (d_total) CUDA_TRY(cudaMemsetAsync(d_total, 0, 8, st));
        return 0;
    }
    u32* part = reinterpret_cast<u32*>(workspace);
    const u64 nb = (m + SCAN_TILE - 1) / SCAN_TILE;
    if (popc) scan_reduce_kernel<true><<<(unsigned)nb, TPB, 0, st>>>(in, m, part);
    else scan_reduce_kernel<false><<<(unsigned)nb, TPB, 0, st>>>(in, m, part);
    scan_partials_kernel<<<1, 1024, 0, st>>>(part, nb, d_total);
    if (popc) scan_final_kernel<true><<<(unsigned)nb, TPB, 0, st>>>(in, out, m, part);
    else scan_final_kernel<false><<<(unsigned)nb, TPB, 0, st>>>(in, out, m, part);
    DEBWT_COUNT(3);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// =============================================================================================
// K1: ASCII -> 2-bit packed text            (reference src/collect#$.c:66-90)
// =============================================================================================
namespace {

// IUPAC ambiguity codes -> one of the bases they stand for: the tables of the reference's pre-processing tool
// (reference otherTool/transferN.c:8-10,17-27: N ACGT, V ACG, D ATG, B TCG, H ATC, W AT, S CG, K TG, M AC, Y CT, R AG), with its
// rand() replaced by a splitmix64 value of (seed, symbol position): the same input and seed always give the same text.
__device__ __forceinline__ u32 resolve_ambiguous(u32 u /* upper case */, u64 seed, u64 pos, bool& known) {
    u32 set;                                          // up to four 2-bit base codes, lowest first; count in bits 8..10
    switch (u) {
        case 'N': set = 0xE4u | (4u << 8); break;     // A C G T
        case 'V': set = 0x24u | (3u << 8); break;     // A C G
        case 'D': set = 0x2Cu | (3u << 8); break;     // A T G
        case 'B': set = 0x27u | (3u << 8); break;     // T C G
        case 'H': set = 0x1Cu | (3u << 8); break;     // A T C
        case 'W': set = 0x0Cu | (2u << 8); break;     // A T
        case 'S': set = 0x09u | (2u << 8); break;     // C G
        case 'K': set = 0x0Bu | (2u << 8); break;     // T G
        case 'M': set = 0x04u | (2u << 8); break;     // A C
        case 'Y': set = 0x0Du | (2u << 8); break;     // C T
        case 'R': set = 0x08u | (2u << 8); break;     // A G
        default: known = false; return 3u;
    }
    known = true;
    u64 z = seed + (pos + 1) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    const u32 pick = (u32)(z % (u64)(set >> 8));
    return (set >> (2 * pick)) & 3u;
}

__device__ __forceinline__ u32 base_code(u32 c, u32& bad, u32& nsep, const PackPolicy& pol, u64 pos) {
    // A/a C/c G/g T/t -> 0 1 2 3; '#' '$' (separators) are stored as T like the reference does
    u32 u = c & 0xDFu;
    u32 code = (u >> 1) & 3u;
    code ^= code >> 1;
    bool ok = (u == 0x41u) | (u == 0x43u) | (u == 0x47u) | (u == 0x54u);
    bool sep = (c == 0x23u) | (c == 0x24u);
    if (!ok && !sep) {
        bool known = false;
        if (pol.resolve) code = resolve_ambiguous(u, pol.seed, pol.pos_base + pos, known);
        if (known) return code;
        bad |= 1u;
    }
    nsep += (u32)sep;
    return ok ? code : 3u;
}

__global__ void __launch_bounds__(TPB) pack_kernel(const u8* __restrict__ ascii, u64 n, u64* __restrict__ words,
                                                  u64 nwords, u32* __restrict__ err, PackPolicy pol) {
    const u64 w = (u64)blockIdx.x * TPB + threadIdx.x;
    if (w >= nwords) return;
    const u64 base = w * 32;
    u64 out = 0;
    u32 bad = 0, nsep = 0;
    if (base + 32 <= n) {
        const uint4* p = reinterpret_cast<const uint4*>(ascii + base);
        uint4 a = __ldg(p), b = __ldg(p + 1);
        u32 v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                u32 c = (v[q] >> (8 * r)) & 255u;
                out = (out << 2) | base_code(c, bad, nsep, pol, base + 4 * q + r);
            }
        }
    } else {
        for (int j = 0; j < 32; ++j) {
            u64 i = base + j;
            u32 code = (i < n + 32) ? 3u : 0u;      // exactly 32 T of padding past the end (src/collect#$.c:87-90)
            if (i < n) code = base_code(ascii[i], bad, nsep, pol, i);
            out = (out << 2) | code;
        }
    }
    words[w] = out;
    if (bad) atomicOr(err, 1u);
    if (nsep) atomicAdd(err + 1, nsep);        // separator bytes seen: must equal the number of records
}

// =============================================================================================
// K2: (k+1)-mer extraction                   (Jellyfish count, src/kmercounting.sh:8; src/mySort.c:54-83)
// =============================================================================================
// A block works on TILE_POS consecutive text positions: the packed words of the tile are staged in
// shared memory once (every window needs two of them), and the record lookup is done once per block when
// the tile lies inside one record (the common case), so the per-position work has no dependent global loads.
constexpr int TILE_POS = 4096;
constexpr int TILE_WORDS = TILE_POS / 32;
constexpr int TILE_ROWS = TILE_POS / TPB;      // positions per thread

struct TileText {
    u64 w[TILE_WORDS + 2];
    u64 rec_first, rec_last;                   // records of the first / last position of the tile
    u64 sep_first, start_first;                // separator and start of record rec_first
};

__device__ __forceinline__ void tile_load(TileText& t, const u64* __restrict__ words, u64 nwords_total, u64 base, u64 n,
                                          const u64* __restrict__ seps, u64 n_rec) {
    const u64 w0 = base >> 5;
    for (int i = threadIdx.x; i < TILE_WORDS + 2; i += TPB) t.w[i] = (w0 + i < nwords_total) ? words[w0 + i] : ~0ull;
    if (threadIdx.x == 0) {
        const u64 last = (base + TILE_POS - 1 < n) ? base + TILE_POS - 1 : n - 1;
        t.rec_first = record_of(seps, n_rec, base);
        t.rec_last = record_of(seps, n_rec, last);
        t.sep_first = t.rec_first < n_rec ? seps[t.rec_first] : 0;
        t.start_first = t.rec_first ? seps[t.rec_first - 1] + 1 : 0;
    }
    __syncthreads();
}

__device__ __forceinline__ u64 tile_window(const TileText& t, u32 local) {      // 32 symbols at tile-local position
    const u32 i = local >> 5, sft = (local & 31) * 2;
    const u64 a = t.w[i];
    return sft ? (a << sft) | (t.w[i + 1] >> (64 - sft)) : a;
}

// positions [pos_lo, pos_hi) of the text (pos_lo a multiple of 32); key index = p - 32 r - idx_base
__global__ void __launch_bounds__(TPB) extract_kernel(const u64* __restrict__ words, u64 nwords_total, u64 n,
                                                     const u64* __restrict__ seps, u64 n_rec,
                                                     u64* __restrict__ keys, u64 pos_lo, u64 pos_hi, u64 idx_base) {
    __shared__ TileText t;
    const u64 base = pos_lo + (u64)blockIdx.x * TILE_POS;
    tile_load(t, words, nwords_total, base, n, seps, n_rec);
    const bool one_record = t.rec_first == t.rec_last;
#pragma unroll
    for (int j = 0; j < TILE_ROWS; ++j) {
        const u32 local = j * TPB + threadIdx.x;
        const u64 p = base + local;
        if (p >= pos_hi) continue;
        u64 r = t.rec_first, sep = t.sep_first;
        if (!one_record) {
            r = record_of(seps, n_rec, p);
            if (r >= n_rec) continue;
            sep = seps[r];
        }
        if (p + KMER > sep) continue;              // window would contain the separator
        st_stream(keys + (p - (u64)KMER * r - idx_base), tile_window(t, local));
    }
}

// =============================================================================================
// K4: count-by-sort                           (src/mySort.c:76-77,194 kmerInfo records)
// =============================================================================================
constexpr int RLE_ITEMS = 8;
constexpr int RLE_TILE = TPB * RLE_ITEMS;

__global__ void __launch_bounds__(TPB) rle_count_kernel(const u64* __restrict__ k, u64 n, u32* __restrict__ tile_cnt) {
    __shared__ u32 sm[40];
    const u64 base = (u64)blockIdx.x * RLE_TILE + (u64)threadIdx.x * RLE_ITEMS;
    u32 c = 0;
#pragma unroll
    for (int j = 0; j < RLE_ITEMS; ++j) {
        u64 i = base + j;
        if (i < n) c += (i == 0 || k[i] != k[i - 1]);
    }
    u32 total;
    block_exclusive_scan<TPB>(c, &total, sm);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}

__global__ void __launch_bounds__(TPB) rle_write_kernel(const u64* __restrict__ k, u64 n, const u32* __restrict__ tile_ex,
                                                       u64* __restrict__ kmers, u64* __restrict__ starts) {
    __shared__ u32 sm[40];
    const u64 base = (u64)blockIdx.x * RLE_TILE + (u64)threadIdx.x * RLE_ITEMS;
    bool h[RLE_ITEMS];
    u32 c = 0;
#pragma unroll
    for (int j = 0; j < RLE_ITEMS; ++j) {
        u64 i = base + j;
        h[j] = i < n && (i == 0 || k[i] != k[i - 1]);
        c += h[j];
    }
    u64 o = (u64)tile_ex[blockIdx.x] + block_exclusive_scan<TPB>(c, nullptr, sm);
#pragma unroll
    for (int j = 0; j < RLE_ITEMS; ++j)
        if (h[j]) { kmers[o] = k[base + j]; starts[o] = base + j; ++o; }
}

}  // namespace

int k_pack_words(const u8* ascii, u64 n, u64* words, u64 nwords, u32* d_err, cudaStream_t st, PackPolicy pol) {
    if (nwords == 0) return 0;
    pack_kernel<<<grid_for(nwords, TPB), TPB, 0, st>>>(ascii, n, words, nwords, d_err, pol);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_extract(const u64* words, u64 n, const u64* d_seps, u64 n_rec, u64* keys, cudaStream_t st) {
    return k_extract_slice(words, n, 0, n, d_seps, n_rec, 0, keys, st);
}

int k_extract_slice(const u64* words, u64 n, u64 pos_lo, u64 pos_hi, const u64* d_seps, u64 n_rec, u64 idx_base, u64* keys,
                    cudaStream_t st) {
    if (pos_hi <= pos_lo) return 0;
    extract_kernel<<<grid_for(pos_hi - pos_lo, TILE_POS), TPB, 0, st>>>(words, text_words(n), n, d_seps, n_rec, keys, pos_lo, pos_hi,
                                                                        idx_base);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- digit histograms of all keys, straight from the packed text ------------------------------
// Every key is a 32-base window of the text, so its digit of pass p (bits 8p..8p+7 = bases 28-4p..31-4p) is the
// 4-mer that starts 28-4p bases after the window: all eight histograms are the 4-mer histogram of the text minus
// the 4-mers too close to a record end to be that digit of any in-record window.  One sweep over n/4 bytes with one
// shared-memory count per base replaces a sweep over 8n bytes with eight counts per key (src/mySort.c:98-103 builds
// its bucket table from the k-mers themselves).
namespace {
constexpr int TH_TPB = 256;

__global__ void __launch_bounds__(TH_TPB) text_hist_kernel(const u64* __restrict__ words, u64 n, u64* __restrict__ ghist) {
    __shared__ u32 sh[TH_TPB / 32][256];
    for (int i = threadIdx.x; i < (TH_TPB / 32) * 256; i += TH_TPB) (&sh[0][0])[i] = 0;
    __syncthreads();
    u32* mine = sh[threadIdx.x >> 5];
    const u64 nw = (n + 31) / 32;
    for (u64 w = (u64)blockIdx.x * TH_TPB + threadIdx.x; w < nw; w += (u64)gridDim.x * TH_TPB) {
        const u64 w0 = words[w], w1 = words[w + 1];
        const u64 left = n - w * 32;
        if (left >= 32) {
#pragma unroll
            for (int b = 0; b < 32; ++b) {
                const u64 x = b ? ((w0 << (2 * b)) | (w1 >> (64 - 2 * b))) : w0;
                atomicAdd(mine + (u32)(x >> 56), 1u);
            }
        } else {
            for (int b = 0; b < (int)left; ++b) {
                const u64 x = b ? ((w0 << (2 * b)) | (w1 >> (64 - 2 * b))) : w0;
                atomicAdd(mine + (u32)(x >> 56), 1u);
            }
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < 256; j += TH_TPB) {
        u32 c = 0;
#pragma unroll
        for (int w = 0; w < TH_TPB / 32; ++w) c += sh[w][j];
        if (c) {
#pragma unroll
            for (int p = 0; p < 8; ++p) atomicAdd(reinterpret_cast<unsigned long long*>(ghist + p * 256 + j), (unsigned long long)c);
        }
    }
}

// one thread per (record, pass): take back the 4-mers at the o = 28-4p positions after the record start and at the
// 32-o positions up to and including the separator
__global__ void __launch_bounds__(TH_TPB) text_hist_fix_kernel(const u64* __restrict__ words, const u64* __restrict__ seps,
                                                              u64 n_rec, u64* __restrict__ ghist) {
    const u64 t = (u64)blockIdx.x * TH_TPB + threadIdx.x;
    if (t >= n_rec * 8) return;
    const u64 r = t >> 3;
    const u32 p = (u32)(t & 7), o = 28 - 4 * p;
    const u64 s = r ? seps[r - 1] + 1 : 0, e = seps[r];
    unsigned long long* h = reinterpret_cast<unsigned long long*>(ghist + p * 256);
    for (u64 q = s; q < s + o; ++q) atomicAdd(h + (text_window32(words, q) >> 56), ~0ull);
    for (u64 q = e - 31 + o; q <= e; ++q) atomicAdd(h + (text_window32(words, q) >> 56), ~0ull);
}
}  // namespace

bool text_digit_hist_applies(u64 n, u64 n_rec) { return n_rec * 2048 <= n; }

int k_text_digit_hist(const u64* words, u64 n, const u64* d_seps, u64 n_rec, u64* ghist, cudaStream_t st) {
    const u64 nw = (n + 31) / 32;
    const u64 want = (nw + TH_TPB - 1) / TH_TPB;
    text_hist_kernel<<<(unsigned)(want < 148u * 8u ? (want ? want : 1) : 148u * 8u), TH_TPB, 0, st>>>(words, n, ghist);
    text_hist_fix_kernel<<<grid_for(n_rec * 8, TH_TPB), TH_TPB, 0, st>>>(words, d_seps, n_rec, ghist);
    DEBWT_COUNT(2);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

namespace {
__global__ void __launch_bounds__(TPB) diff_kernel(const u64* __restrict__ starts, u64 d, u64 n, u64* __restrict__ counts) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i < d) counts[i] = ((i + 1 < d) ? starts[i + 1] : n) - starts[i];
}
}  // namespace

size_t rle_workspace_bytes(u64 n) {
    const u64 nt = (n + RLE_TILE - 1) / RLE_TILE + 1;
    return nt * 8 + scan_workspace_bytes(nt) + n * 8 + 64;
}

int k_rle(const u64* sorted, u64 n, u64* kmers, u64* counts, void* workspace, u64* d_total, cudaStream_t st) {
    if (n == 0) { CUDA_TRY(cudaMemsetAsync(d_total, 0, 8, st)); return 0; }
    const u64 nt = (n + RLE_TILE - 1) / RLE_TILE;
    u32* tile_cnt = reinterpret_cast<u32*>(workspace);
    u32* tile_ex = tile_cnt + nt;
    char* p = reinterpret_cast<char*>(tile_ex + nt);
    p += (8 - (reinterpret_cast<uintptr_t>(p) & 7)) & 7;
    void* scan_ws = p;
    p += (scan_workspace_bytes(nt) + 7) & ~(size_t)7;
    u64* starts = reinterpret_cast<u64*>(p);
    rle_count_kernel<<<(unsigned)nt, TPB, 0, st>>>(sorted, n, tile_cnt);
    if (scan_exclusive_u32(tile_cnt, tile_ex, nt, false, scan_ws, d_total, st)) return -1;
    rle_write_kernel<<<(unsigned)nt, TPB, 0, st>>>(sorted, n, tile_ex, kmers, starts);
    u64 d = 0;
    CUDA_TRY(cudaMemcpyAsync(&d, d_total, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    diff_kernel<<<grid_for(d, TPB), TPB, 0, st>>>(starts, d, n, counts);
    DEBWT_COUNT(3);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// =============================================================================================
// K5/K6: in/out edges per k-mer group         (src/getKmer.c:62-120, src/INandOut.c:260-343)
// =============================================================================================
namespace {

// idx[t] = lower_bound(keys, t << shift).  Two streaming steps: every key that opens a bucket records its
// own position (one coalesced sweep over the keys), then every bucket that stayed empty -- rare inside
// the key range, but a whole prefix / suffix of the table when a device owns a narrow key range --
// resolves itself with a binary search.
__global__ void __launch_bounds__(TPB) key_index_mark_kernel(const u64* __restrict__ k, u64 n, KeyIndex ki) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;
    const int sh = 64 - ki.bits;
    const u64 cur = k[i] >> sh;
    if (i == 0 || (k[i - 1] >> sh) != cur) ki.idx[cur] = (u32)i;
}

__global__ void __launch_bounds__(TPB) key_index_fill_kernel(const u64* __restrict__ k, u64 n, KeyIndex ki) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    const u64 nb = 1ull << ki.bits;
    if (t > nb) return;
    if (t == nb) { ki.idx[t] = (u32)n; return; }
    if (ki.idx[t] == 0xFFFFFFFFu) ki.idx[t] = (u32)lower_bound_u64(k, 0, n, t << (64 - ki.bits));
}

constexpr int ME_ROWS = 4;       // independent keys per thread: four search chains in flight instead of one

// In / out edge marks of ME_ROWS keys per thread: keys base + j * TPB, j < ME_ROWS, below `limit`.
__device__ __forceinline__ void edge_rows(const u64* __restrict__ k, u64 n, const KeyIndex& ki, u16* __restrict__ gmask, u64 base,
                                          u64 limit) {
    u64 key[ME_ROWS], lo[ME_ROWS], hi[ME_ROWS];
    bool act[ME_ROWS];
#pragma unroll
    for (int j = 0; j < ME_ROWS; ++j) {
        const u64 i = base + (u64)j * TPB;
        act[j] = i < limit;
        key[j] = act[j] ? k[i] : 0;
        if (act[j] && i > 0 && k[i - 1] == key[j]) act[j] = false;     // one representative per distinct (k+1)-mer
    }
    // in edge: (k+1)-mer cX marks k-mer X with c
#pragma unroll
    for (int j = 0; j < ME_ROWS; ++j) {
        const u64 t = (key[j] << 2) >> (64 - ki.bits);
        lo[j] = act[j] ? ki.idx[t] : 0;
        hi[j] = act[j] ? ki.idx[t + 1] : 0;
    }
#pragma unroll
    for (int j = 0; j < ME_ROWS; ++j) {
        if (!act[j]) continue;
        const u64 q = key[j] << 2;
        const u64 hs = lower_bound_u64(k, lo[j], hi[j], q);
        if (hs < n && (k[hs] >> 2) == (q >> 2)) atomic_or_u16(gmask, hs, 1u << (u32)(key[j] >> 62));
    }
    // out edge: k-mer = first 31 bases, next symbol = last base
#pragma unroll
    for (int j = 0; j < ME_ROWS; ++j) {
        if (!act[j]) continue;
        const u64 i = base + (u64)j * TPB;
        atomic_or_u16(gmask, group_head(k, i), 1u << (GM_OUT_SHIFT + (u32)(key[j] & 3)));
    }
}

// The in-edge join: (k+1)-mer c.X marks the group of X, and inside each first-base block c the targets ascend with the
// sources, so the join is four merges against the whole key array.  The blocks are scheduled by TARGET: tile t of
// ME_TILE consecutive target keys is served by four thread blocks (one per c, adjacent block ids, so they run together),
// each of which finds by two searches the run of its c block whose targets fall into the tile.  The four runs then search
// and mark the same 64 KB of keys / 16 KB of masks while they are in L2, and every key is fetched from HBM once as a
// source and once as a target (the round-robin over equal SOURCE chunks this replaces drifted apart on repeat-rich
// genomes and re-read the keys 4.7 times at 3.1 Gbp).  A run longer than ME_CAP (a highly repeated (k+1)-mer) leaves its
// tail on a list that the whole grid works off afterwards.
constexpr u64 ME_TILE = 8192;
constexpr u64 ME_CAP = 8 * ME_TILE;
struct EdgeRun { u64 begin, end; };

// bounds[c * (tiles + 1) + t] = first source of the c block whose target lies in tile t or later (one thread per bound, so that
// the join's blocks start without a search and a barrier of their own)
__global__ void __launch_bounds__(TPB) edge_bounds_kernel(const u64* __restrict__ k, u64 n, KeyIndex ki, u64 tiles,
                                                         u64* __restrict__ bounds) {
    const u64 x = (u64)blockIdx.x * TPB + threadIdx.x;
    if (x >= 4 * (tiles + 1)) return;
    const u32 c = (u32)(x / (tiles + 1));
    const u64 t = x % (tiles + 1);
    const u64 cbeg = ki.idx[(u64)c << (ki.bits - 2)];
    const u64 cend = (c == 3) ? n : (u64)ki.idx[(u64)(c + 1) << (ki.bits - 2)];
    // sources whose query (X followed by A) sorts after key a - 1 and not after key b - 1 have their lower bound in [a, b)
    const u64 a = t * ME_TILE;
    u64 r;
    if (a == 0) r = cbeg;
    else if (a >= n) r = cend;
    else {
        const u64 low = (k[a - 1] >> 2) + 1;
        r = (low >> 62) ? cend : indexed_lower_bound(k, ki, ((u64)c << 62) | low);
    }
    bounds[x] = r;
}

__global__ void __launch_bounds__(TPB) mark_edges_kernel(const u64* __restrict__ k, u64 n, KeyIndex ki, u16* __restrict__ gmask,
                                                        const u64* __restrict__ bounds, u64 tiles, EdgeRun* __restrict__ over,
                                                        u32* __restrict__ n_over) {
    const u32 c = blockIdx.x & 3u;
    const u64 tile = blockIdx.x >> 2;
    const u64 sb = bounds[c * (tiles + 1) + tile];
    u64 se = bounds[c * (tiles + 1) + tile + 1];
    if (se - sb > ME_CAP && se > sb) {
        if (threadIdx.x == 0) over[atomicAdd(n_over, 1u)] = EdgeRun{sb + ME_CAP, se};
        se = sb + ME_CAP;
    }
    for (u64 i0 = sb; i0 < se; i0 += (u64)TPB * ME_ROWS) edge_rows(k, n, ki, gmask, i0 + threadIdx.x, se);
}

__global__ void __launch_bounds__(TPB) mark_edges_over_kernel(const u64* __restrict__ k, u64 n, KeyIndex ki, u16* __restrict__ gmask,
                                                             const EdgeRun* __restrict__ over, const u32* __restrict__ n_over) {
    const u32 m = *n_over;
    for (u32 q = 0; q < m; ++q) {
        const EdgeRun r = over[q];
        for (u64 i0 = r.begin + (u64)blockIdx.x * (TPB * ME_ROWS); i0 < r.end; i0 += (u64)gridDim.x * (TPB * ME_ROWS))
            edge_rows(k, n, ki, gmask, i0 + threadIdx.x, r.end);
    }
}

__global__ void __launch_bounds__(TPB) mark_heads_tails_kernel(const u64* __restrict__ words, const u64* __restrict__ seps,
                                                              u64 n_rec, const u64* __restrict__ k, u64 n, KeyIndex ki,
                                                              u16* __restrict__ gmask) {
    const u64 r = (u64)blockIdx.x * TPB + threadIdx.x;
    if (r >= n_rec) return;
    const u64 start = r ? seps[r - 1] + 1 : 0;
    // head k-mer: follows '#' / starts the text -> forced multi-in (src/INandOut.c:282-291)
    u64 x = text_window32(words, start) & ~3ull;
    u64 h = indexed_lower_bound(k, ki, x);
    if (h < n && (k[h] & ~3ull) == x) atomic_or_u16(gmask, h, GM_IN_SEP);
    // tail k-mer: precedes the separator -> forced multi-out (src/INandOut.c:260-266)
    x = text_window32(words, seps[r] - KNODE) & ~3ull;
    h = indexed_lower_bound(k, ki, x);
    if (h < n && (k[h] & ~3ull) == x) atomic_or_u16(gmask, h, GM_OUT_TAIL);
}

__global__ void __launch_bounds__(TPB) propagate_kernel(const u64* __restrict__ k, u64 n, u16* __restrict__ gmask) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i >= n || i == 0) return;
    if ((k[i - 1] >> 2) != (k[i] >> 2)) return;     // group head keeps its own mask
    gmask[i] = gmask[group_head(k, i)];
}

// =============================================================================================
// K7: branch table (red/black tables of the reference, src/INandOut.c:396-417)
// =============================================================================================
constexpr int BR_ITEMS = 8;
constexpr int BR_TILE = TPB * BR_ITEMS;

// Both passes read the keys row by row (thread t of row j handles key base + j*TPB + t: coalesced), find
// group heads from the left neighbour and compact the branch groups in key order with warp ballots.
// The count pass also copies every head's mask to the other members of its group (K6's "propagate").
template <bool WRITE, bool PROPAGATE>
__global__ void __launch_bounds__(TPB) branch_kernel(const u64* __restrict__ k, u64 n, u16* __restrict__ gmask,
                                                    u32* __restrict__ tile_nb, u32* __restrict__ tile_blue,
                                                    const u32* __restrict__ tile_nb_ex, const u32* __restrict__ tile_blue_ex,
                                                    u32* __restrict__ head_bits, BranchTable bt) {
    constexpr int NW = TPB / 32;
    __shared__ u32 s_cnt[BR_ITEMS * NW + 1], s_blue[BR_ITEMS * NW + 1];
    if (WRITE && tile_nb[blockIdx.x] == 0) return;   // the count pass found no branch group in this tile
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u64 base = (u64)blockIdx.x * BR_TILE;
    const u32 lt = lanemask_lt();
    u32 flags[BR_ITEMS], size[BR_ITEMS], bal[BR_ITEMS];
#pragma unroll
    for (int j = 0; j < BR_ITEMS; ++j) {
        const u64 i = base + (u64)j * TPB + threadIdx.x;
        flags[j] = 0;
        size[j] = 0;
        if (WRITE) {
            // the count pass left one bit per key: "heads a branch group".  Only those keys are read again (a few per cent),
            // instead of a second sweep over all keys.
            bal[j] = head_bits[(base + (u64)j * TPB) / 32 + warp];
            if ((bal[j] >> lane) & 1u) {
                const u32 m = gmask[i];
                const u32 f = (gm_multi_out(m) ? 1u : 0u) | (gm_multi_in(m) ? 2u : 0u);
                flags[j] = f | 4u;
                if (f & 2u) size[j] = (u32)(group_end(k, n, i) - i);
            }
        } else {
            const bool valid = i < n;
            bool head = false;
            u32 m = 0;
            if (valid) {
                const u64 key = k[i];
                head = (i == 0) || ((k[i - 1] >> 2) != (key >> 2));
                if (head) {
                    m = gmask[i];
                    const u32 f = (gm_multi_out(m) ? 1u : 0u) | (gm_multi_in(m) ? 2u : 0u);
                    if (f) {
                        flags[j] = f | 4u;
                        if (f & 2u) size[j] = (u32)(group_end(k, n, i) - i);
                    }
                }
            }
            if (PROPAGATE) {
                // every member of a group gets its head's mask: from the nearest head to the left in the warp row (shuffle);
                // the lanes before the row's first head all belong to lane 0's group: one search for the warp
                const u32 hb = __ballot_sync(0xffffffffu, head);
                const u32 mine = hb & (lt | (1u << lane));
                const u32 got = __shfl_sync(0xffffffffu, m, mine ? 31 - __clz(mine) : 0);
                u32 lead = 0;
                if (lane == 0 && valid && !head) lead = gmask[group_head(k, i)];
                lead = __shfl_sync(0xffffffffu, lead, 0);
                if (valid && !head) gmask[i] = (u16)(mine ? got : lead);
            }
            bal[j] = __ballot_sync(0xffffffffu, flags[j] != 0);
            if (lane == 0) head_bits[(base + (u64)j * TPB) / 32 + warp] = bal[j];
        }
        u32 sz = size[j];
        if (bal[j]) {                                 // warp-uniform: most rows hold no branch head
#pragma unroll
            for (int o = 16; o; o >>= 1) sz += __shfl_xor_sync(0xffffffffu, sz, o);
        }
        if (lane == 0) { s_cnt[j * NW + warp] = __popc(bal[j]); s_blue[j * NW + warp] = sz; }
    }
    __syncthreads();
    if (warp == 0) {                              // 64 partials: exclusive scan by the first warp, two per lane
        static_assert(BR_ITEMS * NW == 64, "two partials per lane");
        const u32 c0 = s_cnt[2 * lane], c1 = s_cnt[2 * lane + 1], b0 = s_blue[2 * lane], b1 = s_blue[2 * lane + 1];
        u32 ic = c0 + c1, ib = b0 + b1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 tc = __shfl_up_sync(0xffffffffu, ic, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
            if (lane >= o) { ic += tc; ib += tb; }
        }
        const u32 ec = ic - (c0 + c1), eb = ib - (b0 + b1);
        s_cnt[2 * lane] = ec; s_cnt[2 * lane + 1] = ec + c0;
        s_blue[2 * lane] = eb; s_blue[2 * lane + 1] = eb + b0;
        if (lane == 31) {
            s_cnt[BR_ITEMS * NW] = ic; s_blue[BR_ITEMS * NW] = ib;
            if (!WRITE) { tile_nb[blockIdx.x] = ic; tile_blue[blockIdx.x] = ib; }
        }
    }
    if (!WRITE) return;
    __syncthreads();
    const u64 ob0 = tile_nb_ex[blockIdx.x];
    const u32 ol0 = tile_blue_ex[blockIdx.x];
#pragma unroll
    for (int j = 0; j < BR_ITEMS; ++j) {
        if (bal[j] == 0) continue;                    // warp-uniform
        // exclusive prefix of the sizes inside the warp row
        u32 inc = size[j];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (flags[j]) {
            const u64 i = base + (u64)j * TPB + threadIdx.x;
            const u64 ob = ob0 + s_cnt[j * NW + warp] + __popc(bal[j] & lt);
            bt.kmer[ob] = (k[i] & ~3ull) | (flags[j] & 3u);
            bt.head[ob] = (u32)i;
            bt.blue[ob] = ol0 + s_blue[j * NW + warp] + (inc - size[j]);
        }
    }
}

__global__ void __launch_bounds__(TPB) branch_index_kernel(BranchTable bt) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    const u64 nb = 1ull << bt.bits;
    if (t > nb) return;
    bt.bidx[t] = (t == nb) ? (u32)bt.n_branch : (u32)lower_bound_u64(bt.kmer, 0, bt.n_branch, t << (64 - bt.bits));
}

__global__ void __launch_bounds__(TPB) branch_filter_kernel(BranchTable bt) {
    const u64 b = (u64)blockIdx.x * TPB + threadIdx.x;
    if (b >= bt.n_branch) return;
    const u64 f = bt.filter_of(bt.kmer[b] & ~3ull);
    atomicOr(bt.filter() + (f >> 5), 1u << (f & 31));
}

__global__ void __launch_bounds__(TPB) branch_hash_kernel(BranchTable bt) {
    const u64 b = (u64)blockIdx.x * TPB + threadIdx.x;
    if (b >= bt.n_branch) return;
    const u64 e = bt.kmer[b];
    const u64 mask = (1ull << bt.hbits) - 1;
    for (u64 h = bt.hash_of(e & ~3ull);; h = (h + 1) & mask) {
        unsigned long long* claim = reinterpret_cast<unsigned long long*>(&bt.hslots[h].x);
        if (atomicCAS(claim, 0ull, (unsigned long long)e) == 0ull) {
            bt.hslots[h].y = bt.hmode ? (u64)bt.blue[b] << 32 : b;
            return;
        }
    }
}

__global__ void __launch_bounds__(TPB) special_ins_kernel(const u64* __restrict__ k, u64 n, KeyIndex ki,
                                                         const u64* __restrict__ pads, u64 m, u64* __restrict__ ins) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t < m) ins[t] = indexed_upper_bound(k, ki, pads[t]);
}

}  // namespace

int k_key_index_init(KeyIndex ki, cudaStream_t st) {
    CUDA_TRY(cudaMemsetAsync(ki.idx, 0xFF, ((1ull << ki.bits) + 1) * 4, st));
    return 0;
}

// marked = the last sort pass already recorded every bucket's first position (SortWorkspace::key_index)
int k_key_index_finish(const u64* sorted, u64 n, KeyIndex ki, bool marked, cudaStream_t st) {
    if (n && !marked) {
        key_index_mark_kernel<<<grid_for(n, TPB), TPB, 0, st>>>(sorted, n, ki);
        DEBWT_COUNT(1);
    }
    key_index_fill_kernel<<<grid_for((1ull << ki.bits) + 1, TPB), TPB, 0, st>>>(sorted, n, ki);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_build_key_index(const u64* sorted, u64 n, KeyIndex ki, cudaStream_t st) {
    if (k_key_index_init(ki, st)) return -1;
    return k_key_index_finish(sorted, n, ki, false, st);
}

int k_mark_edges(const u64* sorted, u64 n, KeyIndex ki, u16* gmask, cudaStream_t st) {
    if (n == 0) return 0;
    const u64 tiles = (n + ME_TILE - 1) / ME_TILE;
    const u64 cap = n / ME_CAP + 8;                          // runs that can exceed ME_CAP
    char* ws = nullptr;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&ws), 16 + cap * sizeof(EdgeRun) + 4 * (tiles + 1) * 8, st));
    u32* n_over = reinterpret_cast<u32*>(ws);
    EdgeRun* over = reinterpret_cast<EdgeRun*>(ws + 16);
    u64* bounds = reinterpret_cast<u64*>(ws + 16 + cap * sizeof(EdgeRun));
    cudaMemsetAsync(n_over, 0, 16, st);
    edge_bounds_kernel<<<grid_for(4 * (tiles + 1), TPB), TPB, 0, st>>>(sorted, n, ki, tiles, bounds);
    mark_edges_kernel<<<(unsigned)(4 * tiles), TPB, 0, st>>>(sorted, n, ki, gmask, bounds, tiles, over, n_over);
    mark_edges_over_kernel<<<148 * 8, TPB, 0, st>>>(sorted, n, ki, gmask, over, n_over);
    DEBWT_COUNT(3);
    const cudaError_t e = cudaGetLastError();
    cudaFreeAsync(ws, st);
    if (e != cudaSuccess) { set_error(std::string("mark_edges: ") + cudaGetErrorString(e)); return -1; }
    return 0;
}

int k_mark_heads_tails(const u64* words, const u64* d_seps, u64 n_rec, const u64* sorted, u64 n, KeyIndex ki, u16* gmask,
                       cudaStream_t st) {
    mark_heads_tails_kernel<<<grid_for(n_rec, TPB), TPB, 0, st>>>(words, d_seps, n_rec, sorted, n, ki, gmask);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_propagate(const u64* sorted, u64 n, u16* gmask, cudaStream_t st) {
    if (n == 0) return 0;
    propagate_kernel<<<grid_for(n, TPB), TPB, 0, st>>>(sorted, n, gmask);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

namespace {
struct BranchWs { u32 *nb, *blue, *nb_ex, *blue_ex, *head_bits; void* scan_ws; u64 nt; };
BranchWs branch_ws(void* workspace, u64 n) {
    BranchWs w;
    w.nt = (n + BR_TILE - 1) / BR_TILE;
    u32* p = reinterpret_cast<u32*>(workspace);
    w.nb = p; w.blue = p + w.nt; w.nb_ex = p + 2 * w.nt; w.blue_ex = p + 3 * w.nt;
    char* q = reinterpret_cast<char*>(p + 4 * w.nt);
    q += (8 - (reinterpret_cast<uintptr_t>(q) & 7)) & 7;
    w.scan_ws = q;
    q += (scan_workspace_bytes(w.nt + 1) + 15) & ~(size_t)15;
    w.head_bits = reinterpret_cast<u32*>(q);          // one bit per key, BR_TILE / 32 words per tile
    return w;
}
}  // namespace

size_t branch_workspace_bytes(u64 n) {
    const u64 nt = (n + BR_TILE - 1) / BR_TILE + 1;
    return nt * 16 + 16 + scan_workspace_bytes(nt) + 32 + nt * (BR_TILE / 8);
}

int k_branch_count(const u64* sorted, u64 n, u16* gmask, bool propagate, void* workspace, u64* d_totals, cudaStream_t st) {
    BranchWs w = branch_ws(workspace, n);
    BranchTable none;
    if (propagate) branch_kernel<false, true><<<(unsigned)w.nt, TPB, 0, st>>>(sorted, n, gmask, w.nb, w.blue, nullptr, nullptr, w.head_bits, none);
    else branch_kernel<false, false><<<(unsigned)w.nt, TPB, 0, st>>>(sorted, n, gmask, w.nb, w.blue, nullptr, nullptr, w.head_bits, none);
    DEBWT_COUNT(1);
    if (scan_exclusive_u32(w.nb, w.nb_ex, w.nt, false, w.scan_ws, d_totals, st)) return -1;
    if (scan_exclusive_u32(w.blue, w.blue_ex, w.nt, false, w.scan_ws, d_totals + 1, st)) return -1;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_branch_write(const u64* sorted, u64 n, const u16* gmask, void* workspace, BranchTable bt, cudaStream_t st) {
    BranchWs w = branch_ws(workspace, n);
    branch_kernel<true, false><<<(unsigned)w.nt, TPB, 0, st>>>(sorted, n, const_cast<u16*>(gmask), w.nb, nullptr, w.nb_ex, w.blue_ex, w.head_bits, bt);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_branch_index(BranchTable bt, cudaStream_t st) {
    branch_index_kernel<<<grid_for((1ull << bt.bits) + 1, TPB), TPB, 0, st>>>(bt);
    CUDA_TRY(cudaMemsetAsync(bt.filter(), 0, (1ull << (BranchTable::filter_bits(bt.bits) - 5)) * 4, st));
    if (bt.n_branch) branch_filter_kernel<<<grid_for(bt.n_branch, TPB), TPB, 0, st>>>(bt);
    DEBWT_COUNT(2);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_branch_hash(BranchTable bt, cudaStream_t st) {
    if (!bt.hslots) return 0;
    CUDA_TRY(cudaMemsetAsync(bt.hslots, 0, (1ull << bt.hbits) * sizeof(ulonglong2), st));
    if (bt.n_branch) branch_hash_kernel<<<grid_for(bt.n_branch, TPB), TPB, 0, st>>>(bt);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

namespace {
__global__ void __launch_bounds__(128) special_scan_kernel(const u64* __restrict__ words, const u64* __restrict__ seps,
                                                          u64 n_rec, const u64* __restrict__ k, u64 n_keys, KeyIndex ki,
                                                          SpecialInfo* __restrict__ out) {
    __shared__ u32 s_cnt;
    const u64 m = n_rec * 32;
    const u64 a = blockIdx.x;
    const u64 pa = seps[a >> 5] - (a & 31);
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    u32 cnt = 0;
    for (u64 b = threadIdx.x; b < m; b += blockDim.x) {
        if (b == a) continue;
        const u64 pb = seps[b >> 5] - (b & 31);
        cnt += special_less(words, seps, n_rec, pb, pa) ? 1u : 0u;
    }
    if (cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    if (threadIdx.x == 0) {
        const u32 j = (u32)(a & 31);
        SpecialInfo o;
        o.w0 = text_window32(words, pa);
        o.w1 = text_window32(words, pa + j + 1);
        o.rank = s_cnt;
        o.prev = (u8)text_symbol(words, pa - 1);
        o.next = (u8)text_symbol(words, pa + 31);
        o.pad_[0] = o.pad_[1] = 0;
        // T padding (src/collect#$.c:428-455): j bases then T's; suffixes that start with a separator sort last
        o.ins = j ? indexed_upper_bound(k, ki, (o.w0 & ~(~0ull >> (2 * j))) | (~0ull >> (2 * j))) : n_keys;
        out[a] = o;
    }
}
}  // namespace

namespace {
constexpr u32 SPEC_INF = 0xFFFFFFFFu;

__global__ void __launch_bounds__(TPB) special_ids_kernel(u32* __restrict__ ids, u64 m, u64 mp2) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i < mp2) ids[i] = i < m ? (u32)i : SPEC_INF;
}

__device__ __forceinline__ bool special_id_less(u32 x, u32 y, const u64* __restrict__ words, const u64* __restrict__ seps,
                                                u64 n_rec) {
    if (x == SPEC_INF) return false;                 // padding ids are larger than every suffix
    if (y == SPEC_INF) return true;
    return special_less_rec(words, seps, n_rec, seps[x >> 5] - (x & 31), x >> 5, seps[y >> 5] - (y & 31), y >> 5);
}

// one compare-exchange stage of the bitonic network (partner distance j inside runs of length k)
__global__ void __launch_bounds__(TPB) special_bitonic_kernel(u32* __restrict__ ids, u64 mp2, u64 j, u64 k,
                                                             const u64* __restrict__ words, const u64* __restrict__ seps, u64 n_rec) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i >= mp2) return;
    const u64 l = i ^ j;
    if (l <= i) return;
    const u32 a = ids[i], b = ids[l];
    const bool ascending = (i & k) == 0;
    const bool swap = ascending ? special_id_less(b, a, words, seps, n_rec) : special_id_less(a, b, words, seps, n_rec);
    if (swap) { ids[i] = b; ids[l] = a; }
}

// windows, neighbours and insertion point of the suffix that ended up at sorted position `pos`
__global__ void __launch_bounds__(TPB) special_info_kernel(const u32* __restrict__ ids, u64 m, const u64* __restrict__ words,
                                                          const u64* __restrict__ seps, const u64* __restrict__ k, u64 n_keys,
                                                          KeyIndex ki, SpecialInfo* __restrict__ out) {
    const u64 pos = (u64)blockIdx.x * TPB + threadIdx.x;
    if (pos >= m) return;
    const u32 a = ids[pos];
    const u64 pa = seps[a >> 5] - (a & 31);
    const u32 j = a & 31;
    SpecialInfo o;
    o.w0 = text_window32(words, pa);
    o.w1 = text_window32(words, pa + j + 1);
    o.rank = (u32)pos;
    o.prev = (u8)text_symbol(words, pa - 1);
    o.next = (u8)text_symbol(words, pa + 31);
    o.pad_[0] = o.pad_[1] = 0;
    o.ins = j ? indexed_upper_bound(k, ki, (o.w0 & ~(~0ull >> (2 * j))) | (~0ull >> (2 * j))) : n_keys;
    out[a] = o;
}
}  // namespace

int k_special_scan(const u64* words, const u64* d_seps, u64 n_rec, const u64* sorted, u64 n_keys, KeyIndex ki,
                   SpecialInfo* out, cudaStream_t st) {
    const u64 m = n_rec * 32;
    if (m <= kSpecialAllPairs) {
        special_scan_kernel<<<(unsigned)m, 128, 0, st>>>(words, d_seps, n_rec, sorted, n_keys, ki, out);
        DEBWT_COUNT(1);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (m >= SPEC_INF) { set_error("too many records for the sentinel-window sort (32 R must be below 2^32)"); return -1; }
    u64 mp2 = 1;
    while (mp2 < m) mp2 <<= 1;
    u32* ids = nullptr;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&ids), mp2 * 4, st));
    special_ids_kernel<<<grid_for(mp2, TPB), TPB, 0, st>>>(ids, m, mp2);
    unsigned launches = 1;
    for (u64 k = 2; k <= mp2; k <<= 1)
        for (u64 j = k >> 1; j > 0; j >>= 1) {
            special_bitonic_kernel<<<grid_for(mp2, TPB), TPB, 0, st>>>(ids, mp2, j, k, words, d_seps, n_rec);
            ++launches;
        }
    special_info_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(ids, m, words, d_seps, sorted, n_keys, ki, out);
    DEBWT_COUNT(launches + 1);
    const cudaError_t e = cudaGetLastError();
    cudaFreeAsync(ids, st);
    if (e != cudaSuccess) { set_error(std::string("sentinel-window sort: ") + cudaGetErrorString(e)); return -1; }
    return 0;
}

int k_special_insertion(const u64* sorted, u64 n, KeyIndex ki, const u64* pads, u64 m, u64* ins, cudaStream_t st) {
    if (m == 0) return 0;
    special_ins_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(sorted, n, ki, pads, m, ins);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// =============================================================================================
// K9: branch codes and blue entries             (src/generateSP.c:534-683)
// =============================================================================================
namespace {

// Memory-level parallelism by hand: a thread first issues the presence-filter reads of its 16 positions together, then the
// hash-table probes of the positions that passed, four at a time (the straightforward loop kept one dependent read in
// flight per thread and spent 60 % of its time waiting for the filter and the probe).  No block-wide compaction: the
// candidates of a thread are a 16-bit mask.
constexpr int FP_BATCH = 4;                // 8 measured slower (registers)
__global__ void __launch_bounds__(TPB) flag_positions_kernel(const u64* __restrict__ words, u64 nwords_total, u64 n,
                                                            const u64* __restrict__ seps, u64 n_rec, BranchTable bt,
                                                            u32* __restrict__ mo_bits, u64* __restrict__ blue) {
    __shared__ TileText t;
    const u64 base = (u64)blockIdx.x * TILE_POS;
    tile_load(t, words, nwords_total, base, n, seps, n_rec);
    const bool one_record = t.rec_first == t.rec_last;
    const u32* __restrict__ filter = bt.filter();
    u32 cand = 0, mo_mask = 0;                               // bit j: position j * TPB + tid
    if (one_record && bt.hslots) {
        u32 fi[TILE_ROWS], fw[TILE_ROWS];
#pragma unroll
        for (int j = 0; j < TILE_ROWS; ++j) {
            const u32 local = j * TPB + threadIdx.x;
            const u64 p = base + local;
            const bool ok = p < n && t.rec_first < n_rec && p + KMER <= t.sep_first;
            fi[j] = ok ? (u32)bt.filter_of(tile_window(t, local)) : 0xFFFFFFFFu;
        }
#pragma unroll
        for (int j = 0; j < TILE_ROWS; ++j) fw[j] = ld_nc_u32(filter + (fi[j] == 0xFFFFFFFFu ? 0u : fi[j] >> 5));
#pragma unroll
        for (int j = 0; j < TILE_ROWS; ++j)
            if (fi[j] != 0xFFFFFFFFu && ((fw[j] >> (fi[j] & 31)) & 1u)) cand |= 1u << j;
        const u64 hmask = (1ull << bt.hbits) - 1;
        while (cand) {
            u32 loc[FP_BATCH];
            u64 x[FP_BATCH], hs[FP_BATCH];
            ulonglong2 v[FP_BATCH];
#pragma unroll
            for (int u = 0; u < FP_BATCH; ++u) {
                loc[u] = 0xFFFFFFFFu;
                x[u] = 0; hs[u] = 0;
                if (cand) {
                    const int j = __ffs(cand) - 1;
                    cand &= cand - 1;
                    loc[u] = j * TPB + threadIdx.x;
                    x[u] = tile_window(t, loc[u]) & ~3ull;
                    hs[u] = bt.hash_of(x[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < FP_BATCH; ++u) v[u] = ld_nc_u64x2(bt.hslots + hs[u]);
#pragma unroll
            for (int u = 0; u < FP_BATCH; ++u) {
                if (loc[u] == 0xFFFFFFFFu) continue;
                while (v[u].x != 0 && (v[u].x & ~3ull) != x[u]) {      // collision: next slot
                    hs[u] = (hs[u] + 1) & hmask;
                    v[u] = __ldg(bt.hslots + hs[u]);
                }
                if (v[u].x == 0) continue;
                const u32 f = (u32)(v[u].x & 3ull);
                if (f & 1u) mo_mask |= 1u << (loc[u] / TPB);
                if (f & 2u) {
                    const u64 p = base + loc[u];
                    u32 prev;
                    if (p == t.start_first) prev = t.rec_first ? 4u : 5u;      // '#' / '$'   (src/generateSP.c:584-605)
                    else prev = text_symbol(words, p - 1);
                    u64 at;
                    if (bt.hmode) {                                            // offset and cursor live in the slot just read
                        const unsigned long long old = atomicAdd(reinterpret_cast<unsigned long long*>(&bt.hslots[hs[u]].y), 1ull);
                        at = (old >> 32) + (old & 0xFFFFFFFFull);
                    } else {
                        const u64 b = v[u].y;
                        at = (u64)bt.blue[b] + atomicAdd(bt.cursor + b, 1u);
                    }
                    blue[at] = (p << 4) | prev;
                }
            }
        }
    } else {
#pragma unroll 1
        for (int j = 0; j < TILE_ROWS; ++j) {
            const u32 local = j * TPB + threadIdx.x;
            const u64 p = base + local;
            if (p >= n) continue;
            u64 r = t.rec_first, sep = t.sep_first, start = t.start_first;
            bool in_text = r < n_rec;
            if (!one_record) {
                r = record_of(seps, n_rec, p);
                in_text = r < n_rec;
                if (in_text) { sep = seps[r]; start = r ? seps[r - 1] + 1 : 0; }
            }
            if (!(in_text && p + KMER <= sep)) continue;
            const u64 x = tile_window(t, local) & ~3ull;
            u64 b;
            u32 f;
            if (!branch_lookup(bt, x, b, f)) continue;
            if (f & 1u) mo_mask |= 1u << j;
            if (f & 2u) {
                u32 prev;
                if (p == start) prev = r ? 4u : 5u;                 // '#' / '$'   (src/generateSP.c:584-605)
                else prev = text_symbol(words, p - 1);
                u64 at;
                if (bt.hslots && bt.hmode) {
                    const unsigned long long old = atomicAdd(reinterpret_cast<unsigned long long*>(&bt.hslots[b].y), 1ull);
                    at = (old >> 32) + (old & 0xFFFFFFFFull);
                } else {
                    at = (u64)bt.blue[b] + atomicAdd(bt.cursor + b, 1u);
                }
                blue[at] = (p << 4) | prev;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < TILE_ROWS; ++j) {
        const u64 p = base + (u64)j * TPB + threadIdx.x;
        const u32 bal = __ballot_sync(0xffffffffu, (mo_mask >> j) & 1u);
        if ((threadIdx.x & 31) == 0 && p < n + 32) mo_bits[p >> 5] = bal;
    }
}

// K9 with the blue entries grouped by a sort instead of per-segment cursors: every multi-in position appends one key
//   (branch id << shift) | (position << 4) | 8 | prev          (shift >= 36; the branch id ends at bit 63)
// to a dense array -- one atomic per 4096-position block, coalesced stores -- and the radix passes over the bits from
// `shift` up group the keys by branch id, i.e. into their segments (the order inside a segment is K10's business).
// Replaces 517 M cursor atomics and scattered 8-byte stores at 3.1 Gbp.  Needs N < 2^32 and at most 2^28 branch k-mers.
// The lookups are staged so that many of them are in flight per thread: (A) the 16 presence-filter reads of a thread are
// independent loads; (B) the positions that pass are compacted into a shared-memory list; (C) the index / table reads of four
// list entries per thread are issued together; the keys are collected in shared memory and leave with one atomic per block.
constexpr int FK_UNROLL = 4;
__global__ void __launch_bounds__(TPB) flag_positions_keys_kernel(const u64* __restrict__ words, u64 nwords_total, u64 n,
                                                                 const u64* __restrict__ seps, u64 n_rec, BranchTable bt,
                                                                 int shift, u32* __restrict__ mo_bits, u64* __restrict__ bkeys,
                                                                 unsigned long long* __restrict__ counter) {
    __shared__ TileText t;
    __shared__ u64 s_keys[TILE_POS];
    __shared__ u16 s_hits[TILE_POS];
    __shared__ u32 s_mo[TILE_WORDS];
    __shared__ u32 s_cnt[TILE_ROWS][TPB / 32];
    __shared__ u32 s_nhits, s_nkeys;
    __shared__ u64 s_base;
    const u64 base = (u64)blockIdx.x * TILE_POS;
    tile_load(t, words, nwords_total, base, n, seps, n_rec);
    const bool one_record = t.rec_first == t.rec_last;
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < TILE_WORDS) s_mo[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_nkeys = 0;
    // ---- (A) presence filter of every clean position of the tile ----
    const u32* __restrict__ filter = bt.filter();
    u32 fw[TILE_ROWS];
    if (one_record) {
        // addresses first, then all loads (asm volatile keeps them together and in order: 16 requests in flight per thread),
        // then the bit tests
        u32 fi[TILE_ROWS];
#pragma unroll
        for (int j = 0; j < TILE_ROWS; ++j) {
            const u32 local = j * TPB + threadIdx.x;
            const u64 p = base + local;
            const bool ok = p < n && t.rec_first < n_rec && p + KMER <= t.sep_first;
            fi[j] = ok ? (u32)bt.filter_of(tile_window(t, local)) : 0xFFFFFFFFu;
        }
#pragma unroll
        for (int j = 0; j < TILE_ROWS; ++j) fw[j] = ld_nc_u32(filter + (fi[j] == 0xFFFFFFFFu ? 0u : fi[j] >> 5));
#pragma unroll
        for (int j = 0; j < TILE_ROWS; ++j) fw[j] = fi[j] == 0xFFFFFFFFu ? 0u : (fw[j] >> (fi[j] & 31)) & 1u;
    } else {
#pragma unroll 1
        for (int j = 0; j < TILE_ROWS; ++j) {
            const u32 local = j * TPB + threadIdx.x;
            const u64 p = base + local;
            bool ok = p < n;
            if (ok) {
                const u64 r = record_of(seps, n_rec, p);
                ok = r < n_rec && p + KMER <= seps[r];
            }
            const u64 f = bt.filter_of(tile_window(t, local));
            fw[j] = ok ? (__ldg(filter + (f >> 5)) >> (f & 31)) & 1u : 0u;
        }
    }
    // ---- (B) compact the positions that passed ----
#pragma unroll
    for (int j = 0; j < TILE_ROWS; ++j) {
        const u32 bal = __ballot_sync(0xffffffffu, fw[j] != 0);
        if (lane == 0) s_cnt[j][warp] = __popc(bal);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 run = 0;
        for (int j = 0; j < TILE_ROWS; ++j)
            for (int w = 0; w < TPB / 32; ++w) { const u32 c = s_cnt[j][w]; s_cnt[j][w] = run; run += c; }
        s_nhits = run;
    }
    __syncthreads();
    const u32 lt = lanemask_lt();
#pragma unroll
    for (int j = 0; j < TILE_ROWS; ++j) {
        const u32 bal = __ballot_sync(0xffffffffu, fw[j] != 0);
        if (fw[j]) s_hits[s_cnt[j][warp] + __popc(bal & lt)] = (u16)(j * TPB + threadIdx.x);
    }
    __syncthreads();
    // ---- (C) branch-table lookups of the listed positions, FK_UNROLL per thread at a time ----
    const u32 nh = s_nhits;
    const u64 hmask = (1ull << bt.hbits) - 1;
    for (u32 c0 = 0; c0 < nh; c0 += TPB * FK_UNROLL) {
        u32 loc[FK_UNROLL];
        u64 x[FK_UNROLL], hs[FK_UNROLL], key[FK_UNROLL];
        ulonglong2 v[FK_UNROLL];
#pragma unroll
        for (int u = 0; u < FK_UNROLL; ++u) {
            const u32 h = c0 + u * TPB + threadIdx.x;
            loc[u] = h < nh ? s_hits[h] : 0xFFFFFFFFu;
            x[u] = loc[u] != 0xFFFFFFFFu ? tile_window(t, loc[u]) & ~3ull : 0;
            hs[u] = bt.hash_of(x[u]);
        }
#pragma unroll
        for (int u = 0; u < FK_UNROLL; ++u) v[u] = ld_nc_u64x2(bt.hslots + (loc[u] != 0xFFFFFFFFu ? hs[u] : 0));
#pragma unroll
        for (int u = 0; u < FK_UNROLL; ++u) {
            key[u] = 0;
            if (loc[u] == 0xFFFFFFFFu) v[u].x = 0;
            while (v[u].x != 0 && (v[u].x & ~3ull) != x[u]) {          // collision: next slot
                hs[u] = (hs[u] + 1) & hmask;
                v[u] = __ldg(bt.hslots + hs[u]);
            }
            if (v[u].x != 0) {
                const u32 f = (u32)(v[u].x & 3ull);
                if (f & 1u) atomicOr(&s_mo[loc[u] >> 5], 1u << (loc[u] & 31));
                if (f & 2u) {
                    const u64 p = base + loc[u];
                    u64 r = t.rec_first, rstart = t.start_first;
                    if (!one_record) {
                        r = record_of(seps, n_rec, p);
                        rstart = r ? seps[r - 1] + 1 : 0;
                    }
                    u32 prev;
                    if (p == rstart) prev = r ? 4u : 5u;                    // '#' / '$'   (src/generateSP.c:584-605)
                    else prev = text_symbol(words, p - 1);
                    key[u] = (v[u].y << shift) | (p << 4) | prev | 8ull;   // bit 3: "present" (id, p, prev may all be 0)
                }
            }
        }
#pragma unroll
        for (int u = 0; u < FK_UNROLL; ++u) {                          // warp-aggregated append to the block's key list
            const u32 bal = __ballot_sync(0xffffffffu, key[u] != 0);
            u32 slot = 0;
            if (lane == 0 && bal) slot = atomicAdd(&s_nkeys, (u32)__popc(bal));
            slot = __shfl_sync(0xffffffffu, slot, 0);
            if (key[u]) s_keys[slot + __popc(bal & lt)] = key[u];
        }
    }
    __syncthreads();
    if (threadIdx.x < TILE_WORDS && base + 32ull * threadIdx.x < n + 32) mo_bits[(base >> 5) + threadIdx.x] = s_mo[threadIdx.x];
    const u32 nk = s_nkeys;
    if (threadIdx.x == 0) s_base = nk ? atomicAdd(counter, (unsigned long long)nk) : 0;
    __syncthreads();
    const u64 bb = s_base;
    for (u32 i = threadIdx.x; i < nk; i += TPB) bkeys[bb + i] = s_keys[i];
}

// position -> spIndex inside the keys, in append order (positions nearly ascending: the bitmap and prefix reads are
// sequential, where after the grouping they would be random)
__global__ void __launch_bounds__(TPB) blue_keys_fix_kernel(u64* __restrict__ bkeys, u64 m, const u32* __restrict__ mo_bits,
                                                           const u32* __restrict__ word_prefix) {
    const u64 e = (u64)blockIdx.x * TPB + threadIdx.x;
    if (e >= m) return;
    const u64 v = bkeys[e];
    const u64 field = 0xFFFFFFFFull << 4;
    bkeys[e] = (v & ~field) | (sp_index_of(mo_bits, word_prefix, (v >> 4) & 0xFFFFFFFFull) << 4);
}

// grouped keys -> blue entries (spIndex << 4) | prev, in place
__global__ void __launch_bounds__(TPB) blue_keys_strip_kernel(u64* __restrict__ bkeys, u64 m) {
    const u64 e = (u64)blockIdx.x * TPB + threadIdx.x;
    if (e < m) bkeys[e] &= 0xFFFFFFFF7ull;
}

// patch_bits, emit_codes, mark_sep_codes and blue_fix see one position slice with codes from code_base (stages.cuh).
__global__ void __launch_bounds__(TPB) patch_bits_kernel(u32* __restrict__ mo_bits, u64 pos_lo, u64 pos_hi,
                                                        const u64* __restrict__ pos, u64 m) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= m) return;
    const u64 p = pos[t];
    if (p < pos_lo || p >= pos_hi) return;
    atomicOr(mo_bits + ((p - pos_lo) >> 5), 1u << (p & 31));
}

__global__ void __launch_bounds__(TPB) emit_codes_kernel(const u64* __restrict__ words, u64 word_lo, u64 nbw,
                                                        const u32* __restrict__ mo_bits, const u32* __restrict__ word_prefix,
                                                        u64 code_base, u64* __restrict__ sp_codes) {
    const u64 wl = (u64)blockIdx.x * TPB + threadIdx.x;
    if (wl >= nbw) return;
    u32 bits = mo_bits[wl];
    if (!bits) return;
    // next symbols of positions 32w+b are text positions 32w+31+b: last symbol of word w, then word w+1
    const u64 w = word_lo + wl;
    const u64 w0 = words[w], w1 = words[w + 1];
    u64 c = code_base + word_prefix[wl];
    u64 acc = 0, acc_word = c >> 5;
    while (bits) {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        const u64 code = (b == 0) ? (w0 & 3ull) : ((w1 >> (2 * (32 - b))) & 3ull);
        const u64 cw = c >> 5;
        if (cw != acc_word) {
            if (acc) atomicOr(sp_codes + acc_word, acc);
            acc = 0; acc_word = cw;
        }
        acc |= code << (2 * (31 - (c & 31)));
        ++c;
    }
    if (acc) atomicOr(sp_codes + acc_word, acc);
}

// separator codes of the tail positions that fall into the slice; index of each written to out_idx (entries of other
// slices get 0)
__global__ void __launch_bounds__(TPB) mark_sep_codes_kernel(const u32* __restrict__ mo_bits, const u32* __restrict__ word_prefix,
                                                            u64 pos_lo, u64 pos_hi, u64 code_base,
                                                            const u64* __restrict__ pos, u64 m, u32* __restrict__ sp_sep,
                                                            u64* __restrict__ out_idx) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t >= m) return;
    const u64 p = pos[t];
    if (p < pos_lo || p >= pos_hi) { out_idx[t] = 0; return; }
    const u64 c = code_base + sp_index_of(mo_bits, word_prefix, p - pos_lo);
    atomicOr(sp_sep + (c >> 5), 1u << (c & 31));
    out_idx[t] = c;
}

__global__ void __launch_bounds__(TPB) blue_fix_kernel(u64* __restrict__ blue, u64 m, const u32* __restrict__ mo_bits,
                                                      const u32* __restrict__ word_prefix, u64 pos_lo, u64 code_base) {
    const u64 e = (u64)blockIdx.x * TPB + threadIdx.x;
    if (e >= m) return;
    const u64 v = blue[e];
    blue[e] = ((code_base + sp_index_of(mo_bits, word_prefix, (v >> 4) - pos_lo)) << 4) | (v & 15ull);
}

// The entries sit in their segments, i.e. in no order of position: every one of them reads the bitmap word and the prefix
// of its position at random.  With the two interleaved -- (prefix << 32) | bits per 32 positions -- that is one sector
// instead of two (87 GB -> half of HBM reads for 517 M entries at 3.1 Gbp).
__global__ void __launch_bounds__(TPB) interleave_kernel(const u32* __restrict__ mo_bits, const u32* __restrict__ word_prefix, u64 nw,
                                                        u64* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * TPB + threadIdx.x;
    if (i < nw) out[i] = ((u64)word_prefix[i] << 32) | mo_bits[i];
}

__global__ void __launch_bounds__(TPB) blue_fix2_kernel(u64* __restrict__ blue, u64 m, const u64* __restrict__ bits_prefix) {
    const u64 e = (u64)blockIdx.x * TPB + threadIdx.x;
    if (e >= m) return;
    const u64 v = blue[e];
    const u64 p = v >> 4;
    const u64 w = __ldg(bits_prefix + (p >> 5));
    const u64 sp = (w >> 32) + __popc((u32)w & ((1u << (p & 31)) - 1u));
    blue[e] = (sp << 4) | (v & 15ull);
}

}  // namespace

int k_flag_positions(const u64* words, u64 n, const u64* d_seps, u64 n_rec, BranchTable bt, u32* mo_bits, u64* blue,
                     cudaStream_t st) {
    flag_positions_kernel<<<grid_for(n, TILE_POS), TPB, 0, st>>>(words, text_words(n), n, d_seps, n_rec, bt, mo_bits, blue);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_flag_positions_keys(const u64* words, u64 n, const u64* d_seps, u64 n_rec, BranchTable bt, int shift, u32* mo_bits,
                          u64* bkeys, u64* d_counter, cudaStream_t st) {
    flag_positions_keys_kernel<<<grid_for(n, TILE_POS), TPB, 0, st>>>(words, text_words(n), n, d_seps, n_rec, bt, shift, mo_bits, bkeys,
                                                                      reinterpret_cast<unsigned long long*>(d_counter));
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_blue_keys_fix(u64* bkeys, u64 m, const u32* mo_bits, const u32* word_prefix, cudaStream_t st) {
    if (m == 0) return 0;
    blue_keys_fix_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(bkeys, m, mo_bits, word_prefix);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_blue_keys_strip(u64* bkeys, u64 m, cudaStream_t st) {
    if (m == 0) return 0;
    blue_keys_strip_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(bkeys, m);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_patch_bits(u32* mo_bits, u64 pos_lo, u64 pos_hi, const u64* positions, u64 m, cudaStream_t st) {
    if (m == 0) return 0;
    patch_bits_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(mo_bits, pos_lo, pos_hi, positions, m);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_emit_codes(const u64* words, u64 word_lo, u64 nbw, const u32* mo_bits, const u32* word_prefix, u64 code_base,
                 u64* sp_codes, cudaStream_t st) {
    if (nbw == 0) return 0;
    emit_codes_kernel<<<grid_for(nbw, TPB), TPB, 0, st>>>(words, word_lo, nbw, mo_bits, word_prefix, code_base, sp_codes);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_mark_sep_codes(const u32* mo_bits, const u32* word_prefix, u64 pos_lo, u64 pos_hi, u64 code_base, const u64* positions,
                     u64 m, u32* sp_sep, u64* d_code_index_out, cudaStream_t st) {
    if (m == 0) return 0;
    mark_sep_codes_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(mo_bits, word_prefix, pos_lo, pos_hi, code_base, positions, m, sp_sep,
                                                            d_code_index_out);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_blue_fix_interleaved(u64* blue, u64 m, const u32* mo_bits, const u32* word_prefix, u64 n_words, u64* scratch, cudaStream_t st) {
    if (m == 0) return 0;
    interleave_kernel<<<grid_for(n_words, TPB), TPB, 0, st>>>(mo_bits, word_prefix, n_words, scratch);
    blue_fix2_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(blue, m, scratch);
    DEBWT_COUNT(2);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_blue_fix(u64* blue, u64 m, const u32* mo_bits, const u32* word_prefix, u64 pos_lo, u64 code_base, cudaStream_t st) {
    if (m == 0) return 0;
    blue_fix_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(blue, m, mo_bits, word_prefix, pos_lo, code_base);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// =============================================================================================
// K8 / K11: emission                             (src/INandOut.c:367-395, src/insertCase3.c:56-104)
// =============================================================================================
namespace {

constexpr int FILL_WORDS_PER_WARP = 32;

// output words [word_lo, word_hi); gmask holds the n_keys sorted keys from global key index key_base on
__global__ void __launch_bounds__(TPB) fill_case2_kernel(const u16* __restrict__ gmask, u64 n_keys, u64 key_base, u64 n,
                                                        const u64* __restrict__ spec_rows, u64 m, u64 word_lo, u64 word_hi,
                                                        u64* __restrict__ bwt) {
    __shared__ u64 s_lo, s_hi;
    constexpr int WORDS_PER_BLOCK = (TPB / 32) * FILL_WORDS_PER_WARP;
    const u64 wblock = word_lo + (u64)blockIdx.x * WORDS_PER_BLOCK;
    if (threadIdx.x == 0) s_lo = lower_bound_u64(spec_rows, 0, m, wblock * 32);
    if (threadIdx.x == 32) s_hi = lower_bound_u64(spec_rows, 0, m, (wblock + WORDS_PER_BLOCK) * 32);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u64 lo = s_lo, hi = s_hi;
#pragma unroll 4
    for (int q = 0; q < FILL_WORDS_PER_WARP; ++q) {
        const u64 w = wblock + (u64)warp * FILL_WORDS_PER_WARP + q;
        if (w >= word_hi) break;                      // warp-uniform
        const u64 row = w * 32 + lane;
        u32 code = 0;
        if (row < n) {
            const u64 t = lower_bound_u64(spec_rows, lo, hi, row);   // special rows before this row
            const bool special = t < m && spec_rows[t] == row;
            // index into this device's keys; the rows of keys below key_base wrap around to values far above n_keys
            const u64 i = row - t - key_base;
            if (!special && i < n_keys) {
                const u32 mk = gmask[i];
                if (!gm_multi_in(mk) && (mk & 15u)) code = (u32)__ffs(mk & 15u) - 1u;   // the single in-base (src/INandOut.c:367-395)
            }
        }
        const u32 hi32 = __reduce_or_sync(0xffffffffu, lane < 16 ? code << (2 * (15 - lane)) : 0u);
        const u32 lo32 = __reduce_or_sync(0xffffffffu, lane >= 16 ? code << (2 * (31 - lane)) : 0u);
        if (lane == 0) bwt[w] = ((u64)hi32 << 32) | lo32;
    }
}

// A block owns EB_ITEMS * TPB consecutive blue entries.  Their segments are consecutive branch entries and their rows
// ascend, so the block looks up the branch range and the sentinel range of its first and last entry once, and every
// entry only searches inside those (a handful of steps instead of log2(B) + log2(32 R) per entry).
constexpr int EB_ITEMS = 8;
__global__ void __launch_bounds__(TPB) emit_blue_kernel(const u64* __restrict__ blue, BranchTable bt, u64 key_base,
                                                       const u64* __restrict__ spec_ins, u64 m, u64* __restrict__ bwt,
                                                       u64* __restrict__ sharp_rows, u32* __restrict__ sharp_count,
                                                       u64* __restrict__ dollar_row) {
    __shared__ u64 s_b[2], s_t[2];
    const u64 e0 = (u64)blockIdx.x * (EB_ITEMS * TPB);
    const u64 e1 = e0 + EB_ITEMS * TPB < bt.n_blue ? e0 + EB_ITEMS * TPB : bt.n_blue;      // exclusive
    if (threadIdx.x < 2) {
        // segment = last branch entry whose blue offset is <= e
        const u64 e = threadIdx.x == 0 ? e0 : e1 - 1;
        u64 lo = 0, hi = bt.n_branch;
        while (lo < hi) {
            const u64 mid = (lo + hi) >> 1;
            if ((u64)bt.blue[mid] <= e) lo = mid + 1; else hi = mid;
        }
        const u64 b = lo - 1;
        s_b[threadIdx.x] = b;
        s_t[threadIdx.x] = upper_bound_u64(spec_ins, 0, m, key_base + (u64)bt.head[b] + (e - bt.blue[b]));
    }
    __syncthreads();
    const u64 b_lo = s_b[0], b_hi = s_b[1], t_lo = s_t[0], t_hi = s_t[1];
#pragma unroll
    for (int j = 0; j < EB_ITEMS; ++j) {
        const u64 e = e0 + (u64)j * TPB + threadIdx.x;
        if (e >= e1) break;
        u64 lo = b_lo, hi = b_hi + 1;                        // the answer lies in [b_lo, b_hi]
        while (lo < hi) {
            const u64 mid = (lo + hi) >> 1;
            if ((u64)bt.blue[mid] <= e) lo = mid + 1; else hi = mid;
        }
        const u64 b = lo - 1;
        const u64 i = key_base + (u64)bt.head[b] + (e - bt.blue[b]);
        const u64 row = i + upper_bound_u64(spec_ins, t_lo, t_hi, i);
        const u32 c = (u32)(blue[e] & 15ull);
        if (c >= 4) {
            if (c == 4) sharp_rows[atomicAdd(sharp_count, 1u)] = row; else *dollar_row = row;
            bwt_or(bwt, row, 3u);                                   // '#'/'$' stored as T (src/insertCase3.c:84-95)
        } else if (c) {
            bwt_or(bwt, row, c);
        }
    }
}

__global__ void __launch_bounds__(TPB) emit_special_kernel(const u64* __restrict__ rows, const u8* __restrict__ chr, u64 m,
                                                          u64* __restrict__ bwt) {
    const u64 t = (u64)blockIdx.x * TPB + threadIdx.x;
    if (t < m && chr[t]) bwt_or(bwt, rows[t], chr[t]);
}

}  // namespace

int k_fill_case2(const u16* gmask, u64 n_keys, u64 key_base, u64 n, const u64* spec_rows, u64 m, u64 word_lo, u64 word_hi,
                 u64* bwt, cudaStream_t st) {
    if (word_hi <= word_lo) return 0;
    constexpr int WORDS_PER_BLOCK = (TPB / 32) * FILL_WORDS_PER_WARP;
    fill_case2_kernel<<<grid_for(word_hi - word_lo, WORDS_PER_BLOCK), TPB, 0, st>>>(gmask, n_keys, key_base, n, spec_rows, m,
                                                                                    word_lo, word_hi, bwt);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_emit_blue(const u64* blue, BranchTable bt, u64 key_base, const u64* spec_ins, u64 m, u64* bwt, u64* sharp_rows,
                u32* d_sharp_count, u64* dollar_row, cudaStream_t st) {
    if (bt.n_blue == 0) return 0;
    emit_blue_kernel<<<grid_for(bt.n_blue, EB_ITEMS * TPB), TPB, 0, st>>>(blue, bt, key_base, spec_ins, m, bwt, sharp_rows,
                                                                          d_sharp_count, dollar_row);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_emit_special(const u64* spec_rows, const u8* spec_chr, u64 m, u64* bwt, cudaStream_t st) {
    if (m == 0) return 0;
    emit_special_kernel<<<grid_for(m, TPB), TPB, 0, st>>>(spec_rows, spec_chr, m, bwt);
    DEBWT_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

}  // namespace debwt
