// Device stages of the deBWT-B200 pipeline other than the radix sort (see DESIGN.md section 4).
#pragma once
#include "common.cuh"

namespace debwt {

// ---- generic exclusive scan of u32 values (optionally popcounts of the input words) -----------
size_t scan_workspace_bytes(u64 m);
// out[i] = sum_{j<i} f(in[j]), f = identity or popc; *d_total (device u64) = sum of all
int scan_exclusive_u32(const u32* in, u32* out, u64 m, bool popc, void* workspace, u64* d_total, cudaStream_t st);

// ---- K1 / K2 ------------------------------------------------------------------------------
// ascii: n bytes (bases, '#' between records, '$' last).  A whole text packs into text_words(n) u64.
// what K1 does with a symbol that is not A, C, G or T: reject (default), or resolve IUPAC ambiguity codes to a seeded
// pseudo-random compatible base (reference otherTool/transferN.c); pos_base = text position of ascii[0]
struct PackPolicy {
    bool resolve = false;
    u64 seed = 0;
    u64 pos_base = 0;
};
inline u64 text_words(u64 n) { return (n + 32 + 31) / 32 + 1; }
// packs n symbols into nwords words (T padding for [n, n+32), zeros beyond): a whole text, or the slice of one
int k_pack_words(const u8* ascii, u64 n, u64* words, u64 nwords, u32* d_err, cudaStream_t st, PackPolicy pol = PackPolicy());
// all in-record 32-mers; key index of window p in record r is p - 32 r.  keys: n - 32 R entries.
int k_extract(const u64* words, u64 n, const u64* d_seps, u64 n_rec, u64* keys, cudaStream_t st);
// the same for the positions [pos_lo, pos_hi) only (pos_lo a multiple of 32); key index = p - 32 r - idx_base
int k_extract_slice(const u64* words, u64 n, u64 pos_lo, u64 pos_hi, const u64* d_seps, u64 n_rec, u64 idx_base, u64* keys,
                    cudaStream_t st);

// [8][256] digit counts of the keys k_extract writes, computed from the packed text (see stages.cu); applies when the
// per-record corrections are negligible next to the sweep.
bool text_digit_hist_applies(u64 n, u64 n_rec);
int k_text_digit_hist(const u64* words, u64 n, const u64* d_seps, u64 n_rec, u64* ghist, cudaStream_t st);

// ---- K4 count-by-sort (API parity with the reference's kmerInfo records) -------------------
// returns D through *d_total; kmers/counts sized >= n
int k_rle(const u64* sorted, u64 n, u64* kmers, u64* counts, void* workspace, u64* d_total, cudaStream_t st);
size_t rle_workspace_bytes(u64 n);

// ---- direct index over the sorted keys (the reference's 4^12 bucket table, src/mySort.c:98-103) ----
struct KeyIndex {
    u32* idx = nullptr;   // [2^bits + 1]: idx[t] = first sorted position whose top `bits` bits are >= t
    int bits = 0;
};
inline int key_index_bits(u64 n) {
    int b = 8;
    while (b < 28 && (8ull << b) < n) ++b;      // about 8 keys per bucket (12 at 3.1 G keys: a 1 GB table; 2^29 measured slower)
    return b;
}
int k_build_key_index(const u64* sorted, u64 n, KeyIndex ki, cudaStream_t st);
// the same in two steps around a sort whose last pass marks the buckets (SortWorkspace::key_index)
int k_key_index_init(KeyIndex ki, cudaStream_t st);
int k_key_index_finish(const u64* sorted, u64 n, KeyIndex ki, bool marked, cudaStream_t st);
__host__ __device__ __forceinline__ u64 indexed_lower_bound(const u64* __restrict__ k, const KeyIndex& ki, u64 q) {
    const u64 t = q >> (64 - ki.bits);
    return lower_bound_u64(k, ki.idx[t], ki.idx[t + 1], q);
}
__host__ __device__ __forceinline__ u64 indexed_upper_bound(const u64* __restrict__ k, const KeyIndex& ki, u64 q) {
    const u64 t = q >> (64 - ki.bits);
    return upper_bound_u64(k, ki.idx[t], ki.idx[t + 1], q);
}

// ---- K5..K7 branch k-mer detection ---------------------------------------------------------
int k_mark_edges(const u64* sorted, u64 n, KeyIndex ki, u16* gmask, cudaStream_t st);
int k_mark_heads_tails(const u64* words, const u64* d_seps, u64 n_rec, const u64* sorted, u64 n, KeyIndex ki, u16* gmask,
                       cudaStream_t st);
int k_propagate(const u64* sorted, u64 n, u16* gmask, cudaStream_t st);

struct BranchTable {
    u64 n_branch = 0;      // B
    u64 n_blue = 0;        // M
    u64* kmer = nullptr;   // [B]  (k-mer << 2) | multi_in << 1 | multi_out, ascending
    u32* head = nullptr;   // [B]  index of the group's first sorted key
    u32* blue = nullptr;   // [B+1] exclusive prefix of blue-segment sizes (0 for non multi-in)
    u32* cursor = nullptr; // [B]  fill cursor per segment
    u32* bidx = nullptr;   // [2^bits + 2] direct index on the top `bits` bits of the k-mer, followed by the
                           // presence bitmap: one bit per value of filter_of(k-mer), a filter_bits(bits)-bit HASH of the
                           // k-mer (a prefix would let every k-mer of a repeat family through: its branch k-mers share
                           // their first bases with the family's other k-mers)
    int bits = 0;
    // optional hash table over the k-mers (k_branch_hash): slot.x = kmer entry (never 0: a branch entry has a flag set;
    // 0 = empty slot), linear probing.  Branch k-mers of a repeat family share long prefixes, so the buckets of the direct
    // index get deep there (ten dependent reads per lookup at human scale); a probe is one 16-byte read.
    // slot.y: hmode 0 = branch id; hmode 1 = (blue offset << 32) | fill cursor of the k-mer's segment, so that K9 claims the
    // place of a blue entry with one 64-bit atomic on the sector it has just read (no reads of blue[] / cursor[]).
    ulonglong2* hslots = nullptr;
    int hbits = 0;
    int hmode = 0;
    __host__ __device__ static int hash_bits(u64 n_branch) { int b = 10; while (b < 40 && (1ull << b) < 3 * n_branch) ++b; return b; }
    __host__ __device__ u64 hash_of(u64 x) const { return ((x >> 2) * 0x9E3779B97F4A7C15ull) >> (64 - hbits); }
    __host__ __device__ u64 filter_of(u64 x) const { return ((x >> 2) * 0x9E3779B97F4A7C15ull) >> (64 - filter_bits(bits)); }
    __host__ __device__ static int filter_bits(int bits) { return bits + 3 < 30 ? bits + 3 : 30; }
    __host__ __device__ static u64 index_words(int bits) { return (1ull << bits) + 2 + (1ull << (filter_bits(bits) - 5)); }
    __host__ __device__ u32* filter() const { return bidx + (1ull << bits) + 2; }
};
size_t branch_workspace_bytes(u64 n);
// pass 1: counts (B, M) -> d_totals[0], d_totals[1]
// `propagate`: also copy every group head's mask to the other members of its group (replaces k_propagate)
int k_branch_count(const u64* sorted, u64 n, u16* gmask, bool propagate, void* workspace, u64* d_totals, cudaStream_t st);
// pass 2: fills kmer/head/blue (arrays must be allocated from the counts)
int k_branch_write(const u64* sorted, u64 n, const u16* gmask, void* workspace, BranchTable bt, cudaStream_t st);
int k_branch_index(BranchTable bt, cudaStream_t st);
// fills bt.hslots (2^hbits slots of 16 bytes, allocated by the caller) from bt.kmer
int k_branch_hash(BranchTable bt, cudaStream_t st);

// ---- sentinel-window ("special") suffixes --------------------------------------------------
// ins[t] = upper_bound(sorted, pad[t]) for t < m
int k_special_insertion(const u64* sorted, u64 n, KeyIndex ki, const u64* pads, u64 m, u64* ins, cudaStream_t st);

// ---- K9 branch codes + blue entries --------------------------------------------------------
// mo_bits: ceil(n/32)+1 u32 words; blue: M u64 entries (position << 4 | prev)
int k_flag_positions(const u64* words, u64 n, const u64* d_seps, u64 n_rec, BranchTable bt, u32* mo_bits, u64* blue,
                     cudaStream_t st);
// the same with the blue entries appended as (branch id << shift | position << 4 | 8 | prev) keys to a dense array
// (*d_counter, zeroed, ends up as their number).  k_blue_keys_fix turns the positions into spIndex while the keys are still
// in append order, a radix sort on the bits from `shift` up groups them into their segments, k_blue_keys_strip leaves the
// blue entries (spIndex << 4) | prev.  Needs N < 2^32, shift >= 36.
int k_flag_positions_keys(const u64* words, u64 n, const u64* d_seps, u64 n_rec, BranchTable bt, int shift, u32* mo_bits,
                          u64* bkeys, u64* d_counter, cudaStream_t st);
int k_blue_keys_fix(u64* bkeys, u64 m, const u32* mo_bits, const u32* word_prefix, cudaStream_t st);
int k_blue_keys_strip(u64* bkeys, u64 m, cudaStream_t st);
// blue entries: position -> spIndex (k_blue_fix), or the same through an interleaved copy of the bitmap and its prefix
// (scratch: n_words u64, n_words = words of mo_bits) when there are enough entries to pay for the copy
int k_blue_fix_interleaved(u64* blue, u64 m, const u32* mo_bits, const u32* word_prefix, u64 n_words, u64* scratch, cudaStream_t st);
// The calls below also serve the sharded build, which produces the codes of one position slice [pos_lo, pos_hi) (pos_lo a
// multiple of 32, word_lo = pos_lo / 32) at global code indices from code_base: mo_bits and word_prefix cover the slice
// only.  The single-GPU build passes pos_lo = word_lo = code_base = 0 and the whole text.
// sets the bits of the positions inside the slice; the others are skipped
int k_patch_bits(u32* mo_bits, u64 pos_lo, u64 pos_hi, const u64* positions, u64 m, cudaStream_t st);
// sp_codes: ceil(S/32)+3 u64 zeroed; codes packed 32 per word, code j at bits 2*(31-(j&31)); nbw: words of the slice
int k_emit_codes(const u64* words, u64 word_lo, u64 nbw, const u32* mo_bits, const u32* word_prefix, u64 code_base,
                 u64* sp_codes, cudaStream_t st);
// marks separator codes: sp_sep bit per code (u32 words, zeroed); positions = tail positions whose code is '#'/'$'.
// d_code_index_out[t] = global code index of positions[t], or 0 for a position outside the slice
int k_mark_sep_codes(const u32* mo_bits, const u32* word_prefix, u64 pos_lo, u64 pos_hi, u64 code_base, const u64* positions,
                     u64 m, u32* sp_sep, u64* d_code_index_out, cudaStream_t st);
// every entry's position must lie in the slice
int k_blue_fix(u64* blue, u64 m, const u32* mo_bits, const u32* word_prefix, u64 pos_lo, u64 code_base, cudaStream_t st);

// ---- K10 segmented sort (bluesort.cu) ------------------------------------------------------
struct SpView {
    const u64* codes;   // 2-bit codes
    const u32* sep;     // 1 bit per code: code is '#' or '$'
    u64 dollar_index;   // index of the one '$' code
    u64 n_codes;        // S
    const u32* sep_sum = nullptr;   // optional (k_sort_blue builds it): bit j = some word of sep[32 j, 32 j + 32) is non-zero.  Only
                                    // R separator codes exist, so the one-fetch-per-entry sites test this 64 KB summary and
                                    // leave the S/8-byte bitmap alone (not the string walks: there the extra dependent load costs
                                    // more than the sector it saves)
};
int k_sort_blue(u64* blue, BranchTable bt, SpView sp, u32* d_work /* >= 4 B + 16 u32 */, cudaStream_t st);

// ---- K8 / K11 emission ---------------------------------------------------------------------
// bwt: ceil(n/32) words, indexed by global word number.  spec_rows: m ascending rows of the special suffixes.
// A device that owns the sorted keys [key_base, key_base + n_keys) (gmask: their masks) writes the words [word_lo, word_hi)
// of its rows; the single-GPU build passes key_base = 0 and all ceil(n/32) words.
int k_fill_case2(const u16* gmask, u64 n_keys, u64 key_base, u64 n, const u64* spec_rows, u64 m, u64 word_lo, u64 word_hi,
                 u64* bwt, cudaStream_t st);
// scatter sorted blue symbols; '#'/'$' rows appended to sharp_rows (unordered) / dollar_row.  bt.head is local to the
// device's keys, which start at global key index key_base.
int k_emit_blue(const u64* blue, BranchTable bt, u64 key_base, const u64* spec_ins, u64 m, u64* bwt, u64* sharp_rows,
                u32* d_sharp_count, u64* dollar_row, cudaStream_t st);
int k_emit_special(const u64* spec_rows, const u8* spec_chr, u64 m, u64* bwt, cudaStream_t st);

}  // namespace debwt
