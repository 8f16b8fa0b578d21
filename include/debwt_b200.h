/*
 * deBWT-B200 -- C ABI of the B200-native BWT-construction hot path.
 *
 * This is the drop-in boundary for the reference's stage functions (reference src/main.h:1-8,
 * sequenced by src/main.c:83-149).  The reference has no FFI; its "interface" is a linear pipeline of
 * C functions communicating through process-wide globals and temp files.  Each entry point below
 * names the reference interface it replaces.  Plain pointers and sizes only -- no CUDA, torch or C++
 * types -- so it binds from C (host/debwt_main.c), ctypes (debwt_b200/binding.py), cgo, JNI, ...
 *
 * Conventions: every function returns 0 on success and a negative value on error; the message is
 * available from debwt_last_error().  A context is bound to one CUDA device; calls on one context
 * are synchronous and not thread-safe (the reference's stages are not re-entrant either).  The
 * library owns all device memory.  There is no CPU fallback: without a CUDA device every call fails.
 */
#ifndef DEBWT_B200_H
#define DEBWT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct debwt_ctx debwt_ctx;

/* Per-phase device times (CUDA events on the library's stream) and sizes of the last build.
   Replaces the per-stage clock()/time() printfs of src/main.c:86-170. */
typedef struct debwt_stats {
    uint64_t n_symbols;      /* N = sum(len) + n_records            (BWTLEN, src/collect#$.c:56-57) */
    uint64_t n_records;
    uint64_t n_keys;         /* in-record 32-mer windows n' = N - 32 R */
    uint64_t n_branch;       /* branch k-mers (red table size)      (src/INandOut.c:396-417) */
    uint64_t n_blue;         /* occurrences of multi-in k-mers      (blueTable size) */
    uint64_t n_codes;        /* branch-code (SP) length S           (src/generateSP.c) */
    uint64_t n_special;      /* sentinel-window suffixes, 32 R */
    float ms_h2d;            /* host -> device copy of the ASCII text */
    float ms_pack;           /* K1 */
    float ms_extract;        /* K2 */
    float ms_sort;           /* K3: the named roofline phase (histogram + 8 scatter passes) */
    float ms_sort_sweeps;    /* K3: the scatter passes alone (onesweep_kernel launches) */
    float ms_classify;       /* K5-K7 */
    float ms_special;        /* sentinel-window suffix handling (device + host) */
    float ms_codes;          /* K9 */
    float ms_bluesort;       /* K10 */
    float ms_emit;           /* K8 + K11 */
    float ms_d2h;            /* device -> host copy of the result */
    float ms_total;          /* whole debwt_build() */
    uint32_t sort_launches;  /* kernel launches inside the sort phase */
    uint32_t sort_sweeps;    /* onesweep_kernel launches (8 unless a digit is constant) */
    uint32_t total_launches; /* kernel launches inside debwt_build() */
    uint32_t reserved_;
    uint64_t arena_bytes;      /* HBM held by the context's arena after the build (peak of the build) */
    uint64_t arena_used_bytes; /* of which in use at the high-water mark */
} debwt_stats;

const char* debwt_last_error(void);
/* number of CUDA devices visible (0 when the driver is missing) */
int debwt_device_count(void);
/* kernels launched by this library in this process so far (bookkeeping for the bench's gpu_launches) */
uint64_t debwt_launch_count(void);

/* ---- context ------------------------------------------------------------------------------ */
/* Replaces the process-wide globals of the reference (src/collect#$.h:17-18,31, generateSP.h:1-6,
   sortBlue.h:1-5, insertCase3.h:1-4).  `device` is the CUDA ordinal. */
int debwt_create(debwt_ctx** out, int device);
void debwt_destroy(debwt_ctx* ctx);
/* tuning knob for the sort kernel configuration (0 = default); returns the previous value */
int debwt_set_sort_config(debwt_ctx* ctx, int cfg);
/* how K9 brings the blue entries (src/generateSP.c:584-605) into their segments: 0 / 1 (default) = one cursor per segment
   (atomics + scattered stores), 2 = dense append + radix sort on the branch id (measured slower at 3.1 Gbp; kept, tested).
   Same output either way; returns the previous value */
int debwt_set_blue_grouping(debwt_ctx* ctx, int mode);

/* What to do with symbols other than A, C, G, T.  resolve = 0 (default): the build fails, like the reference asks of its
   input ("make sure your sequence don't contain any uncertain characters like 'N'", src/main.c:178).  resolve = 1: IUPAC
   ambiguity codes are replaced during K1 by one of the bases they stand for -- the tables of the reference's
   pre-processing tool (otherTool/transferN.c:8-27), with its time-seeded rand() replaced by splitmix64(seed, position),
   so that the same input and seed always give the same BWT; anything else still fails.  Set before the input. */
int debwt_set_ambiguity_policy(debwt_ctx* ctx, int resolve, uint64_t seed);

/* ---- input: replaces collect()'s FASTA pass, src/collect#$.c:27-90 ---------------------------- */
/* Host records: `seqs[i]` points at `lens[i]` bases (ACGT, either case; no terminator needed).
   Every record must be longer than 32 bp (src/collect#$.c:41-45) and contain only ACGT.
   The text T = S1 # S2 # ... Sn $ is assembled on the device (H2D copy happens here).
   Size limit of one device, checked by every input call (debwt_set_*, debwt_ingest_end) before anything is allocated:
   N < 2^32 - 64 symbols and N - 32 R < 2^32 - 65536 k-mer keys for R records, i.e. N <= min(2^32 - 65537 + 32 R,
   2^32 - 65); for one record N <= 2^32 - 65505.  Larger texts take the multi-GPU path. */
int debwt_set_records(debwt_ctx* ctx, const char* const* seqs, const uint64_t* lens, uint64_t n_records);
/* Same, from one host buffer that already holds T as ASCII ('#' between records, '$' last).
   `seps[i]` = offset of the i-th separator (ascending; the last one is n_symbols-1). */
int debwt_set_text(debwt_ctx* ctx, const char* text, uint64_t n_symbols, const uint64_t* seps, uint64_t n_records);
/* Same layout, but `d_text` is a DEVICE pointer on the context's device (no host copy); the buffer
   is only read, and must stay valid until debwt_build() returns. */
int debwt_set_text_device(debwt_ctx* ctx, const void* d_text, uint64_t n_symbols, const uint64_t* seps,
                          uint64_t n_records);

/* Streaming input: the text arrives in pieces while the file is still being read and decompressed.  The library keeps
   two pinned staging buffers; the caller writes the next symbols of T (ASCII bases, '#' between records, '$' last)
   straight into the window debwt_ingest_reserve() hands out and commits them; every full staging buffer is copied
   to the device and 2-bit packed (K1) on the library's stream while the caller fills the other one, so file reading,
   H2D and K1 overlap and the ASCII text is never resident on the device.  Replaces the TWO kseq passes of collect
   (src/collect#$.c:37-48 and :66-86).  n_symbols_hint: an upper bound of N when known (plain file size), 0 otherwise. */
int debwt_ingest_begin(debwt_ctx* ctx, uint64_t n_symbols_hint);
int debwt_ingest_reserve(debwt_ctx* ctx, char** buf, uint64_t* capacity);
int debwt_ingest_commit(debwt_ctx* ctx, uint64_t n_written);
/* reserve + memcpy + commit for a caller that already holds a piece of T */
int debwt_ingest_append(debwt_ctx* ctx, const char* chunk, uint64_t n);
/* seps as in debwt_set_text; N is what was committed */
int debwt_ingest_end(debwt_ctx* ctx, const uint64_t* seps, uint64_t n_records);
/* page-locked host memory for the result / input buffers of a C host (no CUDA headers needed there) */
void* debwt_host_alloc(uint64_t bytes);
void debwt_host_free(void* p);

/* ---- build: replaces mySort .. insertCase3, src/main.c:83-149 -------------------------------- */
/* `k` is the CLI -k value (12..32).  The output does not depend on it (SURVEY.md section 0); the
   device path always uses 32-base keys.  The result stays on the device until copied out. */
int debwt_build(debwt_ctx* ctx, int k);

/* ---- output: replaces insertCase3's three fwrite()s, src/insertCase3.c:115-131 ------------- */
int debwt_result_sizes(const debwt_ctx* ctx, uint64_t* n_symbols, uint64_t* n_words, uint64_t* n_sharp);
/* bwt_words: ceil(N/32) u64, symbol j at bits 2*(31-(j&31)) of word j>>5, '#'/'$' stored as T;
   sharp_rows: n_records-1 ascending rows holding '#'; dollar_row: the row holding '$'. */
int debwt_result_copy(debwt_ctx* ctx, uint64_t* bwt_words, uint64_t* sharp_rows, uint64_t* dollar_row);
int debwt_get_stats(const debwt_ctx* ctx, debwt_stats* out);

/* ---- multi-GPU: the sharded build, one rank per GPU (SURVEY.md section 8e; the reference has no distributed code) ----------
   SPMD: every rank -- a process started by torchrun / mpirun, or a thread -- creates its shard with the same group tag,
   passes ITS position slice of T (debwt_shard_slice) and the same separators to debwt_shard_build, and rank 0 ends up with
   the whole result.  Keys are range-partitioned by sampled splitters and stored straight into their owner's memory over
   NVLink; each rank sorts / classifies its key range and emits its own contiguous BWT segment.  same_process = 1 when the
   ranks are threads of one process (peer access instead of CUDA IPC). */
typedef struct debwt_shard debwt_shard;
typedef struct debwt_shard_stats {
    uint64_t n_symbols, n_records, n_keys;
    uint64_t n_keys_local;   /* keys this rank owns after the exchange */
    uint64_t n_branch, n_blue, n_codes;
    uint64_t arena_bytes;    /* HBM held by this rank's arena (shared exchange buffers not included) */
    float ms_total;          /* CUDA events on this rank's stream around the whole build */
    float ms_sort, ms_sort_sweeps;
    uint32_t sort_sweeps;
} debwt_shard_stats;
int debwt_shard_create(debwt_shard** out, int device, int rank, int world, const char* group_tag, int same_process);
void debwt_shard_destroy(debwt_shard* shard);
int debwt_shard_set_sort_config(debwt_shard* shard, int cfg);
/* [lo, hi) of T that rank `rank` of `world` uploads and works on */
int debwt_shard_slice(int rank, int world, uint64_t n_symbols, uint64_t* lo, uint64_t* hi);
/* collective; slice = T[lo .. hi) as ASCII, host or device memory */
int debwt_shard_build(debwt_shard* shard, const void* slice, int slice_on_device, uint64_t n_symbols, const uint64_t* seps,
                      uint64_t n_records);
/* rank 0 holds the result (other ranks: no-ops / NULL) */
int debwt_shard_result_device(const debwt_shard* shard, const uint64_t** d_bwt_words, uint64_t* n_words);
int debwt_shard_result_copy(debwt_shard* shard, uint64_t* bwt_words, uint64_t* sharp_rows, uint64_t* dollar_row);
int debwt_shard_get_stats(const debwt_shard* shard, debwt_shard_stats* out);
/* One call, one process, one thread per GPU: T in host memory in, the reference's three outputs out
   (what `deBWT -g 0,1,2,...` runs).  Replaces mySort .. insertCase3 (src/main.c:83-149) on several GPUs. */
int debwt_build_multi(const int* devices, int n_devices, const char* text, uint64_t n_symbols, const uint64_t* seps,
                      uint64_t n_records, uint64_t* bwt_words, uint64_t* sharp_rows, uint64_t* dollar_row, debwt_shard_stats* stats_out);

/* ---- FM-index tables over the result: the reference's "developer mode", src/insertCase3.c:139-208 ---------- */
/* occ checkpoints every 32 rows in the reference's layout -- occ[(N >> 5) + 1][4] u64, occ[w][c] = rows < 32 w holding
   base c, rows holding '#'/'$' (stored as T) not counted -- and the C-array (src/collect#$.c:92-100).  Built on the
   device from the result of debwt_build(); kept until the next build / input. */
int debwt_index_build(debwt_ctx* ctx);
int debwt_index_sizes(const debwt_ctx* ctx, uint64_t* occ_rows);
/* occ: occ_rows * 4 u64 (may be NULL); c_array: 6 u64 = first row of the suffixes starting with A, C, G, T, '#', '$' */
int debwt_index_copy(debwt_ctx* ctx, uint64_t* occ, uint64_t* c_array);
/* Backward search (count only) of n_patterns ACGT strings on the device; pattern i = patterns[offsets[i] .. offsets[i+1]).
   Uses occ / C the way findSeg does (src/LFsearch.c:167-235).  A pattern with a symbol other than A, C, G, T (either case)
   counts 0. */
int debwt_index_count(debwt_ctx* ctx, const char* patterns, const uint64_t* offsets, uint64_t n_patterns, uint64_t* counts);
/* Loads a finished result into the context in place of a build: the reference's three outputs (bwt_words: ceil(N/32) u64
   as debwt_result_copy writes them; sharp_rows: n_sharp rows holding '#', any order; dollar_row), in host memory.  The files
   do not determine N, so the caller passes it.  Use it to query a result of the sharded build (debwt_build_multi,
   debwt_shard_*), of host/deBWT or of the reference.  Resets the input like debwt_set_*; afterwards debwt_result_*,
   debwt_index_* and debwt_verify_text* work as after debwt_build, and debwt_build fails until a new input is set.  Checks
   dollar_row < N and that the '#' rows are distinct, below N and not the '$' row; then every other row holds a base, so
   the base counts plus n_sharp + 1 add up to N.  Whether the array is a BWT at all is found by debwt_index_sample_sa.
   Held in the context's arena (N/4 bytes) until the next input or result. */
int debwt_set_result(debwt_ctx* ctx, const uint64_t* bwt_words, uint64_t n_symbols, const uint64_t* sharp_rows, uint64_t n_sharp,
                     uint64_t dollar_row);
/* Sampled suffix array (locate support; the reference has none): ranks the LF walk like the verifier (16 bytes of scratch
   HBM per symbol, freed on return; N < 2^32 - 1) and keeps SA[r] for every row whose text position is a multiple of
   `rate` (a power of two, 1..1024): a u64 per 32 rows (sampled-row mask | sampled rows before) and ceil(N / rate) u32
   values, i.e. N/4 + 4N/rate bytes of HBM.  Builds the occ / C tables first if needed.  Fails, keeping no samples, when the
   result is not a BWT (its LF mapping is not one N-cycle).  Kept until the next build / input / set_result or the next
   call.  *ms_out (optional) = device time. */
int debwt_index_sample_sa(debwt_ctx* ctx, uint32_t rate, float* ms_out);
/* positions[i] = SA[rows[i]], the text position of the suffix in row rows[i] (at most rate - 1 LF steps per row on the
   device).  Every row must be < N; otherwise nothing is written. */
int debwt_index_sa(debwt_ctx* ctx, const uint64_t* rows, uint64_t n_rows, uint64_t* positions);
/* Locate: backward search of every pattern (as debwt_index_count; A, C, G, T in either case, so a pattern with any other
   symbol has no hits and the empty pattern has N: every suffix), then the text positions of all hits in SA order:
   positions[hit_offsets[i] + j] = SA[sp_i + j] for the rows [sp_i, sp_i + count_i) of pattern i.  hit_offsets[n_patterns + 1]
   is always written (hit_offsets[i + 1] - hit_offsets[i] = count_i); positions == NULL is a size query; more hits than
   positions_cap fails and names the number needed.  Needs debwt_index_sample_sa. */
int debwt_index_locate(debwt_ctx* ctx, const char* patterns, const uint64_t* offsets, uint64_t n_patterns, uint64_t* hit_offsets,
                       uint64_t* positions, uint64_t positions_cap);
/* At-scale verifier: inverts the BWT by its LF mapping (the walk of src/LFsearch.c:49-166, as parallel list ranking) and
   compares every symbol with the text T given by the caller (ASCII, '#' between records, '$' last; host or device
   pointer).  *n_bad_out = rows that are not on the one N-cycle or whose symbol differs; 0 <=> the result is the BWT of
   T.  Needs 16 bytes of scratch HBM per symbol; N < 2^32 - 1. */
int debwt_verify_text(debwt_ctx* ctx, const char* text, uint64_t n_symbols, uint64_t* n_bad_out, float* ms_out);
int debwt_verify_text_device(debwt_ctx* ctx, const void* d_text, uint64_t n_symbols, uint64_t* n_bad_out, float* ms_out);
/* The same check for a packed BWT that is not a context's result (e.g. the stitched output of the sharded build):
   d_bwt_words / d_text are device pointers on `device`, sharp_rows (host, any order) and dollar_row as written to the
   reference's .# / .$ files. */
int debwt_verify_bwt_device(int device, const uint64_t* d_bwt_words, uint64_t n_symbols, const uint64_t* sharp_rows, uint64_t n_sharp,
                            uint64_t dollar_row, const void* d_text, uint64_t* n_bad_out, float* ms_out);

/* For texts beyond 2^32 symbols (C5): the occ / C tables of the packed BWT (their totals must add up to N) and a sequential
   LF walk of `steps` rows from the row holding '$' -- the reference's developer check, src/LFsearch.c:49-166 --, which must
   spell the last `steps` symbols of T backwards (d_text_tail: those symbols, ASCII, on the device).  c_array_out: 6 u64. */
int debwt_verify_walk_device(int device, const uint64_t* d_bwt_words, uint64_t n_symbols, const uint64_t* sharp_rows, uint64_t n_sharp,
                             uint64_t dollar_row, const void* d_text_tail, uint64_t steps, uint64_t* n_bad_out, uint64_t* c_array_out);

/* ---- synthetic workloads on the device (bench / test plumbing; bit-identical to debwt_b200/synth.py) ------ */
/* n iid-uniform bases (ASCII) of the splitmix64 stream `seed` (SURVEY.md section 8d) into device memory */
int debwt_synth_random_bases(int device, void* d_out, uint64_t n, uint64_t seed);
/* one repeat family written over d_seq (n bases): `copies` copies of a `length`-base master at pseudo-random offsets,
   each with substitutions at threshold `thr` = int(rate * 2^53) (0 = exact copies); later copies overwrite earlier ones.
   d_owner_zeroed: n u32 of zeroed scratch (left zeroed). */
int debwt_synth_insert_family(int device, void* d_seq, uint64_t n, uint64_t seed, uint64_t copies, uint64_t length, uint64_t thr,
                              void* d_owner_zeroed);
/* d_out = d_in with iid substitutions (never to the same base) at threshold `thr` */
int debwt_synth_mutate(int device, const void* d_in, void* d_out, uint64_t n, uint64_t seed, uint64_t thr);

/* ---- per-kernel entry points (host buffers in, host buffers out) for parity tests -------------- */
/* K1: ASCII text -> 2-bit packed words, ceil((n+32)/32) of them (src/collect#$.c:78-90). */
int debwt_k_pack(int device, const char* text, uint64_t n_symbols, uint64_t* words_out);
/* K2: all in-record 32-mers as left-aligned keys in text order; keys_out holds n - 32 R entries
   (Jellyfish count semantics, src/kmercounting.sh:8; packing of src/mySort.c:61-75). */
int debwt_k_extract(int device, const char* text, uint64_t n_symbols, const uint64_t* seps, uint64_t n_records,
                    uint64_t* keys_out);
/* K3: ascending sort of 64-bit keys in place (src/mySort.c:98-176).  *ms_out (optional) = device time. */
int debwt_k_radix_sort_u64(int device, uint64_t* keys, uint64_t n, int cfg, float* ms_out);
/* K4: count-by-sort of sorted keys -> {kmer, count} (kmerInfo, src/mySort.c:76-77,194); returns D. */
int debwt_k_rle(int device, const uint64_t* sorted, uint64_t n, uint64_t* kmers_out, uint64_t* counts_out,
                uint64_t* n_distinct_out);
/* K5-K7 through the production build: per sorted key the in/out mask of its k-mer group (src/INandOut.c:253-343):
   bits 0-3 in-bases, bit 4 '#'/'$' predecessor, bits 8-11 out-bases, bit 12 precedes a separator. */
int debwt_k_group_masks(int device, const char* text, uint64_t n_symbols, const uint64_t* seps, uint64_t n_records,
                        uint16_t* masks_out /* n - 32 R */);
/* K7 through the production build: the branch k-mers (src/INandOut.c:396-417) in ascending order, each as
   (k-mer << 2) | multi_in << 1 | multi_out with the sorted-key index of its group's first key.  *n_branch_out is set
   even when it exceeds `cap` (then the call fails and writes nothing). */
int debwt_k_branch_kmers(int device, const char* text, uint64_t n_symbols, const uint64_t* seps, uint64_t n_records,
                         uint64_t* kmer_out, uint64_t* head_out, uint64_t cap, uint64_t* n_branch_out);

/* K9 through the production build (src/generateSP.c:534-683): the branch ("SP") codes, one byte each -- 0..3 the next
   base, 4 = '#', 5 = '$' -- and the blue entries as K10 receives them: for entry e the sorted-key index of its k-mer's
   group, its spIndex and its previous symbol (0..3, 4 = '#', 5 = '$'), grouped by k-mer, any order inside a group. */
int debwt_k_codes(int device, const char* text, uint64_t n_symbols, const uint64_t* seps, uint64_t n_records, uint8_t* codes_out,
                  uint64_t codes_cap, uint64_t* n_codes_out, uint64_t* blue_head_out, uint64_t* blue_spindex_out,
                  uint8_t* blue_prev_out, uint64_t blue_cap, uint64_t* n_blue_out);
/* K10 alone (src/sortBlue.c:76-280): codes as above ('$' exactly once, as the last code); segment i = entries
   seg_offsets[i] .. seg_offsets[i+1]); every segment is ordered by the code string starting at its entries' spIndex,
   in place.  Runs whose previous symbols are all equal may keep any order (src/sortBlue.c:192-219). */
int debwt_k_sort_blue(int device, const uint8_t* codes, uint64_t n_codes, const uint64_t* seg_offsets, uint64_t n_segments,
                      uint64_t* spindex_inout, uint8_t* prev_inout);

/* Device-resident sort benchmark helper: sorts `n` pseudo-random keys `iters` times on the device
   (keys regenerated on device before each run) and returns the mean device ms per sort. */
int debwt_bench_sort(int device, uint64_t n, int cfg, int iters, float* ms_out);
/* Same, and also the mean device ms of ONE digit pass (the named roofline kernel: 16 B/key algorithmic per launch),
   from CUDA events around the scatter passes. */
int debwt_bench_sort_passes(int device, uint64_t n, int cfg, int iters, float* ms_out, float* ms_per_pass_out);

#ifdef __cplusplus
}
#endif
#endif /* DEBWT_B200_H */
