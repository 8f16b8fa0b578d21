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
/* Extract: T[starts[i] .. ends[i]) for every i -- the text the result is the BWT of -- as ASCII (A, C, G, T upper case,
   '#', '$'), concatenated in order into `out` (sum of ends[i] - starts[i] bytes, no terminator).  Needs
   debwt_index_sample_sa; the first call after it derives the inverse samples from the SA samples (4 ceil(N / rate) more
   bytes of HBM, kept with the samples).  Each rate-aligned block is decoded by at most `rate` LF steps, one thread per
   block, so [0, N) inverts the whole BWT.  Fails, writing nothing, when some 0 <= starts[i] <= ends[i] <= N does not hold
   (the message names i) or the total exceeds out_cap (the message names the total).  n_intervals = 0 does nothing. */
int debwt_index_extract(debwt_ctx* ctx, const uint64_t* starts, const uint64_t* ends, uint64_t n_intervals,
                        char* out, uint64_t out_cap);
/* Super-maximal exact matches (SMEMs, the seeds of BWA-MEM) of reads against a text that holds both strands, by the
   bidirectional FMD-index search of Li (2012) over the occ / C tables.  The text must be closed under reverse complement:
   every record's reverse complement is a record too (python: api.both_strands).  That is the caller's duty; the call only
   checks the necessary count(A) = count(T) and count(C) = count(G) from the C-array.
   Read i = reads[offsets[i] .. offsets[i+1]).  A match is a piece read[s, e) of A, C, G, T (either case) that occurs in
   T; with start(e) the smallest s for which read[s, e) matches (e if none does), the SMEMs are the [start(e), e) with
   start(e) < e and (e = len or start(e+1) > start(e)) -- the matches not contained in another maximal match.  Those with
   qend - qbeg >= min_len (>= 1) are written, read by read, in ascending qbeg (and qend): smems[smem_offsets[i] + j].
   Rows [row, row + count) hold the suffixes that start with read[qbeg, qend) (locate them with debwt_index_sa), rc_row
   the first row of its reverse complement; count covers both strands.  smem_offsets[n_reads + 1] is always written;
   smems == NULL is a size query; more SMEMs than smems_cap fails and names the number needed.  Needs debwt_index_build,
   not the SA samples.  Fails, writing nothing, on an unbalanced text (the message names the four base counts), min_len = 0,
   decreasing offsets, NULL arguments, or a read too long for the 1 GiB of scratch (64 (len + 1) bytes per read in flight;
   reads up to 16 Mbp; the message names the read).  n_reads = 0 only writes smem_offsets[0] = 0. */
typedef struct debwt_smem {
    uint64_t row, rc_row, count;   /* rows [row, row + count) start with read[qbeg, qend); rc_row: its reverse complement */
    uint32_t qbeg, qend;
} debwt_smem;
int debwt_index_smem(debwt_ctx* ctx, const char* reads, const uint64_t* offsets, uint64_t n_reads, uint32_t min_len,
                     uint64_t* smem_offsets /* n_reads + 1 */, debwt_smem* smems, uint64_t smems_cap);
/* BWA-MEM's whole seeding step (bwa's mem_collect_intv and the SA sampling of mem_chain) over a text that holds both
   strands, as for debwt_index_smem, from reads to located seed hits.  Options are bwa's -k, -r, split_width, -y and -c
   (defaults 19, 1.5, 10, 20, 500).  smem1(x, t) is bwa's bwt_smem1a(x, min_intv = t, max_intv = 0); a base that does not
   occur in T is stepped over (x + 1) in every round.  Per read of length m:
     round 1: Li's loop x = smem1(x, 1) (the SMEMs of debwt_index_smem); seeds of at least min_seed_len bases;
     round 2: with split_len = (int)(min_seed_len * split_factor + .499) (float product), for every round-1 seed [b, e)
              with e - b >= split_len and count <= split_width, smem1((b + e) >> 1, count + 1); seeds of at least
              min_seed_len bases (duplicates stay, as in bwa);
     round 3 (only when max_mem_intv > 0): from x, extend forward to the first i with i - x >= min_seed_len and
              count(read[x, i + 1)) < max_mem_intv: [x, i + 1) is a seed if its count is > 0; go on at i + 1.  A non-ACGT
              at i ends the attempt without a seed (on at i + 1); the end of the read ends the round.
   A read's seeds are seeds[seed_offsets[i] .. seed_offsets[i + 1]), in ascending (qbeg, qend, round).  Seed rows
   [row, row + count) start with read[qbeg, qend) (count covers both strands), rc_row is the first row of its reverse
   complement.  A seed has n_hits = min(count, max_occ) hits, hits[hit_begin .. hit_begin + n_hits): hit j is
   SA[row + j step], step = count > max_occ ? count / max_occ : 1, with the record (0 .. R/2 - 1 of the R records), the
   strand (0 forward, 1 reverse: records R/2 .. R - 1) and the offset of the hit's first base on the forward strand
   (python: api.strand_offsets).  Seeds hold A, C, G, T only, so no hit spans a separator.
   seed_offsets[n_reads + 1] and *n_hits_out (all hits) are always written; seeds == NULL is a size query.  More seeds
   than seeds_cap or more hits than hits_cap fails, writes nothing into seeds / hits, and names both totals.  Needs
   debwt_index_sample_sa (the first call after sampling also sorts the separator positions on the device and keeps them
   with the samples).  Fails, writing nothing, on: no samples, an unbalanced text (as debwt_index_smem) or an odd number
   of records, min_seed_len = 0, max_occ = 0, a negative or non-finite split_factor, decreasing offsets, NULL arguments
   (hits may be NULL only with seeds), or a read too long for the 1 GiB of scratch (72 len + 64 bytes per read in flight;
   reads up to 14.9 Mbp; the message names the read and the limit).  n_reads = 0 only writes seed_offsets[0] = 0 and
   *n_hits_out = 0. */
typedef struct debwt_seed_opts {
    uint32_t min_seed_len, split_width, max_mem_intv, max_occ;
    float split_factor;
} debwt_seed_opts;
typedef struct debwt_seed {
    uint64_t row, rc_row, count;   /* as debwt_smem */
    uint32_t qbeg, qend;
    uint64_t hit_begin;            /* its hits are hits[hit_begin, hit_begin + n_hits) */
    uint32_t n_hits, round;        /* min(count, max_occ); 1, 2 or 3 */
} debwt_seed;                      /* 48 bytes */
typedef struct debwt_seed_hit {
    uint64_t pos, offset;          /* text position; offset of the hit's first base on the forward strand of its record */
    uint32_t record, strand;       /* record 0 .. R/2 - 1; strand 0 forward, 1 reverse */
} debwt_seed_hit;                  /* 24 bytes */
int debwt_index_seeds(debwt_ctx* ctx, const char* reads, const uint64_t* offsets, uint64_t n_reads, const debwt_seed_opts* opts,
                      uint64_t* seed_offsets /* n_reads + 1 */, uint64_t* n_hits_out, debwt_seed* seeds, uint64_t seeds_cap,
                      debwt_seed_hit* hits, uint64_t hits_cap);
/* BWA-MEM's seed chaining (bwa 0.7.17's mem_chain and mem_chain_flt) from reads to filtered chains, with the seeding of
   debwt_index_seeds inside (seed_opts as there).  Options are bwa's w, max_chain_gap, -W, max_chain_extend, mask_level
   and -D (defaults 100, 10000, 0, 1 << 30, 0.50, 0.50).
   bwa's coordinate: with l_pac = (N - R) / 2 (the forward bases) and F[r] = the bases of the forward records before r, a
   hit of length len at (record r, strand, forward offset o) has rbeg = F[r] + o on strand 0 (its text position - r) and
   rbeg = 2 l_pac - (F[r] + o + len) on strand 1 (python: api.bwa_rbeg).
   Per read, its hits are visited in the order of debwt_index_seeds (seed by seed, hit j ascending); each is a seed
   s = (rbeg, qbeg, len = qend - qbeg) with rid = its record.
     frac_rep: the union length of [qbeg, qend) over the read's seeds with count > max_occ, swept in seed order as bwa
       does, over the read length (float).  A read of length 0 has no chains.
     chain set: chains are ordered by pos.  For each hit, lower = the chain with the greatest pos <= s.rbeg; among chains
       with that pos the one created first (bwa's kbtree orders equal keys by its node layout).  If there is no lower or
       test_and_merge(lower, s) is 0, a new chain {pos = s.rbeg, seeds = [s], rid} is created.
     test_and_merge(c, p), first / last = c's first / last seed: 0 if p.rid != c.rid; 1 without adding p if p.qbeg >=
       first.qbeg, p.qbeg + p.len <= last.qbeg + last.len, p.rbeg >= first.rbeg and p.rbeg + p.len <= last.rbeg +
       last.len (contained); 0 if (last.rbeg < l_pac or first.rbeg < l_pac) and p.rbeg >= l_pac; with x = p.qbeg -
       last.qbeg, y = p.rbeg - last.rbeg (64-bit): p is appended and 1 returned if y >= 0, x - y <= w, y - x <= w,
       x - last.len < max_chain_gap and y - last.len < max_chain_gap; 0 otherwise.
     weight: a sweep over the chain's seeds in order with end = 0: a seed adds len if qbeg >= end, else max(0, qbeg + len
       - end), then end = max(end, qbeg + len); the same over rbeg; the weight is the smaller sweep.
     filter: chains with weight < min_chain_weight are dropped; the rest sorted by weight descending, ties in chain-set
       order (pos, then creation; bwa's sort is unstable).  a[0].kept = 3, kept list [0], first = -1 everywhere.  For
       each i >= 1 and each j of the kept list in order, over query spans (beg = first seed's qbeg, end = last seed's
       qbeg + len): b = max(beg_i, beg_j), e = min(end_i, end_j); if e > b, min_l = min(end_i - beg_i, end_j - beg_j),
       and e - b >= min_l * mask_level (float) and min_l < max_chain_gap: large_ovlp = 1, first_j = i if first_j < 0,
       and if also w_i < w_j * drop_ratio (float) and w_j - w_i >= 2 min_seed_len, i is dropped (the loop stops).  An i
       no j drops joins the kept list with kept = large_ovlp ? 2 : 3.  Then a[first_j].kept = 1 for every j of the kept
       list with first_j >= 0 (over a 2, or reviving a dropped chain).  Counting the kept-1/2 chains in order, at the
       chain where the count reaches max_chain_extend and after it every chain with kept < 3 becomes 0.  Chains with
       kept 0 are removed.
   A read's chains are chains[chain_offsets[i] .. chain_offsets[i + 1]) in that filter order; a chain's seeds are
   chain_seeds[seed_begin .. seed_begin + n_seeds) in insertion order; record and strand are its first seed's (every
   seed of a chain has them).  chain_offsets[n_reads + 1] and *n_chain_seeds_out are always written; chains == NULL is
   a size query.  More chains than chains_cap or more chain seeds than chain_seeds_cap fails, writes nothing into chains
   / chain_seeds, and names both totals.  Needs debwt_index_sample_sa.  Fails, writing nothing, on every input that
   debwt_index_seeds refuses (the messages name index_chains), on a negative w, max_chain_gap, min_chain_weight or
   max_chain_extend, on a negative or non-finite mask_level or drop_ratio (the message names the option), and on NULL
   arguments (chain_seeds may be NULL only with chains).  Besides the seeding scratch the call holds 68 bytes of device
   memory per hit.  n_reads = 0 only writes chain_offsets[0] = 0 and *n_chain_seeds_out = 0.  Not done here: bwa's
   mem_flt_chained_seeds (it needs the extension's scores; debwt_index_regions runs it) and ALT contigs (is_alt is 0). */
typedef struct debwt_chain_opts {
    int32_t w, max_chain_gap, min_chain_weight, max_chain_extend;  /* bwa: 100, 10000, 0 (-W), 1 << 30 */
    float mask_level, drop_ratio;                                   /* bwa: 0.50, 0.50 (-D) */
} debwt_chain_opts;
typedef struct debwt_chain {
    uint64_t pos;           /* rbeg of its first seed (bwa's coordinate) */
    uint64_t seed_begin;    /* its seeds are chain_seeds[seed_begin, seed_begin + n_seeds) */
    uint32_t n_seeds, weight;
    uint32_t record, strand;
    uint32_t kept;          /* 1, 2 or 3 as bwa sets it */
    float frac_rep;         /* the read's, as bwa copies it into every chain */
} debwt_chain;              /* 40 bytes */
typedef struct debwt_chain_seed {
    uint64_t rbeg;          /* bwa's coordinate */
    uint32_t qbeg, len;
} debwt_chain_seed;         /* 16 bytes */
int debwt_index_chains(debwt_ctx* ctx, const char* reads, const uint64_t* offsets, uint64_t n_reads,
                       const debwt_seed_opts* seed_opts, const debwt_chain_opts* chain_opts,
                       uint64_t* chain_offsets /* n_reads + 1 */, uint64_t* n_chain_seeds_out,
                       debwt_chain* chains, uint64_t chains_cap, debwt_chain_seed* chain_seeds, uint64_t chain_seeds_cap);
/* BWA-MEM's seed extension (bwa 0.7.17's mem_flt_chained_seeds and mem_chain2aln) from reads to alignment regions, with
   the seeding and chaining of debwt_index_chains inside (seed_opts and chain_opts as there; chain_opts->w is also the
   extension's band, as bwa's one -w).  ext_opts are bwa's -A, -B, -O, -E (deletion, insertion), -L (5', 3') and -d.
   Scoring: mat[i][j] = i == j ? a : -b for bases i, j < 4; any pair with code 4 scores -1.  Read symbols A, C, G, T in
   either case are 0-3, anything else 4; reference bases are 0-3.  A deletion skips reference bases (o_del, e_del), an
   insertion skips query bases (o_ins, e_ins); a gap of k costs o + k e.  The reference is bwa's pac: the forward records
   concatenated, l_pac = (N - R) / 2 bases; coordinate x >= l_pac is the complement of forward base 2 l_pac - 1 - x.
     cal_max_gap(L): l_del = (int)((double)(L a - o_del) / e_del + 1.), l_ins likewise; min(max(l_del, l_ins, 1), w << 1).
     fetch(beg, mid, end): [beg, end) clipped to the record holding mid, on mid's strand (the reverse copy of a record at
       forward [fb, fe) spans [2 l_pac - fe, 2 l_pac - fb)).
     seed_sw(s): -1 if len >= 200.  qb = max(qbeg - 50, 0), qe = min(qend + 50, l_query), rb = max(rbeg - 50, 0),
       re = min(rbeg + len + 50, 2 l_pac), mid = (2 rbeg + len) >> 1; if rb < l_pac < re: re = l_pac when mid < l_pac,
       else rb = l_pac.  -1 if qe - qb >= 200 or re - rb >= 200.  Else the best local (Gotoh, H >= 0, gaps open from H)
       score of query[qb, qe) against fetch(rb, mid, re).
     mem_flt_chained_seeds: min_l = min_chain_weight ? 1.1f min_chain_weight : 5.5f log(l_query) (double); min_HSP =
       (int)(a min_l + .499).  If min_l > 0.05f l_query nothing is filtered and every seed's score is len.  Otherwise a
       chain keeps, in order, the seeds with sc = seed_sw < 0 (score len a) or sc >= min_HSP (score sc).
     extend(qlen, q, tlen, t, w, end_bonus, h0) is ksw_extend2: row 0 h[0] = h0, h[1] = max(h0 - oe_ins, 0) when
       h0 > oe_ins, then h[j] = h[j-1] - e_ins while h[j-1] > e_ins; w = min(w, max_ins, max_del), max_ins =
       max(1, (int)((double)(qlen a + end_bonus - o_ins) / e_ins + 1.)), max_del likewise; max = h0, max_i = max_j =
       max_ie = gscore = -1, max_off = 0, beg = 0, end = qlen.  Row i over t: beg = max(beg, i - w), end = min(end, i + w
       + 1, qlen); h1 = beg ? 0 : max(0, h0 - o_del - e_del (i + 1)); f = m = 0, mj = -1; for j in [beg, end): M =
       h[j] ? h[j] + mat : 0, h = max(M, e[j], f), h[j] = h1, h1 = h, if m <= h: m = h, mj = j; e[j] = max(e[j] - e_del,
       M - oe_del, 0); f = max(f - e_ins, M - oe_ins, 0).  Then h[end] = h1, e[end] = 0; if max(beg, end) == qlen:
       max_ie = gscore > h1 ? max_ie : i, gscore = max(gscore, h1).  Stop if m == 0.  If m > max: max = m, max_i = i,
       max_j = mj, max_off = max(max_off, |mj - i|); else with zdrop > 0 stop when max - m - (di - dj) e_del > zdrop
       (di = i - max_i > dj = mj - max_j) or max - m - (dj - di) e_ins > zdrop (otherwise).  beg = the first j in
       [beg, end) with (h, e) != 0 (else end); end = min(j + 2, qlen) for the last j in [beg, end] with (h, e) != 0 (else
       beg - 1).  Returns max, qle = max_j + 1, tle = max_i + 1, gtle = max_ie + 1, gscore, max_off.
     mem_chain2aln(c), over each kept chain in filter order after the seed filter: nothing if it has no seeds.  rmax =
       [min(rbeg - qbeg - cal_max_gap(qbeg)), max(rbeg + len + r + cal_max_gap(r))] (r = l_query - qend) clamped to
       [0, 2 l_pac]; if it crosses l_pac, the side of the first seed's rbeg; then fetch(rmax0, first rbeg, rmax1).  The
       seeds are visited by descending (score, index).  Seed s is covered by an earlier region p of the read when s lies
       inside p on both query and reference, s.len - p.seedlen0 <= .1 l_query, and with qd = s.qbeg - p.qb, rd = s.rbeg -
       p.rb, w' = min(cal_max_gap(min(qd, rd)), p.w): |qd - rd| < w', or the same behind the seed (p.qe - s.qend, p.re -
       s.rend).  A covered seed is skipped (and marked) unless an unmarked seed t visited before it has t.len >= .95 s.len
       and overlaps it by >= s.len >> 2 on the query, on another diagonal (either order).  Else a region: left, if qbeg >
       0, extend(reversed query[0, qbeg), reversed ref[rmax0, rbeg), w << k, pen_clip5, h0 = len a) for k = 0, 1, stopping
       when the score equals the one before (-1 at first) or max_off < (bw >> 1) + (bw >> 2); local (qb = qbeg - qle, rb =
       rbeg - tle, truesc = score) if gscore <= 0 or gscore <= score - pen_clip5, else to-end (qb = 0, rb = rbeg - gtle,
       truesc = gscore); with qbeg = 0, score = truesc = len a, qb = 0, rb = rbeg.  Right, if qend < l_query, the same over
       query[qend, l_query) and ref[rbeg + len, rmax1) with h0 = sc0 = score (so the first try stops when it returns sc0)
       and pen_clip3: qe = qend + qle, re = rbeg + len + tle (local) or qe = l_query, re = rbeg + len + gtle (to-end), and
       truesc += chosen - sc0; else qe = l_query, re = rbeg + len.  seedcov = the len of the chain's seeds inside [qb, qe) x
       [rb, re); w = the widest band used; seedlen0 = len; frac_rep, record and strand the chain's.
   A read's regions are regions[region_offsets[i] .. region_offsets[i + 1]) in bwa's order: chain by chain, inside a
   chain in the order of extension.  region_offsets[n_reads + 1] is always written; regions == NULL is a size query.
   More regions than regions_cap fails, names the total and writes nothing into regions.  The regions are computed once
   per call: a call whose cap is large enough seeds, chains and extends once.  Needs debwt_index_sample_sa; the first
   call after it derives the pac from the index (N / 8 bytes, kept and dropped with the samples).  Fails, writing nothing
   into regions, on every input that debwt_index_chains refuses (the messages name index_regions), on a or e_del or e_ins
   below 1, on a negative b, o_del, o_ins, pen_clip5, pen_clip3 or zdrop, on a or b above 127 (bwa's scoring matrix is
   int8_t), on w above 1024 (the band w << 1 of a retry must fit the kernel's DP window of 4099 columns), and on options
   under which a score could leave int32: (2 x longest read + 4 w + 2) max(a, b, e_del, e_ins) + max(o_del, o_ins,
   pen_clip5, pen_clip3, zdrop) must stay below 2^31.  Not done here: mem_sort_dedup_patch, mem_mark_primary_se, mapq,
   CIGAR, SAM, pairing and ALT contigs. */
typedef struct debwt_ext_opts {
    int32_t a, b;                  /* match score, mismatch penalty        bwa: 1, 4   (-A, -B) */
    int32_t o_del, e_del;          /* deletion open / extend               bwa: 6, 1   (-O, -E) */
    int32_t o_ins, e_ins;          /* insertion open / extend              bwa: 6, 1            */
    int32_t pen_clip5, pen_clip3;  /* clipping penalties                   bwa: 5, 5   (-L)     */
    int32_t zdrop;                 /* Z-dropoff, 0 disables                bwa: 100    (-d)     */
} debwt_ext_opts;
typedef struct debwt_region {      /* bwa's mem_alnreg_t, the fields mem_chain2aln sets */
    uint64_t rb, re;               /* reference span [rb, re) in bwa's forward-reverse coordinate */
    uint32_t qb, qe;               /* query span [qb, qe) */
    int32_t  score, truesc;
    uint32_t w, seedcov, seedlen0;
    uint32_t chain;                /* index of its chain among the read's chains (debwt_index_chains order) */
    uint32_t record, strand;       /* the chain's */
    float    frac_rep;
    uint32_t pad_;
} debwt_region;                    /* 64 bytes */
int debwt_index_regions(debwt_ctx* ctx, const char* reads, const uint64_t* offsets, uint64_t n_reads,
                        const debwt_seed_opts* seed_opts, const debwt_chain_opts* chain_opts, const debwt_ext_opts* ext_opts,
                        uint64_t* region_offsets /* n_reads + 1 */, debwt_region* regions, uint64_t regions_cap);
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
