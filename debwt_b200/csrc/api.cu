// C ABI (include/debwt_b200.h) and the single-GPU build pipeline.
//
// Stage order mirrors the reference driver (reference src/main.c:83-149):
//   mySort            -> K1 pack, K2 extract, K3 radix sort
//   collect ‖ getKmer -> sentinel-window ("special") suffixes, K5/K6 edge marks
//   generateBlocks    -> K7 branch table
//   generateSP        -> K9 branch codes + blue entries
//   sortBlue          -> K10 segmented sort
//   insertCase3       -> K8 case-2 fill, K11 case-3 / special emission
#include <algorithm>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/debwt_b200.h"
#include "../../include/debwt_b200_dev.h"
#include "radix_sort.cuh"
#include "stages.cuh"
#include "special.cuh"
#include "ctx.cuh"

namespace debwt {

static thread_local std::string g_err;
unsigned g_launches = 0;
unsigned long long g_launches_total = 0;
void set_error(const std::string& msg) { g_err = msg; }

#define FAIL(msg)            \
    do {                     \
        debwt::set_error(msg); \
        return -1;           \
    } while (0)

template <typename T>
static int dalloc(DevPool& pool, T** p, size_t count) { return pool.alloc(reinterpret_cast<void**>(p), count * sizeof(T)); }

struct Special {
    u64 pos;
    u32 j;        // bases before the separator (0..31)
    u32 rec;
    u64 ins, row;
    u64 w0, w1;   // 32 symbols at the position / right after its separator
    u8 chr, next;
    bool emit;
};



// Host part of the sentinel-window handling: from the per-suffix scan results (rank, windows, insertion
// point) to the tables the kernels consume.  `info[t]`, t = rec*32 + j.  Outputs are in suffix order.
//   ins      : insertion points (ascending) -- overwritten with info[].ins in suffix order
//   rows     : BWT row of each special suffix = ins + its rank
//   chr      : its BWT symbol
//   emit_pos : positions that emit a branch code (divideKmer, src/collect#$.c:537-598): tails always
//              (src/INandOut.c:260-266); windows holding '#' when their 31-symbol prefix occurs with
//              >= 2 different next symbols.  Windows holding '$' are unique.
//   tail_pos : per record, the position of its tail k-mer
int build_special_tables(const SpecialInfo* info, const u64* seps, u64 R, std::vector<u64>& ins, std::vector<u64>& rows,
                         std::vector<u8>& chr, std::vector<u64>& emit_pos, std::vector<u64>& tail_pos) {
    const u64 nspec = 32 * R;
    std::vector<Special> sp(nspec);
    std::vector<char> seen_rank(nspec, 0);
    for (u64 t = 0; t < nspec; ++t) {
        const SpecialInfo& o = info[t];
        if (o.rank >= nspec || seen_rank[o.rank]) FAIL("internal: special suffix ranks are not a permutation");
        seen_rank[o.rank] = 1;
        Special& x = sp[o.rank];
        x.pos = seps[t >> 5] - (t & 31); x.j = (u32)(t & 31); x.rec = (u32)(t >> 5); x.emit = false;
        x.ins = o.ins; x.chr = o.prev; x.w0 = o.w0; x.w1 = o.w1; x.next = o.next;
    }
    ins.resize(nspec); rows.resize(nspec); chr.resize(nspec); tail_pos.assign(R, 0); emit_pos.clear();
    for (u64 t = 0; t < nspec; ++t) {
        ins[t] = sp[t].ins;
        if (t && ins[t] < ins[t - 1]) FAIL("internal: special insertion points are not monotone");
        rows[t] = ins[t] + t;
        chr[t] = sp[t].chr;
    }
    std::map<std::tuple<u32, u64, u64>, std::vector<u64>> groups;
    for (u64 t = 0; t < nspec; ++t) {
        const u32 j = sp[t].j;
        if (j == 31) { sp[t].emit = true; tail_pos[sp[t].rec] = sp[t].pos; continue; }
        if (sp[t].rec + 1 == R) continue;
        const u64 before = j ? (sp[t].w0 & ~(~0ull >> (2 * j))) : 0;
        const u64 after = sp[t].w1 & ~(~0ull >> (2 * (30 - j)));                                  // 30-j bases (>=0)
        groups[std::make_tuple(j, before, j == 30 ? 0 : after)].push_back(t);
    }
    for (auto& g : groups) {
        if (g.second.size() < 2) continue;
        u32 seen = 0;
        for (u64 t : g.second) seen |= 1u << sp[t].next;
        if (seen & (seen - 1))
            for (u64 t : g.second) sp[t].emit = true;
    }
    for (u64 t = 0; t < nspec; ++t) if (sp[t].emit) emit_pos.push_back(sp[t].pos);
    return 0;
}

}  // namespace debwt

using namespace debwt;

namespace {

std::mutex g_pool_mutex;

int bind_device(int device) {
    CUDA_TRY(cudaSetDevice(device));
    return 0;
}

int make_pool_sticky(int device) {
    std::lock_guard<std::mutex> lk(g_pool_mutex);
    cudaMemPool_t mp;
    CUDA_TRY(cudaDeviceGetDefaultMemPool(&mp, device));
    unsigned long long thr = ~0ull;
    CUDA_TRY(cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &thr));
    return 0;
}

__global__ void write_seps_kernel(u8* text, const u64* seps, u64 n_rec) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_rec) text[seps[r]] = (r + 1 == n_rec) ? '$' : '#';
}

__global__ void splitmix_fill_kernel(u64* keys, u64 n, u64 seed) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 z = seed + (i + 1) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    keys[i] = z ^ (z >> 31);
}

template <typename T>
int check_seps(const T* seps, u64 n_rec, u64 n) {
    if (n_rec == 0) FAIL("no records");
    // the sort takes at most 2^32 - 65537 keys (radix_sort_u64) and there are N - 32 R of them: refuse such a text here,
    // before anything is allocated, rather than in K3 with a message about keys
    if (n >= (1ull << 32) - 64 || (n > 32 * n_rec && n - 32 * n_rec >= (1ull << 32) - (1ull << 16)))
        FAIL("text too long for one device: N = " + std::to_string(n) + " symbols in R = " + std::to_string(n_rec) +
             " records; one device takes N < 2^32 - 64 and N - 32 R < 2^32 - 65536 (so N <= 2^32 - 65505 for one record)");
    u64 start = 0;
    for (u64 r = 0; r < n_rec; ++r) {
        if (seps[r] < start || seps[r] - start <= 32) FAIL("Length <= 32!");      // src/collect#$.c:41-45
        start = seps[r] + 1;
    }
    if (start != n) FAIL("last separator must be the last symbol");
    return 0;
}

void reset_input(debwt_ctx* c) {
    drop_index(c);
    c->pool.release_all();
    c->input_mark.clear();
    c->d_ascii = nullptr;
    c->d_ascii_ext = nullptr;
    c->d_packed = nullptr;
    c->d_packed_err = nullptr;
    c->ing.active = false;
    c->d_bwt = nullptr;
    c->d_sharp = nullptr;
    c->d_sharp_count = nullptr;
    c->d_dollar = nullptr;
    c->built = false;
    c->loaded = false;
    c->n = 0;                            // a refused input leaves no input behind: debwt_build then says so
    c->n_rec = 0;
    c->stats = debwt_stats{};
}

}  // namespace

// =============================================================================================
// ABI
// =============================================================================================
extern "C" {

const char* debwt_last_error(void) { return g_err.c_str(); }

uint64_t debwt_launch_count(void) { return g_launches_total; }

int debwt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int debwt_create(debwt_ctx** out, int device) {
    if (!out) FAIL("null out pointer");
    if (debwt_device_count() <= device || device < 0) FAIL("no such CUDA device (this library has no CPU fallback)");
    if (bind_device(device)) return -1;
    if (make_pool_sticky(device)) return -1;
    debwt_ctx* c = new debwt_ctx();
    c->device = device;
    CUDA_TRY(cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking));
    c->pool.st = c->st;
    for (auto& e : c->ev) CUDA_TRY(cudaEventCreate(&e));
    *out = c;
    return 0;
}

void debwt_destroy(debwt_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->st);
    drop_index(c);
    for (int i = 0; i < 2; ++i) {
        if (c->ing.h_stage[i]) cudaFreeHost(c->ing.h_stage[i]);
        if (c->ing.done[i]) cudaEventDestroy(c->ing.done[i]);
    }
    c->pool.destroy();
    for (auto& e : c->ev) if (e) cudaEventDestroy(e);
    cudaStreamDestroy(c->st);
    delete c;
}

int debwt_set_sort_config(debwt_ctx* c, int cfg) {
    int old = c->sort_cfg;
    c->sort_cfg = cfg > 0 ? cfg : kDefaultSortCfg;          // 0 = default
    return old;
}

int debwt_set_blue_grouping(debwt_ctx* c, int mode) {
    int old = c->blue_grouping;
    c->blue_grouping = mode >= 0 && mode <= 2 ? mode : 0;
    return old;
}

int debwt_set_ambiguity_policy(debwt_ctx* c, int resolve, uint64_t seed) {
    if (!c) FAIL("null context");
    c->resolve_ambiguous = resolve != 0;
    c->ambiguity_seed = seed;
    return 0;
}

int debwt_set_records(debwt_ctx* c, const char* const* seqs, const uint64_t* lens, uint64_t n_records) {
    if (!c || !seqs || !lens) FAIL("null argument");
    if (bind_device(c->device)) return -1;
    reset_input(c);
    if (n_records == 0) FAIL("no records");
    u64 n = 0;
    c->seps.resize(n_records);
    for (u64 r = 0; r < n_records; ++r) {
        if (lens[r] <= 32) FAIL("Length <= 32!");
        n += lens[r];
        c->seps[r] = n;
        ++n;
    }
    if (check_seps(c->seps.data(), n_records, n)) return -1;
    c->n = n; c->n_rec = n_records;
    c->pool.hint(n * 19 + (320ull << 20));
    CUDA_TRY(cudaEventRecord(c->ev[0], c->st));
    if (dalloc(c->pool, &c->d_ascii, n + 64)) return -1;
    u64 off = 0;
    for (u64 r = 0; r < n_records; ++r) {
        CUDA_TRY(cudaMemcpyAsync(c->d_ascii + off, seqs[r], lens[r], cudaMemcpyHostToDevice, c->st));
        off += lens[r] + 1;
    }
    u64* d_seps = nullptr;
    if (dalloc(c->pool, &d_seps, n_records)) return -1;
    CUDA_TRY(cudaMemcpyAsync(d_seps, c->seps.data(), n_records * 8, cudaMemcpyHostToDevice, c->st));
    write_seps_kernel<<<(unsigned)((n_records + 255) / 256), 256, 0, c->st>>>(c->d_ascii, d_seps, n_records);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(c->ev[1], c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    CUDA_TRY(cudaEventElapsedTime(&c->stats.ms_h2d, c->ev[0], c->ev[1]));
    c->input_mark = c->pool.mark();
    return 0;
}

int debwt_set_text(debwt_ctx* c, const char* text, uint64_t n, const uint64_t* seps, uint64_t n_records) {
    if (!c || !text || !seps) FAIL("null argument");
    if (bind_device(c->device)) return -1;
    reset_input(c);
    if (check_seps(seps, n_records, n)) return -1;
    c->seps.assign(seps, seps + n_records);
    c->n = n; c->n_rec = n_records;
    c->pool.hint(n * 19 + (320ull << 20));
    CUDA_TRY(cudaEventRecord(c->ev[0], c->st));
    if (dalloc(c->pool, &c->d_ascii, n + 64)) return -1;
    CUDA_TRY(cudaMemcpyAsync(c->d_ascii, text, n, cudaMemcpyHostToDevice, c->st));
    CUDA_TRY(cudaEventRecord(c->ev[1], c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    CUDA_TRY(cudaEventElapsedTime(&c->stats.ms_h2d, c->ev[0], c->ev[1]));
    c->input_mark = c->pool.mark();
    return 0;
}

int debwt_set_text_device(debwt_ctx* c, const void* d_text, uint64_t n, const uint64_t* seps, uint64_t n_records) {
    if (!c || !d_text || !seps) FAIL("null argument");
    if (bind_device(c->device)) return -1;
    reset_input(c);
    if (check_seps(seps, n_records, n)) return -1;
    if (reinterpret_cast<uintptr_t>(d_text) & 15) FAIL("device text must be 16-byte aligned");
    c->seps.assign(seps, seps + n_records);
    c->n = n; c->n_rec = n_records;
    c->pool.hint(n * 18 + (320ull << 20));
    c->d_ascii_ext = reinterpret_cast<const u8*>(d_text);
    c->input_mark = c->pool.mark();
    return 0;
}

int debwt_build(debwt_ctx* c, int k) {
    if (!c) FAIL("null context");
    if (k < 12 || k > 32) FAIL("-k: k-mer length (from 12 to 32, default 32)");      // src/main.c:45-46
    if (c->loaded) FAIL("the context holds a loaded result (debwt_set_result), not an input: set an input before building");
    if (c->ing.active) FAIL("streaming input is still open: call debwt_ingest_end first");
    if (c->n == 0) FAIL("no input set");
    if (bind_device(c->device)) return -1;
    const u8* ascii = c->d_ascii_ext ? c->d_ascii_ext : c->d_ascii;
    if (!ascii && !c->d_packed) FAIL("input was consumed by a previous build; set it again");
    cudaStream_t st = c->st;
    DevPool& pool = c->pool;
    pool.rewind(c->input_mark);          // a repeated build on the same (device-resident) input reuses the arena
    drop_index(c);
    c->built = false;
    const u64 n = c->n, R = c->n_rec, nk = n - 32 * R;
    debwt_stats& S = c->stats;
    const float keep_h2d = S.ms_h2d;
    S = debwt_stats{};
    S.ms_h2d = keep_h2d;
    S.n_symbols = n; S.n_records = R; S.n_keys = nk; S.n_special = 32 * R;
    g_launches = 0;
    int evi = 0;
    auto mark = [&]() { cudaEventRecord(c->ev[evi++], st); };
    mark();                                                                     // ev0

    // ---- K1 pack ----
    u64* d_seps = nullptr; u64* d_text = nullptr; u32* d_err = nullptr;
    if (dalloc(pool, &d_seps, R)) return -1;
    CUDA_TRY(cudaMemcpyAsync(d_seps, c->seps.data(), R * 8, cudaMemcpyHostToDevice, st));
    if (c->d_packed) {                   // streamed in and packed chunk by chunk (debwt_ingest_*): K1 already ran
        d_text = c->d_packed;
        d_err = c->d_packed_err;
    } else {
        if (dalloc(pool, &d_text, text_words(n)) || dalloc(pool, &d_err, 4)) return -1;
        CUDA_TRY(cudaMemsetAsync(d_err, 0, 16, st));
        PackPolicy pol;
        pol.resolve = c->resolve_ambiguous; pol.seed = c->ambiguity_seed;
        if (k_pack_words(ascii, n, d_text, text_words(n), d_err, st, pol)) return -1;
        if (c->d_ascii) { pool.adopt(c->d_ascii, n + 64); c->d_ascii = nullptr; }
    }
    mark();                                                                     // ev1

    // ---- K2 extract ----
    u64 *d_ka = nullptr, *d_kb = nullptr;
    if (dalloc(pool, &d_ka, nk + 2) || dalloc(pool, &d_kb, nk + 2)) return -1;
    if (k_extract(d_text, n, d_seps, R, d_ka, st)) return -1;
    mark();                                                                     // ev2

    // ---- K3 sort ----
    void* d_sortws = nullptr;
    if (pool.alloc(&d_sortws, sort_workspace_bytes(nk, c->sort_cfg))) return -1;
    SortWorkspace ws;
    sort_workspace_bind(ws, d_sortws, nk, c->sort_cfg);
    int sweeps = 0;
    ws.ev_sweep_begin = c->ev[11]; ws.ev_sweep_end = c->ev[12]; ws.sweeps_out = &sweeps;
    const unsigned launches_before_sort = g_launches;
    u64* d_keys = nullptr;
    KeyIndex ki;                        // direct index over the sorted keys: marked by the last sort pass
    ki.bits = key_index_bits(nk);
    if (dalloc(pool, &ki.idx, (1ull << ki.bits) + 2) || k_key_index_init(ki, st)) return -1;
    bool index_marked = false;
    ws.key_index = ki.idx; ws.key_index_bits = ki.bits; ws.key_index_done = &index_marked;
    const bool text_hist = text_digit_hist_applies(n, R);
    if (text_hist && (radix_sort_clear(ws, st) || k_text_digit_hist(d_text, n, d_seps, R, ws.hist, st))) return -1;
    if (radix_sort_u64(d_ka, d_kb, nk, ws, st, &d_keys, text_hist)) return -1;
    S.sort_launches = g_launches - launches_before_sort;
    S.sort_sweeps = (u32)sweeps;
    pool.adopt(d_keys == d_ka ? d_kb : d_ka, (nk + 2) * 8);       // the ping-pong half the sort did not end in
    pool.adopt(d_sortws, sort_workspace_bytes(nk, c->sort_cfg));
    u32 h_err[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(h_err, d_err, 8, cudaMemcpyDeviceToHost, st));
    mark();                                                                     // ev3

    // ---- K5/K6 edge marks, K7 branch table ----
    u16* d_gmask = nullptr;
    if (dalloc(pool, &d_gmask, nk + 2)) return -1;
    CUDA_TRY(cudaMemsetAsync(d_gmask, 0, (nk + 2) * 2, st));
    if (k_key_index_finish(d_keys, nk, ki, index_marked, st)) return -1;
    if (k_mark_edges(d_keys, nk, ki, d_gmask, st)) return -1;
    if (k_mark_heads_tails(d_text, d_seps, R, d_keys, nk, ki, d_gmask, st)) return -1;
    void* d_brws = nullptr; u64* d_tot = nullptr;
    if (pool.alloc(&d_brws, branch_workspace_bytes(nk)) || dalloc(pool, &d_tot, 4)) return -1;
    if (k_branch_count(d_keys, nk, d_gmask, true, d_brws, d_tot, st)) return -1;
    u64 h_tot[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(h_tot, d_tot, 16, cudaMemcpyDeviceToHost, st));
    if (c->cap.on) {
        c->cap.gmask.resize(nk);
        CUDA_TRY(cudaMemcpyAsync(c->cap.gmask.data(), d_gmask, nk * 2, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    if (h_err[0]) FAIL(c->resolve_ambiguous ? "input contains a symbol that is neither a base nor an IUPAC ambiguity code"
                                            : "input contains a symbol other than A, C, G, T (either case)");
    if (h_err[1] != R) FAIL("input contains '#' or '$' inside a record (they are reserved for the record separators)");
    BranchTable bt;
    bt.n_branch = h_tot[0]; bt.n_blue = h_tot[1];
    S.n_branch = bt.n_branch; S.n_blue = bt.n_blue;
    {
        int bits = 8;
        while (bits < 27 && (1ull << bits) < 2 * bt.n_branch) ++bits;
        bt.bits = bits;
    }
    if (dalloc(pool, &bt.kmer, bt.n_branch + 1) || dalloc(pool, &bt.head, bt.n_branch + 1) ||
        dalloc(pool, &bt.blue, bt.n_branch + 2) || dalloc(pool, &bt.cursor, bt.n_branch + 1) ||
        dalloc(pool, &bt.bidx, BranchTable::index_words(bt.bits)))
        return -1;
    CUDA_TRY(cudaMemsetAsync(bt.cursor, 0, (bt.n_branch + 1) * 4, st));
    if (k_branch_write(d_keys, nk, d_gmask, d_brws, bt, st)) return -1;
    {
        const u32 m32 = (u32)bt.n_blue;
        CUDA_TRY(cudaMemcpyAsync(bt.blue + bt.n_branch, &m32, 4, cudaMemcpyHostToDevice, st));
    }
    if (k_branch_index(bt, st)) return -1;
    // blue entries into their segments: by a cursor per segment (kept in the hash slot of the k-mer), or appended densely
    // and grouped by a radix sort on the branch id (the id sits at the top of the key, so ceil(bits / 8) passes do it)
    int id_bits = 1;
    while (id_bits < 64 && (bt.n_branch >> id_bits)) ++id_bits;
    const bool group_by_sort = id_bits <= 28 && n < (1ull << 32) && bt.n_blue > 1 &&
                               c->blue_grouping == 2;      // measured at 3.1 Gbp: 84 ms against 70 ms for the cursors
    bt.hbits = BranchTable::hash_bits(bt.n_branch);
    bt.hmode = group_by_sort ? 0 : 1;
    if (dalloc(pool, &bt.hslots, 1ull << bt.hbits) || k_branch_hash(bt, st)) return -1;
    mark();                                                                     // ev4

    // ---- sentinel-window suffixes: ranked on the device (all pairs for few records, a bitonic network beyond), tables
    //      built on the host ----
    const u64 nspec = 32 * R;
    std::vector<SpecialInfo> info(nspec);
    std::vector<u64> h_ins(nspec);
    u64* d_ins = nullptr;
    if (dalloc(pool, &d_ins, nspec)) return -1;
    {
        SpecialInfo* d_info = nullptr;
        if (dalloc(pool, &d_info, nspec)) return -1;
        if (k_special_scan(d_text, d_seps, R, d_keys, nk, ki, d_info, st)) return -1;
        CUDA_TRY(cudaMemcpyAsync(info.data(), d_info, nspec * sizeof(SpecialInfo), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    std::vector<u64> h_rows, h_emit_pos, h_tail_pos;
    std::vector<u8> h_chr;
    if (build_special_tables(info.data(), c->seps.data(), R, h_ins, h_rows, h_chr, h_emit_pos, h_tail_pos)) return -1;
    u64 *d_rows = nullptr, *d_emit = nullptr, *d_tail = nullptr, *d_tail_idx = nullptr;
    u8* d_chr = nullptr;
    if (dalloc(pool, &d_rows, nspec) || dalloc(pool, &d_chr, nspec) || dalloc(pool, &d_emit, h_emit_pos.size() + 1) ||
        dalloc(pool, &d_tail, R) || dalloc(pool, &d_tail_idx, R))
        return -1;
    CUDA_TRY(cudaMemcpyAsync(d_rows, h_rows.data(), nspec * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_chr, h_chr.data(), nspec, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_ins, h_ins.data(), nspec * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_emit, h_emit_pos.data(), h_emit_pos.size() * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_tail, h_tail_pos.data(), R * 8, cudaMemcpyHostToDevice, st));
    mark();                                                                     // ev5

    // ---- K9 branch codes + blue entries ----
    const u64 nbw = (n + 31) / 32;
    u32 *d_mo = nullptr, *d_wp = nullptr;
    u64* d_blue = nullptr;
    void* d_scanws = nullptr;
    const int id_shift = 64 - id_bits;
    u64 *d_bka = nullptr, *d_bkb = nullptr, *d_bcount = nullptr;
    void* d_bsortws = nullptr;
    const int bcfg = kDefaultSortCfg;
    if (dalloc(pool, &d_mo, nbw + 2) || dalloc(pool, &d_wp, nbw + 2) || pool.alloc(&d_scanws, scan_workspace_bytes(nbw)))
        return -1;
    if (group_by_sort) {
        if (dalloc(pool, &d_bka, bt.n_blue + 2) || dalloc(pool, &d_bkb, bt.n_blue + 2) || dalloc(pool, &d_bcount, 2) ||
            pool.alloc(&d_bsortws, sort_workspace_bytes(bt.n_blue, bcfg)))
            return -1;
        CUDA_TRY(cudaMemsetAsync(d_bcount, 0, 16, st));
    } else if (dalloc(pool, &d_blue, bt.n_blue + 1)) return -1;
    CUDA_TRY(cudaMemsetAsync(d_mo, 0, (nbw + 2) * 4, st));
    if (group_by_sort) {
        if (k_flag_positions_keys(d_text, n, d_seps, R, bt, id_shift, d_mo, d_bka, d_bcount, st)) return -1;
    } else if (k_flag_positions(d_text, n, d_seps, R, bt, d_mo, d_blue, st)) return -1;
    if (k_patch_bits(d_mo, 0, n, d_emit, h_emit_pos.size(), st)) return -1;
    if (scan_exclusive_u32(d_mo, d_wp, nbw, true, d_scanws, d_tot, st)) return -1;
    u64 n_codes = 0, n_appended = 0;
    CUDA_TRY(cudaMemcpyAsync(&n_codes, d_tot, 8, cudaMemcpyDeviceToHost, st));
    if (group_by_sort) CUDA_TRY(cudaMemcpyAsync(&n_appended, d_bcount, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (group_by_sort && n_appended != bt.n_blue) FAIL("internal: multi-in positions found in the text do not match the k-mer counts");
    S.n_codes = n_codes;
    const u64 ncw = n_codes / 32 + 3;
    u64* d_codes = nullptr; u32* d_sep = nullptr;
    if (dalloc(pool, &d_codes, ncw) || dalloc(pool, &d_sep, ncw + 1)) return -1;
    CUDA_TRY(cudaMemsetAsync(d_codes, 0, ncw * 8, st));
    CUDA_TRY(cudaMemsetAsync(d_sep, 0, (ncw + 1) * 4, st));
    if (k_emit_codes(d_text, 0, nbw, d_mo, d_wp, 0, d_codes, st)) return -1;
    if (k_mark_sep_codes(d_mo, d_wp, 0, n, 0, d_tail, R, d_sep, d_tail_idx, st)) return -1;
    if (group_by_sort) {
        if (k_blue_keys_fix(d_bka, bt.n_blue, d_mo, d_wp, st)) return -1;
        SortWorkspace bws;
        sort_workspace_bind(bws, d_bsortws, bt.n_blue, bcfg);
        bws.first_pass = id_shift / 8;
        if (radix_sort_u64(d_bka, d_bkb, bt.n_blue, bws, st, &d_blue)) return -1;
        if (k_blue_keys_strip(d_blue, bt.n_blue, st)) return -1;
        pool.adopt(d_blue == d_bka ? d_bkb : d_bka, (bt.n_blue + 2) * 8);
        pool.adopt(d_bsortws, sort_workspace_bytes(bt.n_blue, bcfg));
    } else if (bt.n_blue >= nbw / 4) {
        u64* d_mw = nullptr;
        if (dalloc(pool, &d_mw, nbw + 2) || k_blue_fix_interleaved(d_blue, bt.n_blue, d_mo, d_wp, nbw + 1, d_mw, st)) return -1;
    } else if (k_blue_fix(d_blue, bt.n_blue, d_mo, d_wp, 0, 0, st)) return -1;
    u64 dollar_index = 0;
    CUDA_TRY(cudaMemcpyAsync(&dollar_index, d_tail_idx + (R - 1), 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    mark();                                                                     // ev6

    if (c->cap.on) {                     // debwt_k_codes: hand the K9 products to the test before K10 reorders the entries
        auto& q = c->cap;
        q.codes.resize(ncw); q.sep.resize(ncw + 1); q.blue.resize(bt.n_blue); q.seg_off.resize(bt.n_branch + 1);
        q.seg_head.resize(bt.n_branch); q.seg_kmer.resize(bt.n_branch);
        q.dollar_index = dollar_index; q.n_codes = n_codes;
        CUDA_TRY(cudaMemcpyAsync(q.codes.data(), d_codes, ncw * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(q.sep.data(), d_sep, (ncw + 1) * 4, cudaMemcpyDeviceToHost, st));
        if (bt.n_blue) CUDA_TRY(cudaMemcpyAsync(q.blue.data(), d_blue, bt.n_blue * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(q.seg_off.data(), bt.blue, (bt.n_branch + 1) * 4, cudaMemcpyDeviceToHost, st));
        if (bt.n_branch) {
            CUDA_TRY(cudaMemcpyAsync(q.seg_head.data(), bt.head, bt.n_branch * 4, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(q.seg_kmer.data(), bt.kmer, bt.n_branch * 8, cudaMemcpyDeviceToHost, st));
        }
        CUDA_TRY(cudaStreamSynchronize(st));
    }

    // ---- K10 segmented sort ----
    u32* d_work = nullptr;
    if (dalloc(pool, &d_work, 4 * bt.n_branch + 16)) return -1;
    SpView spv{d_codes, d_sep, dollar_index, n_codes};
    if (k_sort_blue(d_blue, bt, spv, d_work, st)) return -1;
    mark();                                                                     // ev7

    // ---- K8 + K11 emission ----
    c->n_words = nbw;
    if (dalloc(pool, &c->d_bwt, nbw + 1) || dalloc(pool, &c->d_sharp, R + 1) || dalloc(pool, &c->d_sharp_count, 4) ||
        dalloc(pool, &c->d_dollar, 2))
        return -1;
    CUDA_TRY(cudaMemsetAsync(c->d_sharp_count, 0, 16, st));
    CUDA_TRY(cudaMemsetAsync(c->d_dollar, 0xff, 16, st));
    if (k_fill_case2(d_gmask, nk, 0, n, d_rows, nspec, 0, nbw, c->d_bwt, st)) return -1;
    if (k_emit_blue(d_blue, bt, 0, d_ins, nspec, c->d_bwt, c->d_sharp, c->d_sharp_count, c->d_dollar, st)) return -1;
    if (k_emit_special(d_rows, d_chr, nspec, c->d_bwt, st)) return -1;
    mark();                                                                     // ev8
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());

    float* ms[] = {&S.ms_pack, &S.ms_extract, &S.ms_sort, &S.ms_classify, &S.ms_special, &S.ms_codes, &S.ms_bluesort, &S.ms_emit};
    for (int i = 0; i < 8; ++i) CUDA_TRY(cudaEventElapsedTime(ms[i], c->ev[i], c->ev[i + 1]));
    CUDA_TRY(cudaEventElapsedTime(&S.ms_total, c->ev[0], c->ev[8]));
    if (S.sort_sweeps) CUDA_TRY(cudaEventElapsedTime(&S.ms_sort_sweeps, c->ev[11], c->ev[12]));
    S.total_launches = g_launches;
    S.arena_bytes = pool.reserved_bytes();
    S.arena_used_bytes = pool.used_bytes();
    c->built = true;
    return 0;
}

int debwt_result_sizes(const debwt_ctx* c, uint64_t* n_symbols, uint64_t* n_words, uint64_t* n_sharp) {
    if (!c || !c->built) FAIL("no result: call debwt_build first");
    if (n_symbols) *n_symbols = c->n;
    if (n_words) *n_words = c->n_words;
    if (n_sharp) *n_sharp = c->n_rec - 1;
    return 0;
}

int debwt_result_copy(debwt_ctx* c, uint64_t* bwt_words, uint64_t* sharp_rows, uint64_t* dollar_row) {
    if (!c || !c->built) FAIL("no result: call debwt_build first");
    if (bind_device(c->device)) return -1;
    CUDA_TRY(cudaEventRecord(c->ev[9], c->st));
    if (bwt_words) CUDA_TRY(cudaMemcpyAsync(bwt_words, c->d_bwt, c->n_words * 8, cudaMemcpyDeviceToHost, c->st));
    u32 cnt = 0;
    CUDA_TRY(cudaMemcpyAsync(&cnt, c->d_sharp_count, 4, cudaMemcpyDeviceToHost, c->st));
    u64 dol = 0;
    CUDA_TRY(cudaMemcpyAsync(&dol, c->d_dollar, 8, cudaMemcpyDeviceToHost, c->st));
    std::vector<u64> sharp(c->n_rec + 1);
    CUDA_TRY(cudaMemcpyAsync(sharp.data(), c->d_sharp, (c->n_rec + 1) * 8, cudaMemcpyDeviceToHost, c->st));
    CUDA_TRY(cudaEventRecord(c->ev[10], c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    CUDA_TRY(cudaEventElapsedTime(&c->stats.ms_d2h, c->ev[9], c->ev[10]));
    if (cnt != c->n_rec - 1) FAIL("internal: wrong number of '#' rows");
    if (dol == ~0ull) FAIL("internal: '$' row missing");
    std::sort(sharp.begin(), sharp.begin() + cnt);                      // ascending (src/insertCase3.c:84-95)
    if (sharp_rows) std::copy(sharp.begin(), sharp.begin() + cnt, sharp_rows);
    if (dollar_row) *dollar_row = dol;
    return 0;
}

int debwt_set_result(debwt_ctx* c, const uint64_t* bwt_words, uint64_t n_symbols, const uint64_t* sharp_rows, uint64_t n_sharp,
                     uint64_t dollar_row) {
    if (!c || !bwt_words || (n_sharp && !sharp_rows)) FAIL("null argument");
    if (bind_device(c->device)) return -1;
    reset_input(c);
    c->n = 0; c->n_rec = 0; c->n_words = 0;
    c->seps.clear();
    if (n_symbols == 0) FAIL("set_result: no symbols");
    if (dollar_row >= n_symbols) FAIL("set_result: the '$' row " + std::to_string(dollar_row) + " is not below n_symbols");
    std::vector<u64> sorted(sharp_rows, sharp_rows + n_sharp);
    std::sort(sorted.begin(), sorted.end());
    for (u64 i = 0; i < n_sharp; ++i) {
        if (sorted[i] >= n_symbols) FAIL("set_result: a '#' row (" + std::to_string(sorted[i]) + ") is not below n_symbols");
        if (i && sorted[i] == sorted[i - 1]) FAIL("set_result: the '#' row " + std::to_string(sorted[i]) + " is listed twice");
        if (sorted[i] == dollar_row) FAIL("set_result: the '$' row is also listed as a '#' row");
    }
    // where a build leaves its result (debwt_build: d_bwt, d_sharp, d_sharp_count, d_dollar)
    const u64 R = n_sharp + 1, nbw = (n_symbols + 31) / 32;
    if (dalloc(c->pool, &c->d_bwt, nbw + 1) || dalloc(c->pool, &c->d_sharp, R + 1) || dalloc(c->pool, &c->d_sharp_count, 4) ||
        dalloc(c->pool, &c->d_dollar, 2))
        return -1;
    const u32 cnt = (u32)n_sharp;
    if (n_sharp != cnt) FAIL("set_result: too many '#' rows");
    CUDA_TRY(cudaMemcpyAsync(c->d_bwt, bwt_words, nbw * 8, cudaMemcpyHostToDevice, c->st));
    CUDA_TRY(cudaMemsetAsync(c->d_bwt + nbw, 0, 8, c->st));
    CUDA_TRY(cudaMemsetAsync(c->d_sharp, 0, (R + 1) * 8, c->st));
    if (n_sharp) CUDA_TRY(cudaMemcpyAsync(c->d_sharp, sorted.data(), n_sharp * 8, cudaMemcpyHostToDevice, c->st));
    CUDA_TRY(cudaMemsetAsync(c->d_sharp_count, 0, 16, c->st));
    CUDA_TRY(cudaMemcpyAsync(c->d_sharp_count, &cnt, 4, cudaMemcpyHostToDevice, c->st));
    CUDA_TRY(cudaMemcpyAsync(c->d_dollar, &dollar_row, 8, cudaMemcpyHostToDevice, c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    c->n = n_symbols; c->n_rec = R; c->n_words = nbw;
    c->stats.n_symbols = n_symbols; c->stats.n_records = R;
    c->built = true;
    c->loaded = true;
    return 0;
}

int debwt_get_stats(const debwt_ctx* c, debwt_stats* out) {
    if (!c || !out) FAIL("null argument");
    *out = c->stats;
    return 0;
}

}  // extern "C"


// ---- streaming ingest: replaces the two kseq passes of collect (src/collect#$.c:37-48, 66-86) -------------------
namespace {
constexpr u64 kStageBytes = 32ull << 20;

// copy + pack what the current stage holds; final: also the T padding and the guard word
int ingest_flush(debwt_ctx* c, bool final) {
    auto& g = c->ing;
    const u64 full = final ? g.fill : (g.fill & ~31ull);
    if (full == 0 && !final) return 0;
    const u64 nwords = final ? text_words(g.n + full) - g.n / 32 : full / 32;
    if (g.n / 32 + nwords > g.cap_words) {                 // the hint was too small: move the packed text to a larger block
        u64 cap = g.cap_words * 2;
        while (cap < g.n / 32 + nwords) cap *= 2;
        u64* bigger = nullptr;
        if (dalloc(c->pool, &bigger, cap)) return -1;
        CUDA_TRY(cudaMemcpyAsync(bigger, c->d_packed, (g.n / 32) * 8, cudaMemcpyDeviceToDevice, c->st));
        c->d_packed = bigger;
        g.cap_words = cap;
    }
    const int i = g.cur;
    if (full) CUDA_TRY(cudaMemcpyAsync(g.d_stage[i], g.h_stage[i], full, cudaMemcpyHostToDevice, c->st));
    PackPolicy pol;
    pol.resolve = c->resolve_ambiguous; pol.seed = c->ambiguity_seed; pol.pos_base = g.n;
    if (k_pack_words(g.d_stage[i], full, c->d_packed + g.n / 32, nwords, c->d_packed_err, c->st, pol)) return -1;
    CUDA_TRY(cudaEventRecord(g.done[i], c->st));
    g.busy[i] = true;
    g.n += full;
    if (!final) {                                          // carry the < 32 leftover symbols into the other stage
        const u64 tail = g.fill - full;
        const int o = i ^ 1;
        if (g.busy[o]) { CUDA_TRY(cudaEventSynchronize(g.done[o])); g.busy[o] = false; }
        if (tail) memcpy(g.h_stage[o], g.h_stage[i] + full, tail);
        g.cur = o;
        g.fill = tail;
    } else {
        g.fill = 0;
    }
    return 0;
}
}  // namespace

extern "C" {

void* debwt_host_alloc(uint64_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void debwt_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int debwt_ingest_begin(debwt_ctx* c, uint64_t n_symbols_hint) {
    if (!c) FAIL("null context");
    if (bind_device(c->device)) return -1;
    reset_input(c);
    auto& g = c->ing;
    for (int i = 0; i < 2; ++i) {
        if (!g.h_stage[i]) CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&g.h_stage[i]), kStageBytes, cudaHostAllocDefault));
        if (!g.done[i]) CUDA_TRY(cudaEventCreateWithFlags(&g.done[i], cudaEventDisableTiming));
        g.busy[i] = false;
    }
    const u64 guess = n_symbols_hint ? n_symbols_hint : (256ull << 20);
    c->pool.hint(guess * 18 + (320ull << 20));
    g.cap_words = text_words(guess) + 2;
    if (dalloc(c->pool, &c->d_packed, g.cap_words) || dalloc(c->pool, &c->d_packed_err, 4) ||
        dalloc(c->pool, &g.d_stage[0], kStageBytes + 64) || dalloc(c->pool, &g.d_stage[1], kStageBytes + 64))
        return -1;
    CUDA_TRY(cudaMemsetAsync(c->d_packed_err, 0, 16, c->st));
    CUDA_TRY(cudaEventRecord(c->ev[0], c->st));
    g.cur = 0; g.fill = 0; g.n = 0;
    g.active = true;
    return 0;
}

int debwt_ingest_reserve(debwt_ctx* c, char** buf, uint64_t* cap) {
    if (!c || !buf || !cap) FAIL("null argument");
    auto& g = c->ing;
    if (!g.active) FAIL("no streaming input open: call debwt_ingest_begin first");
    if (bind_device(c->device)) return -1;
    if (g.fill + 4096 > kStageBytes && ingest_flush(c, false)) return -1;      // nearly full: ship it
    if (g.busy[g.cur]) { CUDA_TRY(cudaEventSynchronize(g.done[g.cur])); g.busy[g.cur] = false; }
    *buf = reinterpret_cast<char*>(g.h_stage[g.cur] + g.fill);
    *cap = kStageBytes - g.fill;
    return 0;
}

int debwt_ingest_commit(debwt_ctx* c, uint64_t n_written) {
    if (!c) FAIL("null context");
    auto& g = c->ing;
    if (!g.active) FAIL("no streaming input open: call debwt_ingest_begin first");
    if (g.fill + n_written > kStageBytes) FAIL("debwt_ingest_commit: more bytes than were reserved");
    if (bind_device(c->device)) return -1;
    g.fill += n_written;
    if (g.fill + 4096 > kStageBytes) return ingest_flush(c, false);
    return 0;
}

int debwt_ingest_append(debwt_ctx* c, const char* chunk, uint64_t n) {
    while (n) {
        char* buf = nullptr;
        uint64_t cap = 0;
        if (debwt_ingest_reserve(c, &buf, &cap)) return -1;
        const u64 m = n < cap ? n : cap;
        memcpy(buf, chunk, m);
        if (debwt_ingest_commit(c, m)) return -1;
        chunk += m;
        n -= m;
    }
    return 0;
}

int debwt_ingest_end(debwt_ctx* c, const uint64_t* seps, uint64_t n_records) {
    if (!c || !seps) FAIL("null argument");
    auto& g = c->ing;
    if (!g.active) FAIL("no streaming input open: call debwt_ingest_begin first");
    if (bind_device(c->device)) return -1;
    if (g.busy[g.cur]) { CUDA_TRY(cudaEventSynchronize(g.done[g.cur])); g.busy[g.cur] = false; }
    if (ingest_flush(c, true)) return -1;
    g.active = false;
    const u64 n = g.n;
    if (check_seps(seps, n_records, n)) { c->d_packed = nullptr; return -1; }
    c->seps.assign(seps, seps + n_records);
    c->n = n; c->n_rec = n_records;
    CUDA_TRY(cudaEventRecord(c->ev[1], c->st));
    CUDA_TRY(cudaStreamSynchronize(c->st));
    CUDA_TRY(cudaEventElapsedTime(&c->stats.ms_h2d, c->ev[0], c->ev[1]));
    c->input_mark = c->pool.mark();
    return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// per-kernel entry points
// ---------------------------------------------------------------------------------------------
namespace {
struct Scratch {
    cudaStream_t st = nullptr;
    std::vector<void*> ptrs;
    ~Scratch() {
        for (void* p : ptrs) cudaFree(p);
        if (st) cudaStreamDestroy(st);
    }
    template <typename T>
    int get(T** p, size_t count) {
        CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(p), (count ? count : 1) * sizeof(T)));
        ptrs.push_back(*p);
        return 0;
    }
};
int open_scratch(Scratch& s, int device) {
    if (debwt_device_count() <= device || device < 0) FAIL("no such CUDA device (this library has no CPU fallback)");
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
    return 0;
}
// one production build of the text with the capture on; `take` reads what it needs from the capture
template <typename F>
int captured_build(int device, const char* text, uint64_t n, const uint64_t* seps, uint64_t R, F take) {
    debwt_ctx* c = nullptr;
    if (debwt_create(&c, device)) return -1;
    c->cap.on = true;
    int rc = debwt_set_text(c, text, n, seps, R);
    if (!rc) rc = debwt_build(c, 32);
    if (!rc) rc = take(c->cap);
    debwt_destroy(c);
    return rc;
}
}  // namespace

extern "C" {

int debwt_k_pack(int device, const char* text, uint64_t n, uint64_t* words_out) {
    Scratch s;
    if (open_scratch(s, device)) return -1;
    u8* d_a; u64* d_w; u32* d_e;
    if (s.get(&d_a, n + 64) || s.get(&d_w, text_words(n)) || s.get(&d_e, 4)) return -1;
    CUDA_TRY(cudaMemcpyAsync(d_a, text, n, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemsetAsync(d_e, 0, 16, s.st));
    if (k_pack_words(d_a, n, d_w, text_words(n), d_e, s.st)) return -1;
    u32 e = 0;
    CUDA_TRY(cudaMemcpyAsync(&e, d_e, 4, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaMemcpyAsync(words_out, d_w, ((n + 32 + 31) / 32) * 8, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaStreamSynchronize(s.st));
    if (e) FAIL("input contains a symbol other than A, C, G, T (either case)");
    return 0;
}

int debwt_k_extract(int device, const char* text, uint64_t n, const uint64_t* seps, uint64_t R, uint64_t* keys_out) {
    if (check_seps(seps, R, n)) return -1;
    Scratch s;
    if (open_scratch(s, device)) return -1;
    const u64 nk = n - 32 * R;
    u8* d_a; u64 *d_w, *d_s, *d_k; u32* d_e;
    if (s.get(&d_a, n + 64) || s.get(&d_w, text_words(n)) || s.get(&d_e, 4) || s.get(&d_s, R) || s.get(&d_k, nk)) return -1;
    CUDA_TRY(cudaMemcpyAsync(d_a, text, n, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemcpyAsync(d_s, seps, R * 8, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemsetAsync(d_e, 0, 16, s.st));
    if (k_pack_words(d_a, n, d_w, text_words(n), d_e, s.st) || k_extract(d_w, n, d_s, R, d_k, s.st)) return -1;
    CUDA_TRY(cudaMemcpyAsync(keys_out, d_k, nk * 8, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaStreamSynchronize(s.st));
    return 0;
}

int debwt_k_radix_sort_u64(int device, uint64_t* keys, uint64_t n, int cfg, float* ms_out) {
    Scratch s;
    if (open_scratch(s, device)) return -1;
    u64 *d_a, *d_b; void* d_ws;
    if (s.get(&d_a, n + 2) || s.get(&d_b, n + 2)) return -1;
    CUDA_TRY(cudaMalloc(&d_ws, sort_workspace_bytes(n, cfg)));
    s.ptrs.push_back(d_ws);
    SortWorkspace ws;
    sort_workspace_bind(ws, d_ws, n, cfg);
    CUDA_TRY(cudaMemcpyAsync(d_a, keys, n * 8, cudaMemcpyHostToDevice, s.st));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, s.st));
    u64* res = nullptr;
    if (radix_sort_u64(d_a, d_b, n, ws, s.st, &res)) return -1;
    CUDA_TRY(cudaEventRecord(e1, s.st));
    CUDA_TRY(cudaMemcpyAsync(keys, res, n * 8, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaStreamSynchronize(s.st));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    if (ms_out) *ms_out = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return 0;
}

int debwt_k_rle(int device, const uint64_t* sorted, uint64_t n, uint64_t* kmers_out, uint64_t* counts_out,
                uint64_t* n_distinct_out) {
    Scratch s;
    if (open_scratch(s, device)) return -1;
    u64 *d_k, *d_km, *d_ct, *d_tot; void* d_ws;
    if (s.get(&d_k, n + 2) || s.get(&d_km, n + 2) || s.get(&d_ct, n + 2) || s.get(&d_tot, 2)) return -1;
    CUDA_TRY(cudaMalloc(&d_ws, rle_workspace_bytes(n)));
    s.ptrs.push_back(d_ws);
    CUDA_TRY(cudaMemcpyAsync(d_k, sorted, n * 8, cudaMemcpyHostToDevice, s.st));
    if (k_rle(d_k, n, d_km, d_ct, d_ws, d_tot, s.st)) return -1;
    u64 d = 0;
    CUDA_TRY(cudaMemcpyAsync(&d, d_tot, 8, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaStreamSynchronize(s.st));
    CUDA_TRY(cudaMemcpyAsync(kmers_out, d_km, d * 8, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaMemcpyAsync(counts_out, d_ct, d * 8, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaStreamSynchronize(s.st));
    if (n_distinct_out) *n_distinct_out = d;
    return 0;
}

// K5-K7 through the production build: the masks as K7's count pass leaves them (key index marked by the sort, text-derived
// digit histogram when it applies, masks propagated inside the branch-count kernel)
int debwt_k_group_masks(int device, const char* text, uint64_t n, const uint64_t* seps, uint64_t R, uint16_t* masks_out) {
    return captured_build(device, text, n, seps, R, [&](const debwt_ctx::Capture& q) {
        std::copy(q.gmask.begin(), q.gmask.end(), masks_out);
        return 0;
    });
}

// K7 through the production build: the branch table (k-mer << 2 | multi_in << 1 | multi_out, group head key index)
int debwt_k_branch_kmers(int device, const char* text, uint64_t n, const uint64_t* seps, uint64_t R, uint64_t* kmer_out,
                         uint64_t* head_out, uint64_t cap, uint64_t* n_branch_out) {
    return captured_build(device, text, n, seps, R, [&](const debwt_ctx::Capture& q) {
        if (n_branch_out) *n_branch_out = q.seg_kmer.size();
        if (q.seg_kmer.size() > cap) { set_error("debwt_k_branch_kmers: output buffers too small"); return -1; }
        std::copy(q.seg_kmer.begin(), q.seg_kmer.end(), kmer_out);
        std::copy(q.seg_head.begin(), q.seg_head.end(), head_out);
        return 0;
    });
}


// K9 through the production build: SP codes (0..3, 4 = '#', 5 = '$') and the blue entries before K10
int debwt_k_codes(int device, const char* text, uint64_t n, const uint64_t* seps, uint64_t R, uint8_t* codes_out, uint64_t codes_cap,
                  uint64_t* n_codes_out, uint64_t* blue_head_out, uint64_t* blue_spindex_out, uint8_t* blue_prev_out, uint64_t blue_cap,
                  uint64_t* n_blue_out) {
    return captured_build(device, text, n, seps, R, [&](const debwt_ctx::Capture& q) {
        if (n_codes_out) *n_codes_out = q.n_codes;
        if (n_blue_out) *n_blue_out = q.blue.size();
        if (q.n_codes > codes_cap || q.blue.size() > blue_cap) { set_error("debwt_k_codes: output buffers too small"); return -1; }
        for (u64 i = 0; i < q.n_codes; ++i) {
            u8 code = (u8)((q.codes[i >> 5] >> (2 * (31 - (i & 31)))) & 3ull);
            if ((q.sep[i >> 5] >> (i & 31)) & 1u) code = i == q.dollar_index ? 5 : 4;
            codes_out[i] = code;
        }
        for (u64 b = 0; b < q.seg_kmer.size(); ++b)
            for (u32 e = q.seg_off[b]; e < q.seg_off[b + 1]; ++e) {
                blue_head_out[e] = q.seg_head[b];
                blue_spindex_out[e] = q.blue[e] >> 4;
                blue_prev_out[e] = (u8)(q.blue[e] & 15ull);
            }
        return 0;
    });
}

// K10 alone: codes (one byte per code, 0..3, 4 = '#', 5 = '$' which must be the last code and unique), segments of
// (spIndex, prev) entries; sorts every segment by the code string starting at spIndex (cmpSP, src/sortBlue.c:109-173)
int debwt_k_sort_blue(int device, const uint8_t* codes, uint64_t n_codes, const uint64_t* seg_offsets, uint64_t n_segments,
                      uint64_t* spindex_inout, uint8_t* prev_inout) {
    Scratch s;
    if (open_scratch(s, device)) return -1;
    const u64 M = seg_offsets[n_segments];
    if (M >= 0xFFFFFFFFull) FAIL("too many entries");
    const u64 ncw = n_codes / 32 + 3;
    std::vector<u64> h_codes(ncw, 0);
    std::vector<u32> h_sep(ncw + 1, 0);
    u64 dollar = 0;
    for (u64 i = 0; i < n_codes; ++i) {
        const u8 cd = codes[i];
        if (cd > 5) FAIL("code out of range");
        h_codes[i >> 5] |= (u64)(cd > 3 ? 3 : cd) << (2 * (31 - (i & 31)));      // separators are stored as T (src/generateSP.c:630-642)
        if (cd > 3) { h_sep[i >> 5] |= 1u << (i & 31); if (cd == 5) dollar = i; }
    }
    std::vector<u64> h_blue(M + 1), h_kmer(n_segments + 1);
    std::vector<u32> h_off(n_segments + 2);
    for (u64 e = 0; e < M; ++e) h_blue[e] = (spindex_inout[e] << 4) | prev_inout[e];
    for (u64 b = 0; b < n_segments; ++b) { h_kmer[b] = (b << 2) | 2ull; h_off[b] = (u32)seg_offsets[b]; }
    h_off[n_segments] = (u32)M;
    u64 *d_codes, *d_blue, *d_kmer; u32 *d_sep, *d_off, *d_work;
    if (s.get(&d_codes, ncw) || s.get(&d_sep, ncw + 1) || s.get(&d_blue, M + 1) || s.get(&d_kmer, n_segments + 1) ||
        s.get(&d_off, n_segments + 2) || s.get(&d_work, 4 * n_segments + 16))
        return -1;
    CUDA_TRY(cudaMemcpyAsync(d_codes, h_codes.data(), ncw * 8, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemcpyAsync(d_sep, h_sep.data(), (ncw + 1) * 4, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemcpyAsync(d_blue, h_blue.data(), (M + 1) * 8, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemcpyAsync(d_kmer, h_kmer.data(), (n_segments + 1) * 8, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemcpyAsync(d_off, h_off.data(), (n_segments + 2) * 4, cudaMemcpyHostToDevice, s.st));
    BranchTable bt;
    bt.n_branch = n_segments; bt.n_blue = M; bt.kmer = d_kmer; bt.blue = d_off;
    SpView spv{d_codes, d_sep, dollar, n_codes};
    if (k_sort_blue(d_blue, bt, spv, d_work, s.st)) return -1;
    CUDA_TRY(cudaMemcpyAsync(h_blue.data(), d_blue, M * 8, cudaMemcpyDeviceToHost, s.st));
    CUDA_TRY(cudaStreamSynchronize(s.st));
    for (u64 e = 0; e < M; ++e) { spindex_inout[e] = h_blue[e] >> 4; prev_inout[e] = (u8)(h_blue[e] & 15ull); }
    return 0;
}

int debwt_special_tables(const void* info_host, const uint64_t* ins_by_t, const uint64_t* seps, uint64_t n_rec,
                         uint64_t* ins_out, uint64_t* rows_out, uint8_t* chr_out, uint64_t* emit_pos_out,
                         uint64_t* n_emit_out, uint64_t* tail_pos_out) {
    const u64 nspec = 32 * n_rec;
    std::vector<SpecialInfo> info(reinterpret_cast<const SpecialInfo*>(info_host),
                                  reinterpret_cast<const SpecialInfo*>(info_host) + nspec);
    for (u64 t = 0; t < nspec; ++t) info[t].ins = ins_by_t[t];
    std::vector<u64> seps64(seps, seps + n_rec), ins, rows, emit, tail;
    std::vector<u8> chr;
    if (build_special_tables(info.data(), seps64.data(), n_rec, ins, rows, chr, emit, tail)) return -1;
    std::copy(ins.begin(), ins.end(), ins_out);
    std::copy(rows.begin(), rows.end(), rows_out);
    std::copy(chr.begin(), chr.end(), chr_out);
    std::copy(emit.begin(), emit.end(), emit_pos_out);
    std::copy(tail.begin(), tail.end(), tail_pos_out);
    *n_emit_out = emit.size();
    return 0;
}

int debwt_bench_sort_passes(int device, uint64_t n, int cfg, int iters, float* ms_out, float* ms_per_pass_out) {
    Scratch s;
    if (open_scratch(s, device)) return -1;
    if (cfg == 0) cfg = kDefaultSortCfg;
    u64 *d_a, *d_b; void* d_ws;
    if (s.get(&d_a, n + 2) || s.get(&d_b, n + 2)) return -1;
    CUDA_TRY(cudaMalloc(&d_ws, sort_workspace_bytes(n, cfg)));
    s.ptrs.push_back(d_ws);
    SortWorkspace ws;
    sort_workspace_bind(ws, d_ws, n, cfg);
    cudaEvent_t e0, e1, e2, e3;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventCreate(&e2)); CUDA_TRY(cudaEventCreate(&e3));
    int sweeps = 0;
    ws.ev_sweep_begin = e2; ws.ev_sweep_end = e3; ws.sweeps_out = &sweeps;
    float total = 0, total_pass = 0;
    for (int it = 0; it < iters + 1; ++it) {
        splitmix_fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s.st>>>(d_a, n, 1234 + it);
        CUDA_TRY(cudaEventRecord(e0, s.st));
        u64* res = nullptr;
        if (radix_sort_u64(d_a, d_b, n, ws, s.st, &res)) return -1;
        CUDA_TRY(cudaEventRecord(e1, s.st));
        CUDA_TRY(cudaStreamSynchronize(s.st));
        float ms = 0, msp = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        if (sweeps) CUDA_TRY(cudaEventElapsedTime(&msp, e2, e3));
        if (it) { total += ms; total_pass += sweeps ? msp / sweeps : 0.f; }      // first run is warm-up
    }
    if (ms_out) *ms_out = total / (iters > 0 ? iters : 1);
    if (ms_per_pass_out) *ms_per_pass_out = total_pass / (iters > 0 ? iters : 1);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2); cudaEventDestroy(e3);
    return 0;
}

int debwt_bench_sort(int device, uint64_t n, int cfg, int iters, float* ms_out) {
    return debwt_bench_sort_passes(device, n, cfg, iters, ms_out, nullptr);
}

}  // extern "C"
