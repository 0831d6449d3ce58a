// varscot_b200/csrc/vs_device.cu — device half of the C ABI in include/varscot_scan.h:
// context, packed-text upload, the scan (extract -> score) and the integer-pipe
// microbenchmarks.  Replaces the index-resident search loop of bidir_mapping.cpp:268,285-295.
// There is NO CPU fallback: every entry point fails with VS_ERR_CUDA / VS_ERR_NODEVICE when no
// sm_100 device is usable.
#include "vs_kernels.cuh"
#include "vs_internal.h"
#include <cub/device/device_radix_sort.cuh>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace vs;

static thread_local std::string g_last_error;

constexpr uint64_t DEFAULT_CHUNK_WORDS = 8ull << 20;      // 256 Mi bases per pipeline chunk

// A grow-only buffer of a context: device memory, or pinned host memory when Pinned.  grow() is its only allocation and the
// destructor frees it; a device buffer counts its bytes in its context's device_bytes while it holds them (ctx_device_bytes).
template <typename T, bool Pinned = false>
struct Buf {
    T *p = nullptr;
    uint64_t cap = 0;                    // elements
    uint64_t *held = nullptr;            // device_bytes of the context that allocated it
    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    ~Buf() { release(); }
    operator T *() const { return p; }
    int grow(vs_ctx *ctx, uint64_t n);
    void release()
    {
        if (!p) return;
        if (Pinned) cudaFreeHost(p);
        else { cudaFree(p); *held -= cap * sizeof(T); }
        p = nullptr; cap = 0;
    }
};
template <typename T> using PinnedBuf = Buf<T, true>;

// Buffers that are only used together: after one of them failed to grow, none of them holds memory.
template <typename... B>
static int release_all(B &...b)
{
    (b.release(), ...);
    return VS_ERR_CUDA;
}

struct vs_ctx {
    int device = -1;
    int n_sm = 148;
    uint64_t device_bytes = 0;           // sum of the capacities of the device buffers below (kept by Buf)
    cudaStream_t stream = nullptr;       // extraction + scoring + hit resolution
    cudaStream_t copy = nullptr;         // H2D of the next chunk (copies only, so that the copy engine never waits for a kernel)
    cudaStream_t prep = nullptr;         // small kernels that turn the uploaded mask source of a chunk into its window masks
    cudaEvent_t ev_copied = nullptr, ev_zeroed = nullptr;
    // timed spans of the scan stream: t0[i] begins span i, t1[i] ends it (T_EXTRACT ends at the last chunk's arrival instead)
    enum Span { T_SCAN, T_BUILD, T_EXTRACT, T_SCORE, T_DELIVER, N_SPANS };
    cudaEvent_t t0[N_SPANS] = {}, t1[N_SPANS] = {};
    std::vector<cudaEvent_t> ev_pool;    // per chunk: copied, extract start, extract done, score start, score done
    uint64_t chunk_words = DEFAULT_CHUNK_WORDS;
    // Resident state, three levels that each rest on the one before: the text shard with its contig starts, the plain candidate
    // index of one PAM set over it, the bucketed form of that index.  Only drop_* and commit_* below write level, text and idx.
    enum Level { NOTHING, TEXT, INDEX, BUCKETED } level = NOTHING;
    struct Shard {
        // device word 0 = global word first_word; every position the device stores or emits (candidate store, bucketed store,
        // hits, contig starts) is global - pos_origin (see pos_origin_of)
        uint64_t n_words = 0, first_word = 0, pos_origin = 0;
        bool has_starts = false;         // d_cstart holds the starts of the n_cstart contigs from first_contig on
        uint32_t n_cstart = 0, first_contig = 0;
    } text;
    struct Index {
        int pam = -2;                    // extra_pam of its PAM set
        uint64_t blocks[2] = {0, 0}, cand[2] = {0, 0}, end[2] = {0, 0};     // end: block claims incl. the padding of every chunk
    } idx;
    Buf<vs_bases> d_bases;
    Buf<vs_masks> d_masks;
    Buf<vs_mask_entry> d_sparse;
    // compact mask source path: the N and contig-end planes of the shard (+ halo word) and a staging area for their runs
    Buf<uint32_t> d_nm, d_em;
    Buf<uint8_t> d_emcode, d_dense;      // code bytes of the shard's contig-end plane; coded-block flags of the whole text
    Buf<vs_plane_run> d_runs;
    // contig starts of the shard (device-side hit resolution): derived from d_em, or uploaded
    Buf<uint32_t> d_cstart, d_tilecnt, d_cs_total;
    PinnedBuf<uint32_t> h_cs_total;
    // counters (u64): [0..3] running candidates fwd / rev, block claims fwd / rev; [4 + 4 c ..] block range of chunk c
    // {lo fwd, lo rev, hi fwd, hi rev}; then the whole-store range [4] at all_at(); then the hit counter at all_at() + 4
    Buf<unsigned long long> d_cnt;
    PinnedBuf<unsigned long long> h_cnt;
    uint64_t cnt_chunks = 0;             // the chunks d_cnt / h_cnt have room for: set once both have grown
    uint64_t all_at() const { return 4 + 4 * (cnt_chunks + 1); }
    // candidate store of the whole shard, per strand (the resident index): blocks of BLK_WORDS plane words and 32 positions
    Buf<uint32_t> d_planes[2], d_pos[2];
    uint64_t blocks_cap() const { return d_pos[0].cap / 32; }      // the four grow together (ensure_blocks)
    int keep_index = 1;
    uint64_t hit_cap_opt = 0;
    // bucketed index (vs_bucket.cuh): the candidates regrouped by PAM kind + the VS_KEYLEN - 2 = 6 bases next to the PAM
    int bucket_mode = 1;                 // VS_OPT_BUCKET_INDEX: 0 never, 1 when a resident index is scanned again and it pays (guide count, shard size), 2 always
    Buf<uint32_t> d_bk_planes[2], d_bk_pos[2];
    Buf<unsigned long long> d_bk_ctl;    // hist [2][BK_N], cursor [2][BK_N], start [2][BK_N + 1]
    PinnedBuf<unsigned long long> h_bk_ctl;
    Buf<uint16_t> d_perm, d_gkey;
    PinnedBuf<uint16_t> h_gkey;
    Buf<uint32_t> d_cls;
    // pattern table [2][n_guides][PAT_STRIDE] of uint16
    Buf<uint16_t> d_pat;
    PinnedBuf<uint16_t> h_pat;
    // hits
    Buf<vs_hit> d_hits;
    uint64_t last_n_hits = 0;
    // resolution: sort keys / payloads (double buffers of the radix sort), packed records, sort scratch, pinned staging
    Buf<unsigned long long> d_keys[2], d_vals[2];
    Buf<vs_loc_hit> d_loc;
    PinnedBuf<vs_loc_hit> h_stage;
    Buf<uint8_t> d_sort_tmp;
    Buf<uint64_t> d_win;                 // genome windows of the sorted hits (scans that ask for them) and their staging
    PinnedBuf<uint64_t> h_win;
    std::string err;
};

// The only writers of the resident state.  A commit replaces its level and drops those above it, and needs the one below it;
// a drop keeps the levels below.
static void drop_text(vs_ctx *ctx) { ctx->level = vs_ctx::NOTHING; ctx->text = {}; ctx->idx = {}; }
static void drop_index(vs_ctx *ctx) { ctx->level = std::min(ctx->level, vs_ctx::TEXT); }
static void drop_bucketed(vs_ctx *ctx) { ctx->level = std::min(ctx->level, vs_ctx::INDEX); }
static void commit_text(vs_ctx *ctx, const vs_ctx::Shard &s) { ctx->text = s; ctx->level = vs_ctx::TEXT; }
static void commit_index(vs_ctx *ctx, const vs_ctx::Index &x)
{
    if (ctx->level >= vs_ctx::TEXT) { ctx->idx = x; ctx->level = vs_ctx::INDEX; }
}
static void commit_bucketed(vs_ctx *ctx) { if (ctx->level == vs_ctx::INDEX) ctx->level = vs_ctx::BUCKETED; }

static int fail(vs_ctx *c, int code, const std::string &msg)
{
    g_last_error = msg;
    if (c) c->err = msg;
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(ctx, VS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));     \
    } while (0)

template <typename T, bool Pinned>
int Buf<T, Pinned>::grow(vs_ctx *ctx, uint64_t n)
{
    if (n <= cap) return VS_OK;
    if (p) {
        // any stream of the context may still use the old allocation (the copy and preparation streams fill the text, masks
        // and planes that the scan stream reads): drain all three before it goes
        for (cudaStream_t s : {ctx->stream, ctx->copy, ctx->prep}) CK(cudaStreamSynchronize(s));
        release();
    }
    const size_t bytes = n * sizeof(T);
    const cudaError_t e = Pinned ? cudaMallocHost(&p, bytes) : cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        p = nullptr;
        return fail(ctx, VS_ERR_CUDA, std::string(Pinned ? "cudaMallocHost(" : "cudaMalloc(") + std::to_string(bytes) + " bytes): " + cudaGetErrorString(e));
    }
    cap = n;
    if (!Pinned) { held = &ctx->device_bytes; *held += bytes; }
    return VS_OK;
}

extern "C" const char *vs_last_error(const vs_ctx *ctx)
{
    if (ctx && !ctx->err.empty()) return ctx->err.c_str();
    return g_last_error.c_str();
}

void vs_set_last_error(const char *msg) { g_last_error = msg ? msg : ""; }

void vs_warmup_device(int device)
{
    if (cudaSetDevice(device) == cudaSuccess) cudaFree(nullptr);
    (void)cudaGetLastError();
}

extern "C" int vs_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        g_last_error = std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e);
        (void)cudaGetLastError();
        return -VS_ERR_NODEVICE;
    }
    return n;
}

extern "C" int vs_ctx_create(int device, vs_ctx **out)
{
    vs_ctx *ctx = nullptr;
    if (!out) return fail(nullptr, VS_ERR_ARG, "vs_ctx_create: out is NULL");
    *out = nullptr;
    int n = vs_device_count();
    if (n <= 0) return fail(nullptr, VS_ERR_NODEVICE, "no CUDA device visible (this library has no CPU fallback)");
    if (device < 0 || device >= n) return fail(nullptr, VS_ERR_ARG, "vs_ctx_create: device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, VS_ERR_NODEVICE, std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
                                                  ", this build contains sm_100a code only");
    ctx = new vs_ctx();
    ctx->device = device;
    ctx->n_sm = prop.multiProcessorCount;
    // The copy and mask-preparation streams get the highest priority: the small kernels that build the window masks of
    // the next chunk must not queue behind the scoring grid of the current one.
    int prio_lo = 0, prio_hi = 0;
    cudaError_t e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi < prio_lo ? prio_hi + 1 : prio_hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->copy, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->prep, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_copied, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_zeroed, cudaEventDisableTiming);
    for (int i = 0; i < vs_ctx::N_SPANS && e == cudaSuccess; ++i)
        if ((e = cudaEventCreate(&ctx->t0[i])) == cudaSuccess) e = cudaEventCreate(&ctx->t1[i]);
    if (e != cudaSuccess) fail(ctx, VS_ERR_CUDA, cudaGetErrorString(e));
    if (e != cudaSuccess || ctx->d_cs_total.grow(ctx, 1) != VS_OK || ctx->h_cs_total.grow(ctx, 1) != VS_OK) {
        std::string m = "vs_ctx_create: " + ctx->err;
        vs_ctx_destroy(ctx);
        return fail(nullptr, VS_ERR_CUDA, m);
    }
    *out = ctx;
    return VS_OK;
}

extern "C" void vs_ctx_destroy(vs_ctx *ctx)
{
    if (!ctx) return;
    if (ctx->device >= 0) cudaSetDevice(ctx->device);
    // with the streams idle no work refers to a buffer; the buffers free themselves when ctx is deleted
    for (cudaStream_t s : {ctx->stream, ctx->copy, ctx->prep}) if (s) cudaStreamSynchronize(s);
    for (int i = 0; i < vs_ctx::N_SPANS; ++i)
        for (cudaEvent_t e : {ctx->t0[i], ctx->t1[i]}) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    for (cudaStream_t s : {ctx->stream, ctx->copy, ctx->prep}) if (s) cudaStreamDestroy(s);
    if (ctx->ev_copied) cudaEventDestroy(ctx->ev_copied);
    if (ctx->ev_zeroed) cudaEventDestroy(ctx->ev_zeroed);
    delete ctx;
}

extern "C" int vs_ctx_set_option(vs_ctx *ctx, int option, int64_t value)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_ctx_set_option: ctx is NULL");
    switch (option) {
    case VS_OPT_KEEP_INDEX: ctx->keep_index = value != 0; if (!ctx->keep_index) drop_index(ctx); return VS_OK;
    case VS_OPT_HIT_CAPACITY: if (value < 0) break; ctx->hit_cap_opt = (uint64_t)value; return VS_OK;
    case VS_OPT_BUCKET_INDEX: if (value < 0 || value > 2) break; ctx->bucket_mode = (int)value; if (!value) drop_bucketed(ctx); return VS_OK;
    default: break;
    }
    return fail(ctx, VS_ERR_ARG, "vs_ctx_set_option: unknown option or bad value");
}

extern "C" int vs_index_drop(vs_ctx *ctx)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_index_drop: ctx is NULL");
    drop_index(ctx);
    return VS_OK;
}

// ---- device memory accounting (vs_mapper) -----------------------------------------------------------------------------
constexpr uint64_t BLOCK_BYTES = BLK_WORDS * 4 + 32 * 4;            // one block of 32 candidates: planes + positions

uint64_t vs::ctx_device_bytes(const vs_ctx *ctx) { return ctx ? ctx->device_bytes : 0; }

// Candidate store of a shard, blocks per strand: the expected n_pam / 16 candidates per strand and base, + 15 %, + one partial
// block per extraction tile and per chunk (what scan_engine allocates before the first extraction)
static uint32_t default_tile_words(int n_pam) { return (uint32_t)(60.0 * 16.0 / (2.0 * n_pam)) & ~7u; }

static uint64_t cand_store_blocks(uint64_t n_words, int n_pam, uint32_t tile_words, uint64_t n_chunks)
{
    const uint64_t tiles = (n_words + tile_words - 1) / tile_words;
    const uint64_t est = (uint64_t)((double)n_words * n_pam / 16.0 * 1.15) + tiles + 64ull * n_chunks + 256;
    return (est + BLK_GROUP - 1) / BLK_GROUP * BLK_GROUP;
}

uint64_t vs::resident_shard_bytes(const ShardShape &s, uint64_t text_words, int n_pam)
{
    const uint64_t w = s.words, n_chunks = (w + DEFAULT_CHUNK_WORDS - 1) / DEFAULT_CHUNK_WORDS + 3;
    // text: bases + window masks, both planes + code bytes of the contig-end plane, coded-block flags of the whole text, the
    // staged runs (or sparse mask entries) of the upload, contig starts and their tile counts, counters
    uint64_t b = (w + 1) * (sizeof(vs_bases) + sizeof(vs_masks) + 2 * sizeof(uint32_t) + 1) + (text_words + VS_EM_BLOCK) / VS_EM_BLOCK;
    b += (s.staged + 4 * n_chunks + 16) * sizeof(vs_plane_run);
    b += (s.contigs + 4 + (w + CS_TILE - 1) / CS_TILE + 1 + 1) * sizeof(uint32_t);
    b += (4 + 4 * (n_chunks + 8 + 1) + 4 + 4) * sizeof(unsigned long long);
    // candidate store of both strands, and its bucketed form: every bucket padded to whole batches, + 1/64 + one batch
    const uint64_t plain = cand_store_blocks(w, n_pam, default_tile_words(n_pam), n_chunks);
    const uint64_t bucketed = plain + (uint64_t)BK_N * SC_NB;
    b += 2 * plain * BLOCK_BYTES + 2 * (bucketed + bucketed / 64 + SC_NB) * BLOCK_BYTES;
    b += (2 * BK_N + 2 * BK_N + 2 * (BK_N + 1)) * sizeof(unsigned long long) + 2ull * BK_N * BK_CLS * sizeof(uint32_t);
    // scan scratch: hit buffer, resolution and sort buffers, pattern and class tables
    b += RESIDENT_SCRATCH_HITS * sizeof(vs_hit) + (RESIDENT_SCRATCH_HITS + RESIDENT_SCRATCH_HITS / 8) * (4 * 8 + sizeof(vs_loc_hit)) + (64ull << 20);
    b += 2ull * RESIDENT_SCRATCH_GUIDES * (PAT_STRIDE + 1 + BK_N) * sizeof(uint16_t);
    return b;
}

int vs::resident_plan_check(const std::vector<ShardShape> &shards, uint64_t text_words, const std::vector<uint64_t> &free_bytes,
                            std::vector<uint64_t> &need)
{
    const size_t nd = free_bytes.size(), per = nd ? shards.size() / nd : 0;
    need.assign(nd, 0);
    int first_short = -1;
    for (size_t i = 0; i < nd; ++i) {
        for (size_t s = i * per; s < (i + 1) * per; ++s)
            if (shards[s].words) need[i] += resident_shard_bytes(shards[s], text_words, 3);
        if (need[i] > free_bytes[i] && first_short < 0) first_short = (int)i;
    }
    return first_short;
}

int vs::device_free_bytes(int device, uint64_t *free_bytes)
{
    vs_ctx *ctx = nullptr;
    size_t f = 0, t = 0;
    CK(cudaSetDevice(device));
    CK(cudaMemGetInfo(&f, &t));
    *free_bytes = f;
    return VS_OK;
}

extern "C" int vs_host_register(void *p, size_t bytes)
{
    if (!p || !bytes) return VS_ERR_ARG;
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) {
        g_last_error = std::string("cudaHostRegister: ") + cudaGetErrorString(cudaGetLastError());
        return VS_ERR_CUDA;
    }
    return VS_OK;
}
extern "C" int vs_host_unregister(void *p)
{
    if (!p) return VS_ERR_ARG;
    if (cudaHostUnregister(p) != cudaSuccess) { (void)cudaGetLastError(); return VS_ERR_CUDA; }
    return VS_OK;
}

extern "C" int vs_ctx_set_chunk_words(vs_ctx *ctx, uint64_t chunk_words)
{
    if (!ctx || chunk_words == 0) return fail(ctx, VS_ERR_ARG, "vs_ctx_set_chunk_words: bad arguments");
    ctx->chunk_words = chunk_words;
    return VS_OK;
}

extern "C" void *vs_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void vs_host_free(void *p) { if (p) cudaFreeHost(p); }

static void make_pam(int extra_pam, PamParams &pp)
{
    // forward {GG, GA} + XY; reverse {CC, TC} + revcomp(XY)   (bidir_mapping.cpp:240-247)
    pp.n = 2;
    pp.fx[0] = 2; pp.fy[0] = 2; pp.fx[1] = 2; pp.fy[1] = 0;
    pp.fx[2] = 0; pp.fy[2] = 0;
    if (extra_pam >= 0) { pp.fx[2] = extra_pam / 4; pp.fy[2] = extra_pam % 4; pp.n = 3; }
    for (int j = 0; j < 3; ++j) { pp.rx[j] = 3 - pp.fy[j]; pp.ry[j] = 3 - pp.fx[j]; }
}

// f(std::integral_constant<int, K>()) for the mismatch count k: the scoring kernels are instantiated per K = 0..8
template <typename F>
static void with_k(int k, F &&f)
{
    switch (k) {
    case 0: f(std::integral_constant<int, 0>()); break;
    case 1: f(std::integral_constant<int, 1>()); break;
    case 2: f(std::integral_constant<int, 2>()); break;
    case 3: f(std::integral_constant<int, 3>()); break;
    case 4: f(std::integral_constant<int, 4>()); break;
    case 5: f(std::integral_constant<int, 5>()); break;
    case 6: f(std::integral_constant<int, 6>()); break;
    case 7: f(std::integral_constant<int, 7>()); break;
    default: f(std::integral_constant<int, 8>()); break;
    }
}

// Pipeline chunks of a shard of n_words words: bounds[0] = 0 < ... < bounds[n] = n_words, chunk_words apart.  For a
// streamed scan the last chunk is cut into 1/2, 1/4, 1/8, 1/8: the scan of a chunk can only start when its copy has
// arrived, so what follows the last copy — the tail of the pipeline — shrinks to the scan of an eighth of a chunk.
static std::vector<uint64_t> chunk_plan(uint64_t n_words, uint64_t chunk_words, bool taper)
{
    std::vector<uint64_t> b{0};
    for (uint64_t c0 = 0; c0 < n_words; c0 += chunk_words) b.push_back(std::min(n_words, c0 + chunk_words));
    if (taper && b.size() >= 3) {                  // at least two chunks: split the last one
        const uint64_t c0 = b[b.size() - 2], len = n_words - c0;
        if (len >= 8192) {
            b.pop_back();
            for (uint64_t cut : {len / 2, len / 2 + len / 4, len / 2 + len / 4 + len / 8}) b.push_back(c0 + (cut & ~255ull));
            b.push_back(n_words);
        }
    }
    return b;
}

// ---- text residency ------------------------------------------------------------------------------
static inline bool has_mask_source(const vs_text_view *t) { return t->em_code && t->em_dense; }

// runs of a sorted run list that overlap the word range [lo, hi): index range [first, last)
static void runs_in_range(const vs_plane_run *r, uint64_t n, uint64_t lo, uint64_t hi, uint64_t &first, uint64_t &last)
{
    first = (uint64_t)(std::partition_point(r, r + n, [&](const vs_plane_run &x) { return (uint64_t)x.word + x.count <= lo; }) - r);
    last = (uint64_t)(std::partition_point(r + first, r + n, [&](const vs_plane_run &x) { return (uint64_t)x.word < hi; }) - r);
}

constexpr uint64_t SKIP_MIN_WORDS = 16384;      // all-N runs at least this long are not copied: their bases are zero

// Enqueue the H2D of chunk [c0, c1) (device word indices) on the copy stream.
//  * view with a compact mask source: bases (minus long all-N runs, which are zero-filled on the device), the N plane as
//    runs, the contig-end plane dense or as runs per block, then k_masks_from_planes computes the chunk's masks;
//  * otherwise the masks travel dense, or — when the view carries a sparse list and it is smaller — as memset + sparse
//    entries + a scatter kernel.
// `ready` returns the stream on which the chunk's data is complete (record the chunk's "arrived" event there).
static int enqueue_chunk_copy(vs_ctx *ctx, const vs_text_view *t, uint64_t first_word, uint64_t c0, uint64_t c1,
                              uint64_t &staged, uint64_t &bytes, uint32_t &launches, cudaStream_t &ready)
{
    cudaStream_t cs = ctx->copy;
    ready = cs;
    const uint64_t n = c1 - c0, g0 = first_word + c0;
    // bases [c0, c1] incl. the halo word; word c0 of a later chunk already arrived as the previous chunk's halo
    const uint64_t skip = c0 ? 1 : 0;
    if (has_mask_source(t)) {
        const uint64_t lo = g0, hi = g0 + n + 1;                 // plane words needed: the chunk and its halo word
        uint64_t r0 = 0, r1 = 0;
        runs_in_range(t->nm_runs, t->n_nm_runs, lo, hi, r0, r1);
        // bases, skipping long all-N runs
        uint64_t w = g0 + skip;
        auto copy_bases = [&](uint64_t a, uint64_t b) -> int {   // global words [a, b)
            if (b <= a) return VS_OK;
            CK(cudaMemcpyAsync(ctx->d_bases + (a - first_word), t->bases + a, (b - a) * sizeof(vs_bases), cudaMemcpyHostToDevice, cs));
            bytes += (b - a) * sizeof(vs_bases);
            return VS_OK;
        };
        int r;
        std::vector<std::pair<uint64_t, uint64_t>> skipped;
        for (uint64_t i = r0; i < r1; ++i) {
            const vs_plane_run &x = t->nm_runs[i];
            if (x.value != ~0u || x.count < SKIP_MIN_WORDS) continue;
            const uint64_t a = std::max<uint64_t>(x.word, w), b = std::min<uint64_t>((uint64_t)x.word + x.count, hi);
            if (b <= a) continue;
            if ((r = copy_bases(w, a)) != VS_OK) return r;
            skipped.emplace_back(a, b);                      // zero-filled on the preparation stream below
            w = b;
        }
        if ((r = copy_bases(w, hi)) != VS_OK) return r;
        // N plane and contig-end plane (zeroed by enqueue_upload): the run lists go to the staging area, the code bytes of
        // coded blocks to their own buffer; the expand, fill and mask kernels run on the preparation stream
        vs_plane_run *nm_dst = nullptr, *em_dst = nullptr;
        uint64_t nm_n = 0, em_n = 0;
        auto stage = [&](const vs_plane_run *runs, uint64_t a, uint64_t b, vs_plane_run *&dst, uint64_t &cnt) -> int {
            cnt = b > a ? b - a : 0;
            if (!cnt) return VS_OK;
            if (staged + cnt > ctx->d_runs.cap) return fail(ctx, VS_ERR_CUDA, "run staging area too small");
            dst = ctx->d_runs + staged;
            CK(cudaMemcpyAsync(dst, runs + a, cnt * sizeof(vs_plane_run), cudaMemcpyHostToDevice, cs));
            staged += cnt;
            bytes += cnt * sizeof(vs_plane_run);
            return VS_OK;
        };
        auto longest_run = [&](const vs_plane_run *runs, uint64_t a, uint64_t b) {     // clipped to [lo, hi): sets grid.y of the fill
            uint64_t m = 1;
            for (uint64_t i = a; i < b; ++i)
                m = std::max<uint64_t>(m, std::min<uint64_t>((uint64_t)runs[i].word + runs[i].count, hi) - std::max<uint64_t>(runs[i].word, lo));
            return m;
        };
        const uint64_t nm_long = longest_run(t->nm_runs, r0, r1);
        if ((r = stage(t->nm_runs, r0, r1, nm_dst, nm_n)) != VS_OK) return r;
        uint64_t span0 = 0, span1 = 0;       // pending span [span0, span1) of coded blocks, in global words
        bool any_coded = false;
        auto flush_span = [&]() -> int {
            if (span1 > span0) {
                CK(cudaMemcpyAsync(ctx->d_emcode + (span0 - first_word), t->em_code + span0, span1 - span0, cudaMemcpyHostToDevice, cs));
                bytes += span1 - span0;
                any_coded = true;
            }
            span0 = span1 = 0;
            return VS_OK;
        };
        for (uint64_t b = lo / VS_EM_BLOCK; b * VS_EM_BLOCK < hi; ++b) {
            if (!t->em_dense[b]) { if ((r = flush_span()) != VS_OK) return r; continue; }
            const uint64_t a = std::max<uint64_t>(b * VS_EM_BLOCK, lo), e = std::min<uint64_t>((b + 1) * VS_EM_BLOCK, hi);
            if (span1 == a && span1 > span0) span1 = e; else { if ((r = flush_span()) != VS_OK) return r; span0 = a; span1 = e; }
        }
        if ((r = flush_span()) != VS_OK) return r;
        runs_in_range(t->em_runs, t->n_em_runs, lo, hi, r0, r1);
        const uint64_t em_long = longest_run(t->em_runs, r0, r1);
        if ((r = stage(t->em_runs, r0, r1, em_dst, em_n)) != VS_OK) return r;
        // everything of this chunk is on its way: hand over to the preparation stream
        cudaStream_t ps = ctx->prep;
        CK(cudaEventRecord(ctx->ev_copied, cs));
        CK(cudaStreamWaitEvent(ps, ctx->ev_copied, 0));
        for (const auto &sk : skipped) CK(cudaMemsetAsync(ctx->d_bases + (sk.first - first_word), 0, (sk.second - sk.first) * sizeof(vs_bases), ps));
        if (nm_n) {
            k_fill_runs<<<dim3((unsigned)((nm_n + 7) / 8), (unsigned)((nm_long + FILL_SEG - 1) / FILL_SEG)), 256, 0, ps>>>(nm_dst, nm_n, lo, hi, first_word, ctx->d_nm);
            launches++;
        }
        if (any_coded) {
            k_expand_em_code<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ps>>>(ctx->d_emcode + c0, ctx->d_dense, lo, n + 1, ctx->d_em + c0);
            launches++;
        }
        if (em_n) {
            k_fill_runs<<<dim3((unsigned)((em_n + 7) / 8), (unsigned)((em_long + FILL_SEG - 1) / FILL_SEG)), 256, 0, ps>>>(em_dst, em_n, lo, hi, first_word, ctx->d_em);
            launches++;
        }
        k_masks_from_planes<<<(unsigned)((n + 255) / 256), 256, 0, ps>>>(ctx->d_nm + c0, ctx->d_em + c0, n, ctx->d_masks + c0);
        launches++;
        ready = ps;
        return VS_OK;
    }
    CK(cudaMemcpyAsync(ctx->d_bases + c0 + skip, t->bases + g0 + skip, (n + 1 - skip) * sizeof(vs_bases), cudaMemcpyHostToDevice, cs));
    bytes += (n + 1 - skip) * sizeof(vs_bases);
    bool sparse = false;
    uint64_t e0 = 0, e1 = 0;
    if (t->sparse) {
        const vs_mask_entry *sb = t->sparse, *se = t->sparse + t->n_sparse;
        auto lb = [&](uint64_t w) { return (uint64_t)(std::lower_bound(sb, se, w, [](const vs_mask_entry &x, uint64_t v) { return x.word < v; }) - sb); };
        e0 = lb(g0); e1 = lb(g0 + n);
        sparse = (e1 - e0) * sizeof(vs_mask_entry) < n * sizeof(vs_masks) * 3 / 4 && staged + (e1 - e0) <= ctx->d_sparse.cap;
    }
    if (sparse) {
        CK(cudaMemsetAsync(ctx->d_masks + c0, 0, n * sizeof(vs_masks), cs));
        if (e1 > e0) {
            vs_mask_entry *dst = ctx->d_sparse + staged;
            CK(cudaMemcpyAsync(dst, t->sparse + e0, (e1 - e0) * sizeof(vs_mask_entry), cudaMemcpyHostToDevice, cs));
            k_scatter_masks<<<(unsigned)((e1 - e0 + 255) / 256), 256, 0, cs>>>(dst, e1 - e0, g0, ctx->d_masks + c0);
            launches++;
            staged += e1 - e0;
            bytes += (e1 - e0) * sizeof(vs_mask_entry);
        }
    } else {
        CK(cudaMemcpyAsync(ctx->d_masks + c0, t->masks + g0, n * sizeof(vs_masks), cudaMemcpyHostToDevice, cs));
        bytes += n * sizeof(vs_masks);
    }
    return VS_OK;
}

// device staging for the sparse mask entries, or — for a view with a compact mask source — the plane buffers and the
// staging area of their runs (a run that straddles a chunk border is staged once per chunk it touches)
static int ensure_sparse_staging(vs_ctx *ctx, const vs_text_view *t, uint64_t first_word, uint64_t n_words)
{
    if (has_mask_source(t)) {
        if (ctx->d_nm.grow(ctx, n_words + 1) || ctx->d_em.grow(ctx, n_words + 1) || ctx->d_emcode.grow(ctx, n_words + 1))
            return release_all(ctx->d_nm, ctx->d_em, ctx->d_emcode);
        int r;
        if ((r = ctx->d_dense.grow(ctx, (t->n_words + VS_EM_BLOCK) / VS_EM_BLOCK)) != VS_OK) return r;
        uint64_t a0, a1, b0, b1;
        runs_in_range(t->nm_runs, t->n_nm_runs, first_word, first_word + n_words + 1, a0, a1);
        runs_in_range(t->em_runs, t->n_em_runs, first_word, first_word + n_words + 1, b0, b1);
        const uint64_t n_chunks = (n_words + ctx->chunk_words - 1) / ctx->chunk_words + 3;     // + the tapered tail of chunk_plan()
        return ctx->d_runs.grow(ctx, (a1 - a0) + (b1 - b0) + 4 * n_chunks + 16);
    }
    if (!t->sparse || t->n_sparse == 0) return VS_OK;
    const vs_mask_entry *sb = t->sparse, *se = t->sparse + t->n_sparse;
    auto lb = [&](uint64_t w) { return (uint64_t)(std::lower_bound(sb, se, w, [](const vs_mask_entry &x, uint64_t v) { return x.word < v; }) - sb); };
    return ctx->d_sparse.grow(ctx, lb(first_word + n_words) - lb(first_word));
}

// ---- contig starts of the shard, for the device-side hit resolution --------------------------------------------------
// Contigs c_first .. c_last overlap the shard.  With a mask source the starts come from the shard's contig-end plane on the
// device (nothing travels); the number of end bits tells whether the range holds empty contigs (an empty contig has no
// end bit), in which case — and for views without a source — the host's offsets are uploaded instead.
struct StartsPlan {
    bool usable = false;          // the view has contig offsets and the shard holds bases
    uint32_t c_first = 0, c_last = 0;
    uint32_t expect_bits = 0;     // end bits inside the shard's words if no contig of the range is empty
};

static StartsPlan plan_contig_starts(const vs_text_view *t, uint64_t first_word, uint64_t n_words)
{
    StartsPlan p;
    if (!t->contig_off || t->n_contigs == 0 || n_words == 0) return p;
    const uint64_t b0 = first_word * 32, b1 = std::min<uint64_t>(t->n_bases, (first_word + n_words) * 32);
    if (b0 >= b1) return p;
    const uint64_t *ob = t->contig_off, *oe = t->contig_off + t->n_contigs + 1;
    p.c_first = (uint32_t)(std::upper_bound(ob, oe, b0) - ob - 1);          // last contig starting at or before the first base
    p.c_last = (uint32_t)(std::upper_bound(ob, oe, b1 - 1) - ob - 1);
    const uint64_t shard_end = (first_word + n_words) * 32;                  // end bits are counted over whole words
    p.expect_bits = p.c_last - p.c_first + (ob[p.c_last + 1] - 1 < shard_end ? 1u : 0u);
    p.usable = true;
    return p;
}

// Origin of the 32-bit positions of a shard.  0 — positions are global — for every shard of a text within 4 Gbases (the
// domain of the unordered vs_hit API) and for a shard that ends at least a word below 2^32; otherwise the shard's first
// base, so that a shard of up to VS_MAX_SHARD_WORDS words anywhere in a longer text keeps every window start + 23 below
// the bucket padding sentinel BK_NOPOS = 2^32 - 1.
static uint64_t pos_origin_of(const vs_text_view *t, uint64_t first_word, uint64_t n_words)
{
    if (t->n_words * 32 <= (1ull << 32) || (first_word + n_words + 1) * 32 <= (1ull << 32)) return 0;
    return first_word * 32;
}

static int check_view(vs_ctx *ctx, const vs_text_view *t, uint64_t first_word, uint64_t n_words)
{
    if (!t || !t->bases) return fail(ctx, VS_ERR_ARG, "text view is incomplete");
    if (first_word + n_words > t->n_words) return fail(ctx, VS_ERR_ARG, "shard lies outside the text");
    if (pos_origin_of(t, first_word, n_words) && n_words > VS_MAX_SHARD_WORDS)
        return fail(ctx, VS_ERR_ARG, "shard of " + std::to_string(n_words) + " words in a text beyond 4 Gbases: a shard holds at most VS_MAX_SHARD_WORDS = " +
                                         std::to_string((uint64_t)VS_MAX_SHARD_WORDS) + " words (32-bit positions relative to the shard); split the text as vs_map_records does");
    // a contig longer than the shard overlaps its first or its last base: only those two can exceed 32-bit positions
    const StartsPlan p = plan_contig_starts(t, first_word, n_words);
    for (uint32_t c : {p.c_first, p.c_last})
        if (p.usable && t->contig_off[c + 1] - t->contig_off[c] > (1ull << 32))
            return fail(ctx, VS_ERR_ARG, "contig " + std::to_string(c) + " has more than 2^32 bases (positions inside a contig are 32-bit)");
    if ((t->em_code != nullptr) != (t->em_dense != nullptr) || (has_mask_source(t) && ((t->n_nm_runs && !t->nm_runs) || (t->n_em_runs && !t->em_runs))))
        return fail(ctx, VS_ERR_ARG, "text view carries an incomplete compact mask source");
    // the window masks may be absent when the view carries their source: the device computes them
    if (!has_mask_source(t) && !t->masks && t->n_words) return fail(ctx, VS_ERR_ARG, "text view has neither window masks nor a mask source");
    return VS_OK;
}

// An upload of the shard [first_word, first_word + n_words) of t (vs_text_upload, or a scan that streams the text)
struct Upload {
    const vs_text_view *t = nullptr;
    vs_ctx::Shard shard;          // what becomes resident (finish_upload)
    uint32_t expect_bits = 0;     // StartsPlan::expect_bits
};

// Start of an upload: nothing is resident until it has completed; reserve the shard's text, staging and contig-start buffers.
static int reserve_shard(vs_ctx *ctx, const vs_text_view *t, uint64_t first_word, uint64_t n_words, Upload &u)
{
    drop_text(ctx);
    if (ctx->d_bases.grow(ctx, n_words + 1) || ctx->d_masks.grow(ctx, n_words + 1)) return release_all(ctx->d_bases, ctx->d_masks);
    int r;
    if ((r = ensure_sparse_staging(ctx, t, first_word, n_words)) != VS_OK) return r;
    const StartsPlan sp = plan_contig_starts(t, first_word, n_words);
    u = {t, {n_words, first_word, pos_origin_of(t, first_word, n_words), sp.usable, sp.c_last - sp.c_first + 1, sp.c_first}, sp.expect_bits};
    if (!sp.usable) return VS_OK;
    if ((r = ctx->d_cstart.grow(ctx, (uint64_t)(sp.c_last - sp.c_first) + 4)) != VS_OK) return r;
    return ctx->d_tilecnt.grow(ctx, (n_words + CS_TILE - 1) / CS_TILE + 1);
}

// Enqueue the upload chunk by chunk over `plan` (after `after`, an event of the caller's stream, if given): each chunk's copies
// [+ mask kernels], after the last one the derivation of the contig starts, then on_chunk(c, the stream the chunk is complete
// on).  No host synchronisation: the caller drains the streams, then calls finish_upload.
template <typename OnChunk>
static int enqueue_upload(vs_ctx *ctx, const Upload &u, const std::vector<uint64_t> &plan, cudaEvent_t after, uint64_t &bytes,
                          uint32_t &launches, OnChunk &&on_chunk)
{
    const vs_ctx::Shard &sh = u.shard;
    if (after) CK(cudaStreamWaitEvent(ctx->copy, after, 0));
    if (has_mask_source(u.t)) {
        // zero both planes of the shard on the preparation stream and make the copy stream wait for it; the dense blocks of
        // the coded-block flags of the contig-end plane go to the device once per upload
        if (after) CK(cudaStreamWaitEvent(ctx->prep, after, 0));
        CK(cudaMemsetAsync(ctx->d_nm, 0, (sh.n_words + 1) * sizeof(uint32_t), ctx->prep));
        CK(cudaMemsetAsync(ctx->d_em, 0, (sh.n_words + 1) * sizeof(uint32_t), ctx->prep));
        CK(cudaMemcpyAsync(ctx->d_dense, u.t->em_dense, (u.t->n_words + VS_EM_BLOCK) / VS_EM_BLOCK, cudaMemcpyHostToDevice, ctx->prep));
        CK(cudaEventRecord(ctx->ev_zeroed, ctx->prep));
        CK(cudaStreamWaitEvent(ctx->copy, ctx->ev_zeroed, 0));
    }
    uint64_t staged = 0;
    const uint32_t n_chunks = (uint32_t)(plan.size() - 1);
    for (uint32_t c = 0; c < n_chunks; ++c) {
        cudaStream_t ready;
        int r;
        if ((r = enqueue_chunk_copy(ctx, u.t, sh.first_word, plan[c], plan[c + 1], staged, bytes, launches, ready)) != VS_OK) return r;
        if (c + 1 == n_chunks && sh.has_starts && has_mask_source(u.t)) {
            // the contig starts derived from the contig-end plane (the first may lie before the origin: modulo 2^32, see k_resolve_hits)
            const unsigned tiles = (unsigned)((sh.n_words + CS_TILE - 1) / CS_TILE);
            k_contig_starts_count<<<tiles, 256, 0, ctx->prep>>>(ctx->d_em, sh.n_words, ctx->d_tilecnt);
            k_contig_starts_scan<<<1, 1024, 0, ctx->prep>>>(ctx->d_tilecnt, tiles, ctx->d_cs_total);
            k_contig_starts_scatter<<<tiles, 256, 0, ctx->prep>>>(ctx->d_em, sh.n_words, ctx->d_tilecnt, sh.first_word * 32 - sh.pos_origin,
                                                                  (uint32_t)(u.t->contig_off[sh.first_contig] - sh.pos_origin), ctx->d_cstart);
            launches += 3;
            CK(cudaMemcpyAsync(ctx->h_cs_total, ctx->d_cs_total, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->prep));
        }
        if ((r = on_chunk(c, ready)) != VS_OK) return r;
    }
    return VS_OK;
}

// After the upload's streams have drained: the contig starts (the derived ones, or — empty contigs inside the range, or no
// contig-end plane on the device — the host's offsets, 32-bit relative to the origin), then the shard is resident.
static int finish_upload(vs_ctx *ctx, const Upload &u, uint64_t &h2d_bytes)
{
    const vs_ctx::Shard &s = u.shard;
    if (s.has_starts && (!has_mask_source(u.t) || *ctx->h_cs_total != u.expect_bits)) {
        std::vector<uint32_t> h(s.n_cstart);
        for (uint32_t i = 0; i < s.n_cstart; ++i) h[i] = (uint32_t)(u.t->contig_off[s.first_contig + i] - s.pos_origin);
        CK(cudaMemcpyAsync(ctx->d_cstart, h.data(), (size_t)s.n_cstart * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        h2d_bytes += (uint64_t)s.n_cstart * sizeof(uint32_t);
    }
    commit_text(ctx, s);
    return VS_OK;
}

// leave no copy in flight that still reads the caller's buffers, and no half-resident text behind
static int abandon_upload(vs_ctx *ctx, int rc)
{
    cudaStreamSynchronize(ctx->copy); cudaStreamSynchronize(ctx->prep); cudaStreamSynchronize(ctx->stream);
    (void)cudaGetLastError();
    drop_text(ctx);
    return rc;
}

// Make the shard resident (vs_text_upload; a streamed scan with nothing to score): upload, drain, finish
static int upload_text(vs_ctx *ctx, const vs_text_view *t, uint64_t first_word, uint64_t n_words)
{
    Upload u;
    int r;
    if ((r = reserve_shard(ctx, t, first_word, n_words, u)) != VS_OK) return r;
    uint64_t bytes = 0;
    uint32_t launches = 0;
    if ((r = enqueue_upload(ctx, u, chunk_plan(n_words, ctx->chunk_words, false), nullptr, bytes, launches,
                            [](uint32_t, cudaStream_t) { return (int)VS_OK; })) != VS_OK)
        return abandon_upload(ctx, r);
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(ctx->copy) != cudaSuccess || cudaStreamSynchronize(ctx->prep) != cudaSuccess)
        return abandon_upload(ctx, fail(ctx, VS_ERR_CUDA, "vs_text_upload: the upload failed on the device"));
    if ((r = finish_upload(ctx, u, bytes)) != VS_OK) return abandon_upload(ctx, r);
    return VS_OK;
}

extern "C" int vs_text_upload(vs_ctx *ctx, const vs_text_view *t, uint64_t first_word, uint64_t n_words)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_text_upload: ctx is NULL");
    int r = check_view(ctx, t, first_word, n_words);
    if (r != VS_OK) return r;
    CK(cudaSetDevice(ctx->device));
    if ((r = upload_text(ctx, t, first_word, n_words)) == VS_OK) ctx->err.clear();
    return r;
}

// ---- the scan -----------------------------------------------------------------------------------
// Expected hits per guide and text base on uniform-random text (SURVEY.md 8d): both strands, sum over the PAMs of
// (1/16) P[Bin(21, 3/4) <= k] (no credit for a guide whose own PAM differs from the site's: an upper bound).
static double hit_density(int k, int n_pam)
{
    double p = 0, c = 1;                                    // c = C(21, j)
    for (int j = 0; j <= k && j <= 21; ++j) {
        p += c * std::pow(0.75, j) * std::pow(0.25, 21 - j);
        c = c * (21 - j) / (j + 1);
    }
    return 2.0 * n_pam / 16.0 * p;
}

double vs::expected_hits_per_base(int k, int extra_pam)
{
    PamParams pp;
    make_pam(extra_pam, pp);
    return hit_density(k, pp.n);
}

// ---- bucketed index (vs_bucket.cuh) --------------------------------------------------------------------------------
// Built from the resident plain index and the resident text: bucket histogram -> padded bucket starts -> positions
// regrouped by bucket -> blocks gathered from the text.  Two host synchronisations: the store is sized by the padded total
// read back half-way, and the build is timed.
static_assert(BK_HIST_SMEM <= 48 * 1024, "k_bucket_hist and k_bucket_scatter launch within the default dynamic shared memory limit");
static int build_bucket_index(vs_ctx *ctx, const PamParams &pp, uint32_t &launches, float &build_ms)
{
    cudaStream_t st = ctx->stream;
    if (ctx->d_bk_ctl.grow(ctx, 2 * BK_N + 2 * BK_N + 2 * (BK_N + 1)) || ctx->h_bk_ctl.grow(ctx, 2 * (BK_N + 1)))
        return release_all(ctx->d_bk_ctl, ctx->h_bk_ctl);
    unsigned long long *d_hist = ctx->d_bk_ctl, *d_cursor = d_hist + 2 * BK_N, *d_start = d_cursor + 2 * BK_N;
    const unsigned long long *d_all = ctx->d_cnt + ctx->all_at();
    CK(cudaEventRecord(ctx->t0[vs_ctx::T_BUILD], st));
    CK(cudaMemsetAsync(d_hist, 0, 2 * BK_N * sizeof(unsigned long long), st));
    const uint64_t max_blocks = std::max(ctx->idx.end[0], ctx->idx.end[1]);
    const dim3 grid((unsigned)((max_blocks + BKB_THREADS - 1) / BKB_THREADS), 2);
    if (max_blocks) k_bucket_hist<<<grid, BKB_THREADS, BK_HIST_SMEM, st>>>(ctx->d_planes[0], ctx->d_planes[1], d_all, pp, d_hist);
    k_bucket_scan<<<2, 1024, 0, st>>>(d_hist, d_start, d_cursor);
    launches += 2;
    CK(cudaMemcpyAsync(ctx->h_bk_ctl, d_start, 2 * (BK_N + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    uint64_t nb[2];
    for (int s = 0; s < 2; ++s) {
        nb[s] = ctx->h_bk_ctl[s * (BK_N + 1) + BK_N];
        if (nb[s] > ctx->d_bk_pos[s].cap / 32) {
            const uint64_t cap = nb[s] + nb[s] / 64 + SC_NB;
            if (ctx->d_bk_planes[s].grow(ctx, cap * BLK_WORDS) || ctx->d_bk_pos[s].grow(ctx, cap * 32))
                return release_all(ctx->d_bk_planes[s], ctx->d_bk_pos[s]);
        }
        if (nb[s]) CK(cudaMemsetAsync(ctx->d_bk_pos[s], 0xFF, nb[s] * 32 * sizeof(uint32_t), st));
    }
    if (max_blocks) {
        k_bucket_scatter<<<grid, BKB_THREADS, BK_HIST_SMEM, st>>>(ctx->d_planes[0], ctx->d_planes[1], ctx->d_pos[0], ctx->d_pos[1], d_all, pp, d_cursor,
                                                                  ctx->d_bk_pos[0], ctx->d_bk_pos[1], nb[0] * 32, nb[1] * 32);
        launches++;
    }
    for (int s = 0; s < 2; ++s)
        if (nb[s]) {
            k_bucket_gather<<<(unsigned)((nb[s] + 63) / 64), 64, 0, st>>>(ctx->d_bases, ctx->d_masks, ctx->text.first_word * 32 - ctx->text.pos_origin,
                                                                          ctx->d_bk_pos[s], nb[s], ctx->d_bk_planes[s]);
            launches++;
        }
    CK(cudaEventRecord(ctx->t1[vs_ctx::T_BUILD], st));
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    CK(cudaEventElapsedTime(&build_ms, ctx->t0[vs_ctx::T_BUILD], ctx->t1[vs_ctx::T_BUILD]));
    commit_bucketed(ctx);
    return VS_OK;
}

const char *vs::scan_arg_error(const uint8_t *guides, uint32_t n_guides, int k, int extra_pam)
{
    if (k < 0 || k > VS_MAX_MISMATCHES) return "mismatches must lie between 0 and 8";
    if (extra_pam < -1 || extra_pam > 15) return "extra_pam must be -1 or 4*x+y";
    if (n_guides && !guides) return "guides is NULL";
    if (n_guides >= (1u << 24)) return "at most 2^24-1 guides per call";
    for (uint64_t i = 0; i < (uint64_t)n_guides * VS_GLEN; ++i)
        if (guides[i] > 3) return "guide codes must be 0..3";
    return nullptr;
}

// A scan: the request (vs_scan, vs_scan_text, vs_scan_resolved), what scan_engine plans for it, and what it counts
struct Scan {
    const vs_text_view *src = nullptr;       // stream the text from the host (vs_scan_text) or scan the resident shard
    uint64_t first_word = 0, n_words = 0, origin = 0;
    const uint8_t *guides = nullptr;
    uint32_t n_guides = 0;
    int k = 0, extra_pam = -1;
    bool resolved = false;                   // raw unordered vs_hit, or resolved + sorted vs_loc_hit
    vs_hit *out_raw = nullptr;
    vs_loc_hit *out_loc = nullptr;
    uint64_t out_cap = 0;
    uint64_t *n_hits = nullptr;
    bool windows = false;                    // resolved: the genome window of every hit too (k_loc_windows)
    loc_sink sink = nullptr;
    void *user = nullptr;
    vs_scan_stats *stats = nullptr;
    Upload up;                               // the text from the host: not resident while up.t is set
    PamParams pp;
    std::vector<uint64_t> plan;              // pipeline chunks of the shard
    uint32_t n_chunks = 0, tile_words = 0;
    bool use_bk = false;                     // score the bucketed index
    unsigned score_ctas = 0;
    vs_scan_stats S{};
    uint64_t total_out = 0;                  // hits delivered so far (all super-chunks)
};

constexpr int EVC = 5;      // events per chunk in ev_pool: arrived, extract start, extract done, score start, score done

// candidate store of the shard, room for `need` blocks per strand (a regrown store holds no index)
static int ensure_blocks(vs_ctx *ctx, uint64_t need)
{
    if (need <= ctx->blocks_cap()) return VS_OK;
    drop_index(ctx);
    for (int s = 0; s < 2; ++s)
        if (ctx->d_planes[s].grow(ctx, need * BLK_WORDS) || ctx->d_pos[s].grow(ctx, need * 32))
            return release_all(ctx->d_planes[0], ctx->d_pos[0], ctx->d_planes[1], ctx->d_pos[1]);
    return VS_OK;
}

// The guides' host tables: the pattern table [strand][guide][PAT_STRIDE] (uint16 plane offsets, see pat_slot; grown by
// scan_engine) and, for the bucketed index, the keys of the patterns (per guide pass the guides of every bucket are sorted by
// their key mismatches)
static int stage_guides(vs_ctx *ctx, const Scan &s)
{
    if (s.use_bk && (ctx->d_gkey.grow(ctx, 2ull * s.n_guides) || ctx->h_gkey.grow(ctx, 2ull * s.n_guides))) return release_all(ctx->d_gkey, ctx->h_gkey);
    for (int st = 0; st < 2; ++st)
        for (uint32_t g = 0; g < s.n_guides; ++g) {
            uint16_t *dst = ctx->h_pat + ((size_t)st * s.n_guides + g) * PAT_STRIDE;
            const uint8_t *gd = s.guides + (size_t)g * VS_GLEN;
            for (int j = 0; j < VS_GLEN; ++j) {
                const int i = slot_position(st, j);
                const int b = st ? 3 - gd[VS_GLEN - 1 - i] : gd[i];      // reverse pass scores revcomp(guide), bidir_mapping.cpp:293
                dst[j] = pat_slot(st, j, b);
            }
            dst[VS_GLEN] = 0;
            if (!s.use_bk) continue;
            uint8_t patc[VS_GLEN];
            for (int i = 0; i < VS_GLEN; ++i) patc[i] = st ? (uint8_t)(3 - gd[VS_GLEN - 1 - i]) : gd[i];
            ctx->h_gkey[(size_t)st * s.n_guides + g] = (uint16_t)key_of_codes(st, patc);
        }
    return s.use_bk ? ctx->d_cls.grow(ctx, 2ull * BK_N * BK_CLS) : VS_OK;
}

// CTA size of k_score: one warp per 32 guides, at most SC_WARPS; a short tail (<= 8 guides) does not get a warp of its own
// — it would idle most of the time and hold a warp slot (100 guides: 3 warps; the tail's 4-guide segments rotate over them)
static unsigned score_cta(uint32_t ng)
{
    static const int fold_tail = getenv("VARSCOT_SCORE_FOLD_TAIL") ? atoi(getenv("VARSCOT_SCORE_FOLD_TAIL")) : 1;       // tuning knob
    if (ng >= (uint32_t)SC_THREADS) return (unsigned)SC_THREADS;
    const unsigned full = ng / 32, tail = ng % 32;
    return 32u * std::max(1u, full + ((tail > (fold_tail ? 8u : 0u) || full == 0) ? 1u : 0u));
}

// k_score of the guides [g0, g0 + ng) over the block range `rng` of the plain store
static void launch_plain_score(vs_ctx *ctx, Scan &s, const unsigned long long *rng, uint32_t g0, uint32_t ng)
{
    static const int rot_shift = getenv("VARSCOT_SCORE_ROT") ? atoi(getenv("VARSCOT_SCORE_ROT")) : 3;                  // tuning knob
    ScoreArgs a;
    for (int i = 0; i < 2; ++i) { a.planes[i] = ctx->d_planes[i]; a.pos[i] = ctx->d_pos[i]; }
    a.rng = rng; a.cap = ctx->blocks_cap();
    a.n_guides = ng; a.guide_base = g0; a.pat_guides = s.n_guides; a.pat = ctx->d_pat;
    a.rot_shift = (uint32_t)rot_shift;
    a.hits = ctx->d_hits; a.n_hits = ctx->d_cnt + ctx->all_at() + 4; a.hit_cap = ctx->d_hits.cap;
    with_k(s.k, [&](auto K) { k_score<K.value><<<s.score_ctas, score_cta(ng), SC_SMEM_BYTES, ctx->stream>>>(a); });
    s.S.launches++; s.S.score_launches++;
}

// The index is resident: one launch over the whole store, plain or bucketed (after the class sort of the pass's guides)
static int score_resident(vs_ctx *ctx, Scan &s, uint32_t g0, uint32_t ng)
{
    cudaStream_t st = ctx->stream;
    CK(cudaEventRecord(ctx->t0[vs_ctx::T_SCORE], st));
    if (s.use_bk) {
        const int r = ctx->d_perm.grow(ctx, 2ull * BK_N * ng);
        if (r != VS_OK) return r;
        // the keys of this pass's guides, strand by strand ([2][ng])
        for (int i = 0; i < 2; ++i)
            CK(cudaMemcpyAsync(ctx->d_gkey + (size_t)i * ng, ctx->h_gkey + (size_t)i * s.n_guides + g0, (size_t)ng * sizeof(uint16_t), cudaMemcpyHostToDevice, st));
        s.S.h2d_bytes += 2ull * ng * sizeof(uint16_t);
        k_guide_classes<<<dim3(BK_N, 2), 128, 0, st>>>(ctx->d_gkey, ng, s.pp, ctx->d_perm, ctx->d_cls);
        BkScoreArgs b;
        for (int i = 0; i < 2; ++i) { b.planes[i] = ctx->d_bk_planes[i]; b.pos[i] = ctx->d_bk_pos[i]; }
        b.start = ctx->d_bk_ctl + 4 * BK_N;
        b.n_guides = ng; b.guide_base = g0; b.pat_guides = s.n_guides; b.pat = ctx->d_pat;
        b.perm = ctx->d_perm; b.cls = ctx->d_cls;
        b.hits = ctx->d_hits; b.n_hits = ctx->d_cnt + ctx->all_at() + 4; b.hit_cap = ctx->d_hits.cap;
        with_k(s.k, [&](auto K) { k_score_bucketed<K.value><<<s.score_ctas, SC_THREADS, SC_SMEM_BYTES, st>>>(b); });
        s.S.launches += 2; s.S.score_launches++;
    } else {
        launch_plain_score(ctx, s, ctx->d_cnt + ctx->all_at(), g0, ng);
    }
    CK(cudaEventRecord(ctx->t1[vs_ctx::T_SCORE], st));
    return VS_OK;
}

// The index is not resident: for every pipeline chunk [its upload, when the text comes from the host] -> k_extract into the
// whole-shard store -> k_score of the chunk's block range, all enqueued without host synchronisation
static int extract_pass(vs_ctx *ctx, Scan &s, uint32_t g0, uint32_t ng)
{
    cudaStream_t st = ctx->stream;
    CK(cudaMemsetAsync(ctx->d_cnt, 0, (ctx->all_at() + 4) * sizeof(unsigned long long), st));
    CK(cudaEventRecord(ctx->t0[vs_ctx::T_EXTRACT], st));
    auto extract_score = [&](uint32_t c) -> int {
        cudaEvent_t *E = &ctx->ev_pool[(size_t)EVC * c];
        const uint64_t c0 = s.plan[c], c1 = s.plan[c + 1];
        CK(cudaEventRecord(E[1], st));
        k_extract<<<(unsigned)((c1 - c0 + s.tile_words - 1) / s.tile_words), EX_THREADS, 0, st>>>(
            ctx->d_bases, ctx->d_masks, c0, c1, s.tile_words, s.first_word * 32 - s.origin, s.pp, ctx->d_planes[0], ctx->d_pos[0],
            ctx->d_planes[1], ctx->d_pos[1], ctx->blocks_cap(), ctx->d_cnt);
        k_extract_mark<<<1, 32, 0, st>>>(ctx->d_cnt, ctx->d_cnt + 4 + 4ull * c, ctx->d_cnt + ctx->all_at(), ctx->d_planes[0], ctx->d_planes[1], ctx->blocks_cap());
        s.S.launches += 2;
        CK(cudaEventRecord(E[2], st));
        CK(cudaEventRecord(E[3], st));
        launch_plain_score(ctx, s, ctx->d_cnt + 4 + 4ull * c, g0, ng);
        CK(cudaEventRecord(E[4], st));
        return VS_OK;
    };
    if (s.up.t) {
        const int r = enqueue_upload(ctx, s.up, s.plan, ctx->t0[vs_ctx::T_EXTRACT], s.S.h2d_bytes, s.S.launches, [&](uint32_t c, cudaStream_t ready) -> int {
            CK(cudaEventRecord(ctx->ev_pool[(size_t)EVC * c], ready));
            CK(cudaStreamWaitEvent(st, ctx->ev_pool[(size_t)EVC * c], 0));
            return extract_score(c);
        });
        return r == VS_OK ? VS_OK : abandon_upload(ctx, r);
    }
    for (uint32_t c = 0; c < s.n_chunks; ++c) {
        CK(cudaEventRecord(ctx->ev_pool[(size_t)EVC * c], st));
        const int r = extract_score(c);
        if (r != VS_OK) return r;
    }
    return VS_OK;
}

// One guide super-chunk [g0, g0 + ng): score the resident index or extract it, then read the counters back (one host
// synchronisation per attempt).  A buffer that proved too small (candidate store or hit buffer: only on text far from uniform)
// is regrown, or ng halved, and the pass repeated from the resident text / index.  found = the pass's hits, in d_hits.
static int run_pass(vs_ctx *ctx, Scan &s, uint32_t g0, uint32_t &ng, uint64_t &found)
{
    cudaStream_t st = ctx->stream;
    const unsigned long long *h = ctx->h_cnt, *h_rng = h + 4;
    const uint64_t cnt_words = ctx->all_at() + 8;
    int r;
    for (int attempt = 0;; ++attempt) {
        if (attempt == 4) return fail(ctx, VS_ERR_CUDA, "vs_scan: device buffers still too small after regrowing");
        CK(cudaMemsetAsync(ctx->d_cnt + ctx->all_at() + 4, 0, sizeof(unsigned long long), st));
        const bool resident = ctx->level >= vs_ctx::INDEX;
        if ((r = resident ? score_resident(ctx, s, g0, ng) : extract_pass(ctx, s, g0, ng)) != VS_OK) return r;
        if (cudaGetLastError() != cudaSuccess) return abandon_upload(ctx, fail(ctx, VS_ERR_CUDA, "vs_scan: a kernel launch failed"));
        CK(cudaMemcpyAsync(ctx->h_cnt, ctx->d_cnt, cnt_words * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        if (cudaStreamSynchronize(st) != cudaSuccess) return abandon_upload(ctx, fail(ctx, VS_ERR_CUDA, std::string("vs_scan: ") + cudaGetErrorString(cudaGetLastError())));
        s.S.d2h_bytes += cnt_words * sizeof(unsigned long long);
        if (resident) {
            float b = 0.f;
            CK(cudaEventElapsedTime(&b, ctx->t0[vs_ctx::T_SCORE], ctx->t1[vs_ctx::T_SCORE]));
            s.S.score_ms += b;
        } else {
            if (s.up.t) {                                    // the text is resident from here on
                if ((r = finish_upload(ctx, s.up, s.S.h2d_bytes)) != VS_OK) return abandon_upload(ctx, r);
                s.up.t = nullptr;
            }
            const uint64_t bf = h[2], br = h[3], most = std::max(bf, br);
            if (most > ctx->blocks_cap()) {                // the store overflowed (k_score skipped everything): regrow, extract again
                if ((r = ensure_blocks(ctx, (most + most / 32 + 64ull * s.n_chunks + BLK_GROUP) / BLK_GROUP * BLK_GROUP)) != VS_OK) return r;
                s.S.redo_chunks += s.n_chunks;
                continue;
            }
            vs_ctx::Index x{s.extra_pam, {0, 0}, {h[0], h[1]}, {bf, br}};
            for (uint32_t c = 0; c < s.n_chunks; ++c) { x.blocks[0] += h_rng[4 * c + 2] - h_rng[4 * c]; x.blocks[1] += h_rng[4 * c + 3] - h_rng[4 * c + 1]; }
            commit_index(ctx, x);
            for (uint32_t c = 0; c < s.n_chunks; ++c) {
                const cudaEvent_t *E = &ctx->ev_pool[(size_t)EVC * c];
                float a = 0.f, b = 0.f;
                CK(cudaEventElapsedTime(&a, E[1], E[2]));
                CK(cudaEventElapsedTime(&b, E[3], E[4]));
                s.S.extract_ms += a; s.S.score_ms += b;
            }
            if (s.src) CK(cudaEventElapsedTime(&s.S.upload_ms, ctx->t0[vs_ctx::T_EXTRACT], ctx->ev_pool[(size_t)EVC * (s.n_chunks - 1)]));
        }
        found = h[ctx->all_at() + 4];
        if (found <= ctx->d_hits.cap) return VS_OK;
        // device hit buffer too small: grow it (or halve the super-chunk once it is large) and repeat the pass over the index
        s.S.redo_chunks += s.n_chunks;
        if (found > (256ull << 20) && ng > 1) { ng = (ng + 1) / 2; continue; }
        if ((r = ctx->d_hits.grow(ctx, found + found / 8 + 1024)) != VS_OK) return r;
    }
}

// Deliver the hits of the super-chunk [g0, g0 + ng): raw as they are, or resolved to (contig, pos) and sorted on the device
// (k_resolve_hits -> radix sort -> k_pack_loc_hits) into the caller's buffer or through the sink.  One host synchronisation.
static int deliver(vs_ctx *ctx, Scan &s, uint32_t g0, uint32_t ng, uint64_t found)
{
    cudaStream_t st = ctx->stream;
    const uint64_t room = s.out_cap > s.total_out ? s.out_cap - s.total_out : 0, ncopy = std::min(found, room);
    int r;
    CK(cudaEventRecord(ctx->t0[vs_ctx::T_DELIVER], st));
    if (!s.resolved) {
        if (s.out_raw && ncopy) CK(cudaMemcpyAsync(s.out_raw + s.total_out, ctx->d_hits, ncopy * sizeof(vs_hit), cudaMemcpyDeviceToHost, st));
        s.S.d2h_bytes += ncopy * sizeof(vs_hit);
    } else if (found) {
        if (found > ctx->d_loc.cap) {
            const uint64_t cap = std::max<uint64_t>(found + found / 8, 1u << 16);
            if (ctx->d_keys[0].grow(ctx, cap) || ctx->d_keys[1].grow(ctx, cap) || ctx->d_vals[0].grow(ctx, cap) || ctx->d_vals[1].grow(ctx, cap) ||
                ctx->d_loc.grow(ctx, cap))
                return release_all(ctx->d_keys[0], ctx->d_keys[1], ctx->d_vals[0], ctx->d_vals[1], ctx->d_loc);
        }
        int guide_bits = 1;
        while ((1u << guide_bits) < ng) ++guide_bits;
        cub::DoubleBuffer<unsigned long long> dk(ctx->d_keys[0], ctx->d_keys[1]), dv(ctx->d_vals[0], ctx->d_vals[1]);
        size_t tmp = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp, dk, dv, (unsigned long long)found, 0, 49 + guide_bits, st));
        if (tmp > ctx->d_sort_tmp.cap && (r = ctx->d_sort_tmp.grow(ctx, tmp + tmp / 4)) != VS_OK) return r;
        const unsigned gb = (unsigned)((found + 255) / 256);
        k_resolve_hits<<<gb, 256, 0, st>>>(ctx->d_hits, found, ctx->d_cstart, ctx->text.n_cstart, ctx->text.first_contig, g0, ctx->d_keys[0], ctx->d_vals[0]);
        tmp = ctx->d_sort_tmp.cap;
        CK(cub::DeviceRadixSort::SortPairs(ctx->d_sort_tmp, tmp, dk, dv, (unsigned long long)found, 0, 49 + guide_bits, st));
        k_pack_loc_hits<<<gb, 256, 0, st>>>(dk.Current(), dv.Current(), found, ctx->d_loc);
        s.S.launches += 2 + 8;                              // + the radix sort's passes (CUB: histogram + one pass per 8 key bits)
        CK(cudaGetLastError());
        if (s.windows) {
            if (found > ctx->d_win.cap && (ctx->d_win.grow(ctx, found + found / 8) || ctx->h_win.grow(ctx, found + found / 8)))
                return release_all(ctx->d_win, ctx->h_win);
            k_loc_windows<<<gb, 256, 0, st>>>(ctx->d_loc, found, ctx->d_cstart, ctx->text.first_contig, ctx->d_bases,
                                              ctx->text.first_word * 32 - ctx->text.pos_origin, ctx->d_win);
            s.S.launches++;
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(ctx->h_win, ctx->d_win, found * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            s.S.d2h_bytes += found * sizeof(uint64_t);
        }
        if (s.sink) {
            if (found > ctx->h_stage.cap && (r = ctx->h_stage.grow(ctx, found + found / 8)) != VS_OK) return r;
            CK(cudaMemcpyAsync(ctx->h_stage, ctx->d_loc, found * sizeof(vs_loc_hit), cudaMemcpyDeviceToHost, st));
            s.S.d2h_bytes += found * sizeof(vs_loc_hit);
        } else {
            if (s.out_loc && ncopy) CK(cudaMemcpyAsync(s.out_loc + s.total_out, ctx->d_loc, ncopy * sizeof(vs_loc_hit), cudaMemcpyDeviceToHost, st));
            s.S.d2h_bytes += ncopy * sizeof(vs_loc_hit);
        }
    }
    CK(cudaEventRecord(ctx->t1[vs_ctx::T_DELIVER], st));
    CK(cudaStreamSynchronize(st));
    float a = 0.f;
    CK(cudaEventElapsedTime(&a, ctx->t0[vs_ctx::T_DELIVER], ctx->t1[vs_ctx::T_DELIVER]));
    s.S.resolve_ms += a;
    if (s.resolved && s.sink && found && s.sink(s.user, ctx->h_stage, s.windows ? ctx->h_win.p : nullptr, found, g0, g0 + ng) != 0)
        return fail(ctx, VS_ERR_ARG, "vs_scan_resolved: the sink aborted the scan");
    return VS_OK;
}

// One scan = guide super-chunks (sized to the device hit buffer; a single one for all but the densest configs), each a pass
// (run_pass) and a delivery (deliver).  The first pass over a shard whose index is not resident extracts it chunk by chunk,
// streaming the text in first when it comes from the host; later passes (later super-chunks; later scans with the same PAM
// set) score the resident index with one launch.
static int scan_engine(vs_ctx *ctx, Scan &s)
{
    if (const char *why = scan_arg_error(s.guides, s.n_guides, s.k, s.extra_pam)) return fail(ctx, VS_ERR_ARG, std::string("vs_scan: ") + why);
    CK(cudaSetDevice(ctx->device));
    if (s.n_hits) *s.n_hits = 0;
    ctx->last_n_hits = 0;
    const vs_text_view *src = s.src;
    if (!src) { s.n_words = ctx->text.n_words; s.first_word = ctx->text.first_word; }
    s.origin = src ? pos_origin_of(src, s.first_word, s.n_words) : ctx->text.pos_origin;
    int r = VS_OK;
    if (s.n_words == 0 || s.n_guides == 0) {             // nothing to score: a text from the host is made resident all the same
        if (src) r = s.n_words ? upload_text(ctx, src, s.first_word, s.n_words) : reserve_shard(ctx, src, s.first_word, 0, s.up);
        if (r != VS_OK) return r;
        if (s.stats) *s.stats = s.S;
        ctx->err.clear();
        return VS_OK;
    }
    if (src && (r = reserve_shard(ctx, src, s.first_word, s.n_words, s.up)) != VS_OK) return r;
    if (s.resolved && !src && !ctx->text.has_starts)
        return fail(ctx, VS_ERR_ARG, "vs_scan_resolved: the resident text was uploaded from a view without contig offsets");
    if (s.resolved && src && !s.up.shard.has_starts) return fail(ctx, VS_ERR_ARG, "vs_scan_resolved: the text view carries no contig offsets");
    make_pam(s.extra_pam, s.pp);
    s.plan = chunk_plan(s.n_words, ctx->chunk_words, src != nullptr);
    s.n_chunks = s.S.n_chunks = (uint32_t)(s.plan.size() - 1);
    // tile size: about 60 blocks (both strands) per 64-thread CTA at the expected PAM density pp.n / 16 per strand
    s.tile_words = default_tile_words(s.pp.n);
    if (const char *e = getenv("VARSCOT_TILE_WORDS")) s.tile_words = (uint32_t)atoi(e);      // tuning knob
    s.tile_words = std::max<uint32_t>(8, std::min<uint32_t>(s.tile_words, EX_MAX_WORDS));
    const uint64_t pat_entries = 2ull * s.n_guides * PAT_STRIDE;
    if (ctx->d_pat.grow(ctx, pat_entries) || ctx->h_pat.grow(ctx, pat_entries)) return release_all(ctx->d_pat, ctx->h_pat);
    // counters
    if (s.n_chunks > ctx->cnt_chunks) {
        const uint64_t nc = s.n_chunks + 8, words = 4 + 4 * (nc + 1) + 4 + 4;
        ctx->cnt_chunks = 0;
        drop_index(ctx);                                 // the whole-store range lived in the old buffer
        if (ctx->d_cnt.grow(ctx, words) || ctx->h_cnt.grow(ctx, words)) return release_all(ctx->d_cnt, ctx->h_cnt);
        ctx->cnt_chunks = nc;
    }
    // candidate store sized for the shard at the expected density (+15 %), regrown when it overflows
    const bool reuse = !src && ctx->level >= vs_ctx::INDEX && ctx->idx.pam == s.extra_pam;
    if (!reuse) {
        drop_index(ctx);
        if ((r = ensure_blocks(ctx, cand_store_blocks(s.n_words, s.pp.n, s.tile_words, s.n_chunks))) != VS_OK) return r;
    }
    // a resident index that is scanned again gets its bucketed form (built once; this scan pays for it)
    // (with few guides the classes of a bucket are a handful of 4-guide segments, and a small shard is scanned in about the
    // time the per-scan class sort takes: there the plain index is as fast or faster.  Measured on B200: 100 guides x 3.5
    // Gbases + 8 %, 100 guides x 0.44 Gbases - 9 %, 1000 guides + 58 %)
    const bool bucket_pays = s.n_guides >= 256 || (s.n_guides >= 64 && (double)s.n_guides * (double)s.n_words >= 5e9);
    s.use_bk = reuse && (ctx->bucket_mode == 2 || (ctx->bucket_mode == 1 && bucket_pays));
    if (s.use_bk && ctx->level != vs_ctx::BUCKETED && (r = build_bucket_index(ctx, s.pp, s.S.launches, s.S.index_build_ms)) != VS_OK) return r;
    s.S.index_reused = reuse ? (s.use_bk ? 2u : 1u) : 0u;
    if ((r = stage_guides(ctx, s)) != VS_OK) return r;
    // hit buffer and guide super-chunks
    const double per_guide = (double)s.n_words * 32.0 * hit_density(s.k, s.pp.n);
    const uint64_t want_hits = ctx->hit_cap_opt ? ctx->hit_cap_opt
                                                : std::min<uint64_t>(64ull << 20, std::max<uint64_t>(4ull << 20, (uint64_t)(per_guide * s.n_guides * 1.5) + 65536));
    if ((r = ctx->d_hits.grow(ctx, want_hits)) != VS_OK) return r;
    auto guides_per_pass = [&]() -> uint32_t {
        const double fit = per_guide > 0 ? (double)ctx->d_hits.cap / (per_guide * 1.5) : 1e30;
        uint64_t g = fit >= (double)s.n_guides ? s.n_guides : (uint64_t)std::max(1.0, fit);
        if (g > 32768) g = 32768;                            // the sort key holds 15 bits of guide index per delivery (and k_guide_classes 16)
        if (g < s.n_guides && g > SC_THREADS) g = g / SC_THREADS * SC_THREADS;
        return (uint32_t)g;
    };
    while (ctx->ev_pool.size() < (size_t)EVC * s.n_chunks) {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        ctx->ev_pool.push_back(e);
    }
    s.score_ctas = (unsigned)ctx->n_sm * 32;         // persistent: a multiple of the SM count, about four waves of resident CTAs (16 / 32 / 64 per SM measured: 32 is 3 % faster than 16, 64 no better)
    if (const char *e = getenv("VARSCOT_SCORE_CTAS_PER_SM")) s.score_ctas = (unsigned)ctx->n_sm * (unsigned)std::max(1, atoi(e));   // tuning knob
    cudaStream_t st = ctx->stream;
    CK(cudaEventRecord(ctx->t0[vs_ctx::T_SCAN], st));
    CK(cudaMemcpyAsync(ctx->d_pat, ctx->h_pat, pat_entries * sizeof(uint16_t), cudaMemcpyHostToDevice, st));
    s.S.h2d_bytes += pat_entries * sizeof(uint16_t);
    for (uint32_t g0 = 0, ng = 0; g0 < s.n_guides; g0 += ng) {
        ng = std::min<uint32_t>(guides_per_pass(), s.n_guides - g0);
        uint64_t found = 0;
        if ((r = run_pass(ctx, s, g0, ng, found)) != VS_OK) return r;
        s.S.guide_passes++;
        if ((r = deliver(ctx, s, g0, ng, found)) != VS_OK) return r;
        s.total_out += found;
        ctx->last_n_hits = found;                        // vs_scan_fetch serves the last super-chunk only (single-pass scans)
    }
    CK(cudaEventRecord(ctx->t1[vs_ctx::T_SCAN], st));
    CK(cudaStreamSynchronize(st));
    vs_scan_stats &S = s.S;
    CK(cudaEventElapsedTime(&S.total_ms, ctx->t0[vs_ctx::T_SCAN], ctx->t1[vs_ctx::T_SCAN]));
    S.n_cand_fwd = ctx->idx.cand[0]; S.n_cand_rev = ctx->idx.cand[1];
    S.n_blocks_fwd = ctx->idx.blocks[0]; S.n_blocks_rev = ctx->idx.blocks[1];
    S.n_hits = s.total_out;
    if (s.n_hits) *s.n_hits = s.total_out;
    if (!ctx->keep_index) drop_index(ctx);
    if (s.stats) *s.stats = S;
    ctx->err.clear();
    if (!s.sink && s.total_out > s.out_cap) {             // the caller's buffer took the first out_cap hits
        if (S.guide_passes > 1) return fail(ctx, VS_ERR_OVERFLOW, "vs_scan: caller hit buffer too small (several guide passes: enlarge it or use a sink)");
        return fail(ctx, VS_ERR_OVERFLOW, "vs_scan: caller hit buffer too small; use vs_scan_fetch");
    }
    return VS_OK;
}

// vs_hit carries a global 32-bit position: vs_scan, vs_scan_text and vs_scan_fetch serve texts within 4 Gbases only
static const char *const LEGACY_BEYOND_4G =
    "unordered hits carry global 32-bit positions, which end at 4 Gbases of text: scan this text with vs_scan_resolved or vs_map_records";

extern "C" int vs_scan(vs_ctx *ctx, const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                       vs_hit *out, uint64_t out_cap, uint64_t *n_hits, vs_scan_stats *stats)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_scan: ctx is NULL");
    if (ctx->text.pos_origin) return fail(ctx, VS_ERR_ARG, LEGACY_BEYOND_4G);
    Scan q;
    q.guides = guides; q.n_guides = n_guides; q.k = k; q.extra_pam = extra_pam;
    q.out_raw = out; q.out_cap = out_cap; q.n_hits = n_hits; q.stats = stats;
    return scan_engine(ctx, q);
}

extern "C" int vs_scan_text(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words,
                            const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                            vs_hit *out, uint64_t out_cap, uint64_t *n_hits, vs_scan_stats *stats)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_scan_text: ctx is NULL");
    int r = check_view(ctx, text, first_word, n_words);
    if (r != VS_OK) return r;
    if (text->n_words * 32 > (1ull << 32)) return fail(ctx, VS_ERR_ARG, LEGACY_BEYOND_4G);
    Scan q;
    q.src = text; q.first_word = first_word; q.n_words = n_words;
    q.guides = guides; q.n_guides = n_guides; q.k = k; q.extra_pam = extra_pam;
    q.out_raw = out; q.out_cap = out_cap; q.n_hits = n_hits; q.stats = stats;
    return scan_engine(ctx, q);
}

int vs::scan_resolved_ex(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words,
                         const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                         vs_loc_hit *out, uint64_t out_cap, uint64_t *n_hits, bool windows, loc_sink sink, void *user, vs_scan_stats *stats)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_scan_resolved: ctx is NULL");
    if (text) {
        int r = check_view(ctx, text, first_word, n_words);
        if (r != VS_OK) return r;
    }
    Scan q;
    q.src = text; q.first_word = first_word; q.n_words = n_words;
    q.guides = guides; q.n_guides = n_guides; q.k = k; q.extra_pam = extra_pam;
    q.resolved = true; q.out_loc = out; q.out_cap = out_cap; q.n_hits = n_hits; q.stats = stats;
    q.windows = windows; q.sink = sink; q.user = user;
    return scan_engine(ctx, q);
}

namespace {
struct PublicSink {
    vs_hit_sink sink;
    void *user;
    static int call(void *u, const vs_loc_hit *h, const uint64_t *, uint64_t n, uint32_t g0, uint32_t g1)
    {
        const PublicSink *p = static_cast<const PublicSink *>(u);
        return p->sink(p->user, h, n, g0, g1);
    }
};
}  // namespace

extern "C" int vs_scan_resolved(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words,
                                const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                                vs_loc_hit *out, uint64_t out_cap, uint64_t *n_hits, vs_hit_sink sink, void *user, vs_scan_stats *stats)
{
    PublicSink p{sink, user};
    return scan_resolved_ex(ctx, text, first_word, n_words, guides, n_guides, k, extra_pam, out, out_cap, n_hits, false,
                            sink ? &PublicSink::call : nullptr, &p, stats);
}

extern "C" int vs_scan_fetch(vs_ctx *ctx, vs_hit *out, uint64_t out_cap, uint64_t *n_hits)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_scan_fetch: ctx is NULL");
    if (ctx->text.pos_origin) return fail(ctx, VS_ERR_ARG, LEGACY_BEYOND_4G);
    if (n_hits) *n_hits = ctx->last_n_hits;
    if (ctx->last_n_hits > out_cap) return fail(ctx, VS_ERR_OVERFLOW, "vs_scan_fetch: buffer too small");
    CK(cudaSetDevice(ctx->device));
    if (ctx->last_n_hits) {
        if (!out) return fail(ctx, VS_ERR_ARG, "vs_scan_fetch: out is NULL");
        CK(cudaMemcpyAsync(out, ctx->d_hits, ctx->last_n_hits * sizeof(vs_hit), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    ctx->err.clear();
    return VS_OK;
}

extern "C" int vs_measure_int_peaks(vs_ctx *ctx, double *lop3_per_s, double *lds_words_per_s)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_measure_int_peaks: ctx is NULL");
    CK(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->device));
    const int grid = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    Buf<uint32_t> d_out;
    int r;
    if ((r = d_out.grow(ctx, (uint64_t)grid * threads)) != VS_OK) return r;
    cudaStream_t st = ctx->stream;
    const cudaEvent_t t0 = ctx->t0[vs_ctx::T_SCORE], t1 = ctx->t1[vs_ctx::T_SCORE];      // timed as a score launch
    float best[2] = {1e30f, 1e30f};                 // k_peak_lop3, k_peak_lds
    for (int rep = 0; rep < 5; ++rep)
        for (int i = 0; i < 2; ++i) {
            float ms = 0;
            CK(cudaEventRecord(t0, st));
            if (i == 0) k_peak_lop3<<<grid, threads, 0, st>>>(d_out, iters);
            else k_peak_lds<<<grid, threads, 0, st>>>(d_out, iters);
            CK(cudaEventRecord(t1, st));
            CK(cudaStreamSynchronize(st));
            CK(cudaEventElapsedTime(&ms, t0, t1));
            if (rep && ms < best[i]) best[i] = ms;
        }
    CK(cudaGetLastError());
    const double nthreads = (double)grid * threads;
    if (lop3_per_s) *lop3_per_s = nthreads * iters * 64.0 / (best[0] * 1e-3);
    if (lds_words_per_s) *lds_words_per_s = nthreads * iters * 8.0 / (best[1] * 1e-3);
    return VS_OK;
}
