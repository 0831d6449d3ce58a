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

struct vs_ctx {
    int device = -1;
    int n_sm = 148;
    cudaStream_t stream = nullptr;       // extraction + scoring + hit resolution
    cudaStream_t copy = nullptr;         // H2D of the next chunk (copies only, so that the copy engine never waits for a kernel)
    cudaStream_t prep = nullptr;         // small kernels that turn the uploaded mask source of a chunk into its window masks
    cudaEvent_t ev_copied = nullptr, ev_zeroed = nullptr, ev_starts = nullptr;
    cudaEvent_t ev[8] = {};
    std::vector<cudaEvent_t> ev_pool;    // per chunk: copied, extract start, extract done, score start, score done
    uint64_t chunk_words = DEFAULT_CHUNK_WORDS;
    // resident text shard: device word 0 = global word first_word; every position the device stores or emits (candidate
    // store, bucketed store, hits, contig starts) is global - pos_origin (see pos_origin_of)
    vs_bases *d_bases = nullptr;
    vs_masks *d_masks = nullptr;
    uint64_t words_cap = 0, n_words = 0, first_word = 0, pos_origin = 0;
    vs_mask_entry *d_sparse = nullptr;
    uint64_t sparse_cap = 0;
    // compact mask source path: the N and contig-end planes of the shard (+ halo word) and a staging area for their runs
    uint32_t *d_nm = nullptr, *d_em = nullptr;
    uint8_t *d_emcode = nullptr, *d_dense = nullptr;     // code bytes of the shard's contig-end plane; coded-block flags of the whole text
    uint64_t planes_cap = 0, dense_cap = 0;
    vs_plane_run *d_runs = nullptr;
    uint64_t runs_cap = 0;
    // contig starts of the shard (device-side hit resolution): derived from d_em, or uploaded
    uint32_t *d_cstart = nullptr, *d_tilecnt = nullptr, *d_cs_total = nullptr, *h_cs_total = nullptr;
    uint64_t cstart_cap = 0, tilecnt_cap = 0;
    uint32_t n_cstart = 0, first_contig = 0;
    bool cstart_valid = false;
    // counters (u64): [0..3] running candidates fwd / rev, block claims fwd / rev; [4 + 4 c ..] block range of chunk c
    // {lo fwd, lo rev, hi fwd, hi rev}; then the whole-store range [4]; then the hit counter
    unsigned long long *d_cnt = nullptr, *h_cnt = nullptr;
    uint64_t cnt_chunks = 0;
    // candidate store of the whole shard, per strand (the resident index)
    uint32_t *d_planes[2] = {nullptr, nullptr}, *d_pos[2] = {nullptr, nullptr};
    uint64_t blocks_cap = 0;
    bool idx_valid = false;
    int idx_pam = -2;
    uint64_t idx_blocks[2] = {0, 0}, idx_cand[2] = {0, 0};
    uint32_t idx_chunks = 0;
    uint64_t idx_end[2] = {0, 0};       // block claims incl. the padding of every chunk = the whole-store range
    int keep_index = 1;
    uint64_t hit_cap_opt = 0;
    // bucketed index (vs_bucket.cuh): the candidates regrouped by PAM kind + the VS_KEYLEN - 2 = 6 bases next to the PAM
    int bucket_mode = 1;                 // VS_OPT_BUCKET_INDEX: 0 never, 1 when a resident index is scanned again and it pays (guide count, shard size), 2 always
    bool bk_valid = false;
    uint32_t *d_bk_planes[2] = {nullptr, nullptr}, *d_bk_pos[2] = {nullptr, nullptr};
    uint64_t bk_cap[2] = {0, 0}, bk_blocks[2] = {0, 0};
    unsigned long long *d_bk_ctl = nullptr, *h_bk_ctl = nullptr;     // hist [2][BK_N], cursor [2][BK_N], start [2][BK_N + 1]
    uint16_t *d_perm = nullptr, *d_gkey = nullptr, *h_gkey = nullptr;
    uint32_t *d_cls = nullptr;
    uint64_t perm_cap = 0, gkey_cap = 0;
    float bk_build_ms = 0.f;
    // pattern table [2][n_guides][PAT_STRIDE] of uint16
    uint16_t *d_pat = nullptr, *h_pat = nullptr;
    uint64_t pat_cap = 0;
    // hits
    vs_hit *d_hits = nullptr;
    uint64_t hits_cap = 0, last_n_hits = 0;
    // resolution: sort keys / payloads (double buffers of the radix sort), packed records, sort scratch, pinned staging
    unsigned long long *d_keys[2] = {nullptr, nullptr}, *d_vals[2] = {nullptr, nullptr};
    vs_loc_hit *d_loc = nullptr, *h_stage = nullptr;
    uint64_t loc_cap = 0, stage_cap = 0;
    void *d_sort_tmp = nullptr;
    size_t sort_tmp_bytes = 0;
    std::string err;
};

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
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_starts, cudaEventDisableTiming);
    for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreate(&ctx->ev[i]);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_cs_total, sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMallocHost(&ctx->h_cs_total, sizeof(uint32_t));
    if (e != cudaSuccess) {
        std::string m = std::string("vs_ctx_create: ") + cudaGetErrorString(e);
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
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy) cudaStreamSynchronize(ctx->copy);
    if (ctx->prep) cudaStreamSynchronize(ctx->prep);
    cudaFree(ctx->d_bases); cudaFree(ctx->d_masks); cudaFree(ctx->d_sparse);
    cudaFree(ctx->d_nm); cudaFree(ctx->d_em); cudaFree(ctx->d_runs); cudaFree(ctx->d_emcode); cudaFree(ctx->d_dense);
    cudaFree(ctx->d_cstart); cudaFree(ctx->d_tilecnt); cudaFree(ctx->d_cs_total);
    if (ctx->h_cs_total) cudaFreeHost(ctx->h_cs_total);
    cudaFree(ctx->d_cnt);
    if (ctx->h_cnt) cudaFreeHost(ctx->h_cnt);
    for (int s = 0; s < 2; ++s) { cudaFree(ctx->d_planes[s]); cudaFree(ctx->d_pos[s]); cudaFree(ctx->d_keys[s]); cudaFree(ctx->d_vals[s]); }
    cudaFree(ctx->d_pat);
    if (ctx->h_pat) cudaFreeHost(ctx->h_pat);
    cudaFree(ctx->d_hits); cudaFree(ctx->d_loc); cudaFree(ctx->d_sort_tmp);
    for (int s = 0; s < 2; ++s) { cudaFree(ctx->d_bk_planes[s]); cudaFree(ctx->d_bk_pos[s]); }
    cudaFree(ctx->d_bk_ctl); cudaFree(ctx->d_perm); cudaFree(ctx->d_gkey); cudaFree(ctx->d_cls);
    if (ctx->h_bk_ctl) cudaFreeHost(ctx->h_bk_ctl);
    if (ctx->h_gkey) cudaFreeHost(ctx->h_gkey);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    for (int i = 0; i < 8; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy) cudaStreamDestroy(ctx->copy);
    if (ctx->prep) cudaStreamDestroy(ctx->prep);
    if (ctx->ev_copied) cudaEventDestroy(ctx->ev_copied);
    if (ctx->ev_zeroed) cudaEventDestroy(ctx->ev_zeroed);
    if (ctx->ev_starts) cudaEventDestroy(ctx->ev_starts);
    delete ctx;
}

extern "C" int vs_ctx_set_option(vs_ctx *ctx, int option, int64_t value)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_ctx_set_option: ctx is NULL");
    switch (option) {
    case VS_OPT_KEEP_INDEX: ctx->keep_index = value != 0; if (!ctx->keep_index) ctx->idx_valid = false; return VS_OK;
    case VS_OPT_HIT_CAPACITY: if (value < 0) break; ctx->hit_cap_opt = (uint64_t)value; return VS_OK;
    case VS_OPT_BUCKET_INDEX: if (value < 0 || value > 2) break; ctx->bucket_mode = (int)value; if (!value) ctx->bk_valid = false; return VS_OK;
    default: break;
    }
    return fail(ctx, VS_ERR_ARG, "vs_ctx_set_option: unknown option or bad value");
}

extern "C" int vs_index_drop(vs_ctx *ctx)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_index_drop: ctx is NULL");
    ctx->idx_valid = false; ctx->bk_valid = false;
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

// persistent grid: `ctas` CTAs of `threads` threads stride over the batches of the block range in a.rng
template <int K>
static void launch_score(const ScoreArgs &a, unsigned ctas, unsigned threads, cudaStream_t st)
{
    k_score<K><<<ctas, threads, SC_SMEM_BYTES, st>>>(a);
}

static void dispatch_score(int k, const ScoreArgs &a, unsigned ctas, unsigned threads, cudaStream_t st)
{
    switch (k) {
    case 0: launch_score<0>(a, ctas, threads, st); break;
    case 1: launch_score<1>(a, ctas, threads, st); break;
    case 2: launch_score<2>(a, ctas, threads, st); break;
    case 3: launch_score<3>(a, ctas, threads, st); break;
    case 4: launch_score<4>(a, ctas, threads, st); break;
    case 5: launch_score<5>(a, ctas, threads, st); break;
    case 6: launch_score<6>(a, ctas, threads, st); break;
    case 7: launch_score<7>(a, ctas, threads, st); break;
    default: launch_score<8>(a, ctas, threads, st); break;
    }
}

template <int K>
static void launch_score_bk(const BkScoreArgs &a, unsigned ctas, unsigned threads, cudaStream_t st)
{
    k_score_bucketed<K><<<ctas, threads, SC_SMEM_BYTES, st>>>(a);
}

static void dispatch_score_bk(int k, const BkScoreArgs &a, unsigned ctas, unsigned threads, cudaStream_t st)
{
    switch (k) {
    case 0: launch_score_bk<0>(a, ctas, threads, st); break;
    case 1: launch_score_bk<1>(a, ctas, threads, st); break;
    case 2: launch_score_bk<2>(a, ctas, threads, st); break;
    case 3: launch_score_bk<3>(a, ctas, threads, st); break;
    case 4: launch_score_bk<4>(a, ctas, threads, st); break;
    case 5: launch_score_bk<5>(a, ctas, threads, st); break;
    case 6: launch_score_bk<6>(a, ctas, threads, st); break;
    case 7: launch_score_bk<7>(a, ctas, threads, st); break;
    default: launch_score_bk<8>(a, ctas, threads, st); break;
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
static int ensure_text_buffers(vs_ctx *ctx, uint64_t n_words)
{
    if (n_words + 1 > ctx->words_cap) {
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaStreamSynchronize(ctx->copy));
        cudaFree(ctx->d_bases); cudaFree(ctx->d_masks);
        ctx->d_bases = nullptr; ctx->d_masks = nullptr; ctx->words_cap = 0;
        CK(cudaMalloc(&ctx->d_bases, (n_words + 1) * sizeof(vs_bases)));
        CK(cudaMalloc(&ctx->d_masks, (n_words + 1) * sizeof(vs_masks)));
        ctx->words_cap = n_words + 1;
    }
    return VS_OK;
}

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
        // N plane and contig-end plane (zeroed by begin_mask_source): the run lists go to the staging area, the code bytes of
        // coded blocks to their own buffer; the expand, fill and mask kernels run on the preparation stream
        vs_plane_run *nm_dst = nullptr, *em_dst = nullptr;
        uint64_t nm_n = 0, em_n = 0;
        auto stage = [&](const vs_plane_run *runs, uint64_t a, uint64_t b, vs_plane_run *&dst, uint64_t &cnt) -> int {
            cnt = b > a ? b - a : 0;
            if (!cnt) return VS_OK;
            if (staged + cnt > ctx->runs_cap) return fail(ctx, VS_ERR_CUDA, "run staging area too small");
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
        sparse = (e1 - e0) * sizeof(vs_mask_entry) < n * sizeof(vs_masks) * 3 / 4 && staged + (e1 - e0) <= ctx->sparse_cap;
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
        if (n_words + 1 > ctx->planes_cap) {
            CK(cudaStreamSynchronize(ctx->copy));
            cudaFree(ctx->d_nm); cudaFree(ctx->d_em); cudaFree(ctx->d_emcode);
            ctx->d_nm = ctx->d_em = nullptr; ctx->d_emcode = nullptr; ctx->planes_cap = 0;
            CK(cudaMalloc(&ctx->d_nm, (n_words + 1) * sizeof(uint32_t)));
            CK(cudaMalloc(&ctx->d_em, (n_words + 1) * sizeof(uint32_t)));
            CK(cudaMalloc(&ctx->d_emcode, n_words + 1));
            ctx->planes_cap = n_words + 1;
        }
        const uint64_t n_blocks = (t->n_words + VS_EM_BLOCK) / VS_EM_BLOCK;
        if (n_blocks > ctx->dense_cap) {
            CK(cudaStreamSynchronize(ctx->copy));
            CK(cudaStreamSynchronize(ctx->prep));
            cudaFree(ctx->d_dense); ctx->d_dense = nullptr; ctx->dense_cap = 0;
            CK(cudaMalloc(&ctx->d_dense, n_blocks));
            ctx->dense_cap = n_blocks;
        }
        uint64_t a0, a1, b0, b1;
        runs_in_range(t->nm_runs, t->n_nm_runs, first_word, first_word + n_words + 1, a0, a1);
        runs_in_range(t->em_runs, t->n_em_runs, first_word, first_word + n_words + 1, b0, b1);
        const uint64_t n_chunks = (n_words + ctx->chunk_words - 1) / ctx->chunk_words + 3;     // + the tapered tail of chunk_plan()
        const uint64_t need = (a1 - a0) + (b1 - b0) + 4 * n_chunks + 16;
        if (need > ctx->runs_cap) {
            CK(cudaStreamSynchronize(ctx->copy));
            cudaFree(ctx->d_runs); ctx->d_runs = nullptr; ctx->runs_cap = 0;
            CK(cudaMalloc(&ctx->d_runs, need * sizeof(vs_plane_run)));
            ctx->runs_cap = need;
        }
        return VS_OK;
    }
    if (!t->sparse || t->n_sparse == 0) return VS_OK;
    const vs_mask_entry *sb = t->sparse, *se = t->sparse + t->n_sparse;
    auto lb = [&](uint64_t w) { return (uint64_t)(std::lower_bound(sb, se, w, [](const vs_mask_entry &x, uint64_t v) { return x.word < v; }) - sb); };
    uint64_t need = lb(first_word + n_words) - lb(first_word);
    if (need > ctx->sparse_cap) {
        CK(cudaStreamSynchronize(ctx->copy));
        cudaFree(ctx->d_sparse); ctx->d_sparse = nullptr; ctx->sparse_cap = 0;
        CK(cudaMalloc(&ctx->d_sparse, need * sizeof(vs_mask_entry)));
        ctx->sparse_cap = need;
    }
    return VS_OK;
}

// Start of an upload of a view with a compact mask source: zero both planes of the shard on the preparation stream
// (after `after`, an event of the caller's stream, if given) and make the copy stream wait for it — the dense blocks of
// the coded-block flags of the contig-end plane go to the device once per upload.
static int begin_mask_source(vs_ctx *ctx, const vs_text_view *t, uint64_t n_words, cudaEvent_t after)
{
    if (!has_mask_source(t)) return VS_OK;
    if (after) CK(cudaStreamWaitEvent(ctx->prep, after, 0));
    CK(cudaMemsetAsync(ctx->d_nm, 0, (n_words + 1) * sizeof(uint32_t), ctx->prep));
    CK(cudaMemsetAsync(ctx->d_em, 0, (n_words + 1) * sizeof(uint32_t), ctx->prep));
    CK(cudaMemcpyAsync(ctx->d_dense, t->em_dense, (t->n_words + VS_EM_BLOCK) / VS_EM_BLOCK, cudaMemcpyHostToDevice, ctx->prep));
    CK(cudaEventRecord(ctx->ev_zeroed, ctx->prep));
    CK(cudaStreamWaitEvent(ctx->copy, ctx->ev_zeroed, 0));
    return VS_OK;
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

static int ensure_starts_buffers(vs_ctx *ctx, const StartsPlan &p, uint64_t n_words)
{
    const uint64_t need = (uint64_t)(p.c_last - p.c_first) + 4;
    if (need > ctx->cstart_cap) {
        CK(cudaStreamSynchronize(ctx->stream)); CK(cudaStreamSynchronize(ctx->prep));
        cudaFree(ctx->d_cstart); ctx->d_cstart = nullptr; ctx->cstart_cap = 0;
        CK(cudaMalloc(&ctx->d_cstart, need * sizeof(uint32_t)));
        ctx->cstart_cap = need;
    }
    const uint64_t tiles = (n_words + CS_TILE - 1) / CS_TILE + 1;
    if (tiles > ctx->tilecnt_cap) {
        CK(cudaStreamSynchronize(ctx->prep));
        cudaFree(ctx->d_tilecnt); ctx->d_tilecnt = nullptr; ctx->tilecnt_cap = 0;
        CK(cudaMalloc(&ctx->d_tilecnt, tiles * sizeof(uint32_t)));
        ctx->tilecnt_cap = tiles;
    }
    return VS_OK;
}

// enqueue the derivation from the contig-end plane on `st` (after the last chunk's planes are complete on that stream)
// (positions relative to `origin`; the first contig may start before it: its start is stored modulo 2^32, see k_resolve_hits)
static int enqueue_starts_from_plane(vs_ctx *ctx, const vs_text_view *t, const StartsPlan &p, uint64_t first_word, uint64_t n_words,
                                     uint64_t origin, cudaStream_t st, uint32_t &launches)
{
    const unsigned tiles = (unsigned)((n_words + CS_TILE - 1) / CS_TILE);
    k_contig_starts_count<<<tiles, 256, 0, st>>>(ctx->d_em, n_words, ctx->d_tilecnt);
    k_contig_starts_scan<<<1, 1024, 0, st>>>(ctx->d_tilecnt, tiles, ctx->d_cs_total);
    k_contig_starts_scatter<<<tiles, 256, 0, st>>>(ctx->d_em, n_words, ctx->d_tilecnt, first_word * 32 - origin,
                                                   (uint32_t)(t->contig_off[p.c_first] - origin), ctx->d_cstart);
    launches += 3;
    CK(cudaMemcpyAsync(ctx->h_cs_total, ctx->d_cs_total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    return VS_OK;
}

// after the stream that ran enqueue_starts_from_plane has been synchronised: accept the derived starts, or upload the host's
static int finish_contig_starts(vs_ctx *ctx, const vs_text_view *t, const StartsPlan &p, bool derived, uint64_t origin, uint64_t &h2d_bytes)
{
    ctx->cstart_valid = false;
    if (!p.usable) return VS_OK;
    ctx->first_contig = p.c_first;
    if (derived && *ctx->h_cs_total == p.expect_bits) {
        ctx->n_cstart = p.c_last - p.c_first + 1;
        ctx->cstart_valid = true;
        return VS_OK;
    }
    // empty contigs inside the range, or no contig-end plane on the device: the offsets themselves (32-bit, relative to origin)
    const uint32_t n = p.c_last - p.c_first + 1;
    std::vector<uint32_t> h(n);
    for (uint32_t i = 0; i < n; ++i) h[i] = (uint32_t)(t->contig_off[p.c_first + i] - origin);
    CK(cudaMemcpyAsync(ctx->d_cstart, h.data(), (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    h2d_bytes += (uint64_t)n * sizeof(uint32_t);
    ctx->n_cstart = n;
    ctx->cstart_valid = true;
    return VS_OK;
}

// leave no copy in flight that still reads the caller's buffers, and no half-resident text behind
static int abandon_upload(vs_ctx *ctx, int rc)
{
    cudaStreamSynchronize(ctx->copy); cudaStreamSynchronize(ctx->prep); cudaStreamSynchronize(ctx->stream);
    (void)cudaGetLastError();
    ctx->n_words = 0; ctx->pos_origin = 0; ctx->idx_valid = false; ctx->bk_valid = false; ctx->cstart_valid = false;
    return rc;
}

extern "C" int vs_text_upload(vs_ctx *ctx, const vs_text_view *t, uint64_t first_word, uint64_t n_words)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_text_upload: ctx is NULL");
    int r = check_view(ctx, t, first_word, n_words);
    if (r != VS_OK) return r;
    CK(cudaSetDevice(ctx->device));
    const uint64_t origin = pos_origin_of(t, first_word, n_words);
    ctx->n_words = 0; ctx->pos_origin = 0; ctx->idx_valid = false; ctx->bk_valid = false; ctx->cstart_valid = false;      // nothing is resident until the upload has completed
    if ((r = ensure_text_buffers(ctx, n_words)) != VS_OK) return r;
    if ((r = ensure_sparse_staging(ctx, t, first_word, n_words)) != VS_OK) return r;
    const StartsPlan sp = plan_contig_starts(t, first_word, n_words);
    if (sp.usable && (r = ensure_starts_buffers(ctx, sp, n_words)) != VS_OK) return r;
    uint64_t sparse_used = 0, bytes = 0;
    uint32_t launches = 0;
    cudaStream_t ready = ctx->copy;
    if ((r = begin_mask_source(ctx, t, n_words, nullptr)) != VS_OK) return abandon_upload(ctx, r);
    for (uint64_t c0 = 0; c0 < n_words; c0 += ctx->chunk_words) {
        uint64_t c1 = std::min(n_words, c0 + ctx->chunk_words);
        if ((r = enqueue_chunk_copy(ctx, t, first_word, c0, c1, sparse_used, bytes, launches, ready)) != VS_OK) return abandon_upload(ctx, r);
    }
    const bool derive = sp.usable && has_mask_source(t);
    if (derive && (r = enqueue_starts_from_plane(ctx, t, sp, first_word, n_words, origin, ctx->prep, launches)) != VS_OK) return abandon_upload(ctx, r);
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(ctx->copy) != cudaSuccess || cudaStreamSynchronize(ctx->prep) != cudaSuccess)
        return abandon_upload(ctx, fail(ctx, VS_ERR_CUDA, "vs_text_upload: the upload failed on the device"));
    if ((r = finish_contig_starts(ctx, t, sp, derive, origin, bytes)) != VS_OK) return abandon_upload(ctx, r);
    ctx->n_words = n_words;
    ctx->first_word = first_word;
    ctx->pos_origin = origin;
    ctx->err.clear();
    return VS_OK;
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

// ---- bucketed index (vs_bucket.cuh) --------------------------------------------------------------------------------
// Built from the resident plain index and the resident text: bucket histogram -> padded bucket starts -> positions
// regrouped by bucket -> blocks gathered from the text.  One host synchronisation (the store is sized by the padded total).
static int build_bucket_index(vs_ctx *ctx, const PamParams &pp, uint32_t &launches)
{
    cudaStream_t st = ctx->stream;
    const size_t ctl_words = 2 * BK_N + 2 * BK_N + 2 * (BK_N + 1);
    if (!ctx->d_bk_ctl) {
        CK(cudaMalloc(&ctx->d_bk_ctl, ctl_words * sizeof(unsigned long long)));
        CK(cudaMallocHost(&ctx->h_bk_ctl, 2 * (BK_N + 1) * sizeof(unsigned long long)));
    }
    unsigned long long *d_hist = ctx->d_bk_ctl, *d_cursor = d_hist + 2 * BK_N, *d_start = d_cursor + 2 * BK_N;
    const unsigned long long *d_all = ctx->d_cnt + 4 + 4 * (ctx->cnt_chunks + 1);
    CK(cudaEventRecord(ctx->ev[7], st));
    CK(cudaMemsetAsync(d_hist, 0, 2 * BK_N * sizeof(unsigned long long), st));
    const uint64_t max_blocks = std::max(ctx->idx_end[0], ctx->idx_end[1]);
    const dim3 grid((unsigned)((max_blocks + BKB_THREADS - 1) / BKB_THREADS), 2);
    static bool smem_opt_in = false;                 // 48 KB of dynamic shared memory: at the default limit, opt in anyway
    if (!smem_opt_in) {
        CK(cudaFuncSetAttribute(k_bucket_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, BK_HIST_SMEM));
        CK(cudaFuncSetAttribute(k_bucket_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, BK_HIST_SMEM));
        smem_opt_in = true;
    }
    if (max_blocks) k_bucket_hist<<<grid, BKB_THREADS, BK_HIST_SMEM, st>>>(ctx->d_planes[0], ctx->d_planes[1], d_all, pp, d_hist);
    k_bucket_scan<<<2, 1024, 0, st>>>(d_hist, d_start, d_cursor);
    launches += 2;
    CK(cudaMemcpyAsync(ctx->h_bk_ctl, d_start, 2 * (BK_N + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int s = 0; s < 2; ++s) {
        const uint64_t nb = ctx->h_bk_ctl[s * (BK_N + 1) + BK_N];
        ctx->bk_blocks[s] = nb;
        if (nb > ctx->bk_cap[s]) {
            cudaFree(ctx->d_bk_planes[s]); cudaFree(ctx->d_bk_pos[s]);
            ctx->d_bk_planes[s] = ctx->d_bk_pos[s] = nullptr; ctx->bk_cap[s] = 0;
            const uint64_t cap = nb + nb / 64 + SC_NB;
            CK(cudaMalloc(&ctx->d_bk_planes[s], cap * BLK_WORDS * sizeof(uint32_t)));
            CK(cudaMalloc(&ctx->d_bk_pos[s], cap * 32 * sizeof(uint32_t)));
            ctx->bk_cap[s] = cap;
        }
        if (nb) CK(cudaMemsetAsync(ctx->d_bk_pos[s], 0xFF, nb * 32 * sizeof(uint32_t), st));
    }
    if (max_blocks) {
        k_bucket_scatter<<<grid, BKB_THREADS, BK_HIST_SMEM, st>>>(ctx->d_planes[0], ctx->d_planes[1], ctx->d_pos[0], ctx->d_pos[1], d_all, pp, d_cursor,
                                                        ctx->d_bk_pos[0], ctx->d_bk_pos[1], ctx->bk_blocks[0] * 32, ctx->bk_blocks[1] * 32);
        launches++;
    }
    for (int s = 0; s < 2; ++s)
        if (ctx->bk_blocks[s]) {
            k_bucket_gather<<<(unsigned)((ctx->bk_blocks[s] + 63) / 64), 64, 0, st>>>(ctx->d_bases, ctx->d_masks, ctx->first_word * 32 - ctx->pos_origin, ctx->d_bk_pos[s],
                                                                                     ctx->bk_blocks[s], ctx->d_bk_planes[s]);
            launches++;
        }
    CK(cudaEventRecord(ctx->ev[6], st));
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    CK(cudaEventElapsedTime(&ctx->bk_build_ms, ctx->ev[7], ctx->ev[6]));
    ctx->bk_valid = true;
    return VS_OK;
}

struct ScanReq {
    const vs_text_view *src = nullptr;       // stream the text from the host (vs_scan_text) or scan the resident shard
    uint64_t first_word = 0, n_words = 0;
    const uint8_t *guides = nullptr;
    uint32_t n_guides = 0;
    int k = 0, extra_pam = -1;
    bool resolved = false;                   // raw unordered vs_hit, or resolved + sorted vs_loc_hit
    vs_hit *out_raw = nullptr;
    vs_loc_hit *out_loc = nullptr;
    uint64_t out_cap = 0;
    uint64_t *n_hits = nullptr;
    vs_hit_sink sink = nullptr;
    void *user = nullptr;
    vs_scan_stats *stats = nullptr;
};

// One scan = guide super-chunks (sized to the device hit buffer; a single one for all but the densest configs) x
//   * the candidate index is not resident: for every pipeline chunk of the shard [H2D on the copy stream when the text
//     comes from the host] -> k_extract into the whole-shard store -> k_score of that chunk's block range, all enqueued
//     without host synchronisation; this leaves the index resident;
//   * the index is resident (later super-chunks; later scans with the same PAM set): one k_score launch over the store.
// After each super-chunk the counters are read back; raw hits are downloaded as they are, resolved hits go through
// k_resolve_hits -> radix sort -> k_pack_loc_hits first.  A buffer that proves too small (candidate store or hit buffer:
// only on text far from uniform) is regrown and the pass repeated from the resident text / index.
static int scan_engine(vs_ctx *ctx, const ScanReq &q)
{
    const int k = q.k;
    const uint32_t n_guides = q.n_guides;
    if (k < 0 || k > VS_MAX_MISMATCHES) return fail(ctx, VS_ERR_ARG, "vs_scan: mismatches must lie between 0 and 8");
    if (q.extra_pam < -1 || q.extra_pam > 15) return fail(ctx, VS_ERR_ARG, "vs_scan: extra_pam must be -1 or 4*x+y");
    if (n_guides && !q.guides) return fail(ctx, VS_ERR_ARG, "vs_scan: guides is NULL");
    if (n_guides >= (1u << 24)) return fail(ctx, VS_ERR_ARG, "vs_scan: at most 2^24-1 guides per call");
    for (uint64_t i = 0; i < (uint64_t)n_guides * VS_GLEN; ++i)
        if (q.guides[i] > 3) return fail(ctx, VS_ERR_ARG, "vs_scan: guide codes must be 0..3");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    vs_scan_stats S;
    memset(&S, 0, sizeof(S));
    if (q.n_hits) *q.n_hits = 0;
    ctx->last_n_hits = 0;
    int r;
    const vs_text_view *src = q.src;
    uint64_t n_words = src ? q.n_words : ctx->n_words;
    const uint64_t first_word = src ? q.first_word : ctx->first_word;
    const uint64_t origin = src ? pos_origin_of(src, first_word, n_words) : ctx->pos_origin;
    StartsPlan sp;
    if (src) {
        ctx->n_words = 0; ctx->pos_origin = 0; ctx->idx_valid = false; ctx->bk_valid = false; ctx->cstart_valid = false;      // nothing is resident until the pass has completed
        if ((r = ensure_text_buffers(ctx, n_words)) != VS_OK) return r;
        if ((r = ensure_sparse_staging(ctx, src, first_word, n_words)) != VS_OK) return r;
        sp = plan_contig_starts(src, first_word, n_words);
        if (sp.usable && (r = ensure_starts_buffers(ctx, sp, n_words)) != VS_OK) return r;
    }
    if (n_words == 0 || n_guides == 0) {
        if (src && n_words) { r = vs_text_upload(ctx, src, first_word, n_words); if (r != VS_OK) return r; }
        if (q.stats) *q.stats = S;
        ctx->err.clear();
        return VS_OK;
    }
    if (q.resolved && !src && !ctx->cstart_valid)
        return fail(ctx, VS_ERR_ARG, "vs_scan_resolved: the resident text was uploaded from a view without contig offsets");
    if (q.resolved && src && !sp.usable) return fail(ctx, VS_ERR_ARG, "vs_scan_resolved: the text view carries no contig offsets");
    PamParams pp;
    make_pam(q.extra_pam, pp);
    const uint64_t chunk_words = ctx->chunk_words;
    const std::vector<uint64_t> plan = chunk_plan(n_words, chunk_words, src != nullptr);
    const uint32_t n_chunks = (uint32_t)(plan.size() - 1);
    // tile size: about 60 blocks (both strands) per 64-thread CTA at the expected PAM density pp.n / 16 per strand
    uint32_t tile_words = (uint32_t)(60.0 * 16.0 / (2.0 * pp.n)) & ~7u;
    if (const char *e = getenv("VARSCOT_TILE_WORDS")) tile_words = (uint32_t)atoi(e);      // tuning knob
    if (tile_words > (uint32_t)EX_MAX_WORDS) tile_words = EX_MAX_WORDS;
    if (tile_words < 8) tile_words = 8;
    S.n_chunks = n_chunks;

    // pattern table [strand][guide][PAT_STRIDE] (uint16 plane offsets, see pat_slot), staged in pinned memory
    const uint64_t pat_entries = 2ull * n_guides * PAT_STRIDE;
    if (pat_entries > ctx->pat_cap) {
        CK(cudaStreamSynchronize(st));
        cudaFree(ctx->d_pat); if (ctx->h_pat) cudaFreeHost(ctx->h_pat);
        ctx->d_pat = ctx->h_pat = nullptr; ctx->pat_cap = 0;
        CK(cudaMalloc(&ctx->d_pat, pat_entries * sizeof(uint16_t)));
        CK(cudaMallocHost(&ctx->h_pat, pat_entries * sizeof(uint16_t)));
        ctx->pat_cap = pat_entries;
    }
    for (int s = 0; s < 2; ++s)
        for (uint32_t g = 0; g < n_guides; ++g) {
            uint16_t *dst = ctx->h_pat + ((size_t)s * n_guides + g) * PAT_STRIDE;
            const uint8_t *gd = q.guides + (size_t)g * VS_GLEN;
            for (int j = 0; j < VS_GLEN; ++j) {
                const int i = slot_position(s, j);
                const int b = s ? 3 - gd[VS_GLEN - 1 - i] : gd[i];      // reverse pass scores revcomp(guide), bidir_mapping.cpp:293
                dst[j] = pat_slot(s, j, b);
            }
            dst[VS_GLEN] = 0;
        }
    // counters
    if (n_chunks > ctx->cnt_chunks) {
        CK(cudaStreamSynchronize(st));
        cudaFree(ctx->d_cnt); if (ctx->h_cnt) cudaFreeHost(ctx->h_cnt);
        ctx->d_cnt = ctx->h_cnt = nullptr; ctx->cnt_chunks = 0;
        uint64_t nc = n_chunks + 8;
        CK(cudaMalloc(&ctx->d_cnt, (4 + 4 * (nc + 1) + 4 + 4) * sizeof(unsigned long long)));
        CK(cudaMallocHost(&ctx->h_cnt, (4 + 4 * (nc + 1) + 4 + 4) * sizeof(unsigned long long)));
        ctx->cnt_chunks = nc;
        ctx->idx_valid = false; ctx->bk_valid = false;       // the whole-store range lived in the old buffer
    }
    const uint64_t cnt_words = 4 + 4 * (ctx->cnt_chunks + 1) + 4 + 4;
    unsigned long long *d_rng = ctx->d_cnt + 4, *d_all = ctx->d_cnt + 4 + 4 * (ctx->cnt_chunks + 1), *d_hitcnt = d_all + 4;
    unsigned long long *h_rng = ctx->h_cnt + 4, *h_hitcnt = ctx->h_cnt + (d_hitcnt - ctx->d_cnt);
    // candidate store sized for the shard at the expected density (+15 %), regrown when it overflows
    auto ensure_blocks = [&](uint64_t need) -> int {
        if (need <= ctx->blocks_cap) return VS_OK;
        CK(cudaStreamSynchronize(st));
        for (int s = 0; s < 2; ++s) {
            cudaFree(ctx->d_planes[s]); cudaFree(ctx->d_pos[s]);
            ctx->d_planes[s] = ctx->d_pos[s] = nullptr;
        }
        ctx->blocks_cap = 0; ctx->idx_valid = false; ctx->bk_valid = false;
        for (int s = 0; s < 2; ++s) {
            CK(cudaMalloc(&ctx->d_planes[s], need * BLK_WORDS * sizeof(uint32_t)));
            CK(cudaMalloc(&ctx->d_pos[s], need * 32 * sizeof(uint32_t)));
        }
        ctx->blocks_cap = need;
        return VS_OK;
    };
    const bool reuse = !src && ctx->idx_valid && ctx->idx_pam == q.extra_pam;
    if (!reuse) {
        ctx->idx_valid = false; ctx->bk_valid = false;
        const uint64_t tiles = (n_words + tile_words - 1) / tile_words;
        uint64_t est = (uint64_t)((double)n_words * pp.n / 16.0 * 1.15) + tiles + 64ull * n_chunks + 256;
        est = (est + BLK_GROUP - 1) / BLK_GROUP * BLK_GROUP;
        if ((r = ensure_blocks(est)) != VS_OK) return r;
    }
    // a resident index that is scanned again gets its bucketed form (built once; this scan pays for it)
    bool use_bk = false;
    // (with few guides the classes of a bucket are a handful of 4-guide segments, and a small shard is scanned in about the
    // time the per-scan class sort takes: there the plain index is as fast or faster.  Measured on B200: 100 guides x 3.5
    // Gbases + 8 %, 100 guides x 0.44 Gbases - 9 %, 1000 guides + 58 %)
    const bool bucket_pays = n_guides >= 256 || (n_guides >= 64 && (double)n_guides * (double)n_words >= 5e9);
    if (reuse && (ctx->bucket_mode == 2 || (ctx->bucket_mode == 1 && bucket_pays))) {
        if (!ctx->bk_valid) {
            if ((r = build_bucket_index(ctx, pp, S.launches)) != VS_OK) return r;
            S.index_build_ms = ctx->bk_build_ms;
        }
        use_bk = true;
    }
    if (use_bk) {
        // keys of the patterns and, per guide pass, the guides of every bucket sorted by their key mismatches
        const uint64_t gk = 2ull * n_guides;
        if (gk > ctx->gkey_cap) {
            CK(cudaStreamSynchronize(st));
            cudaFree(ctx->d_gkey); if (ctx->h_gkey) cudaFreeHost(ctx->h_gkey);
            ctx->d_gkey = ctx->h_gkey = nullptr; ctx->gkey_cap = 0;
            CK(cudaMalloc(&ctx->d_gkey, gk * sizeof(uint16_t)));
            CK(cudaMallocHost(&ctx->h_gkey, gk * sizeof(uint16_t)));
            ctx->gkey_cap = gk;
        }
        for (int s = 0; s < 2; ++s)
            for (uint32_t g = 0; g < n_guides; ++g) {
                uint8_t patc[VS_GLEN];
                const uint8_t *gd = q.guides + (size_t)g * VS_GLEN;
                for (int i = 0; i < VS_GLEN; ++i) patc[i] = s ? (uint8_t)(3 - gd[VS_GLEN - 1 - i]) : gd[i];
                ctx->h_gkey[(size_t)s * n_guides + g] = (uint16_t)key_of_codes(s, patc);
            }
        if (!ctx->d_cls) CK(cudaMalloc(&ctx->d_cls, 2ull * BK_N * BK_CLS * sizeof(uint32_t)));
    }
    // hit buffer and guide super-chunks
    const double per_guide = (double)n_words * 32.0 * hit_density(k, pp.n);
    uint64_t want_hits = ctx->hit_cap_opt ? ctx->hit_cap_opt
                                          : std::min<uint64_t>(64ull << 20, std::max<uint64_t>(4ull << 20, (uint64_t)(per_guide * n_guides * 1.5) + 65536));
    auto ensure_hits = [&](uint64_t cap) -> int {
        if (cap <= ctx->hits_cap) return VS_OK;
        CK(cudaStreamSynchronize(st));
        cudaFree(ctx->d_hits); ctx->d_hits = nullptr; ctx->hits_cap = 0;
        CK(cudaMalloc(&ctx->d_hits, cap * sizeof(vs_hit)));
        ctx->hits_cap = cap;
        return VS_OK;
    };
    if ((r = ensure_hits(want_hits)) != VS_OK) return r;
    auto guides_per_pass = [&]() -> uint32_t {
        const double fit = per_guide > 0 ? (double)ctx->hits_cap / (per_guide * 1.5) : 1e30;
        uint64_t g = fit >= (double)n_guides ? n_guides : (uint64_t)std::max(1.0, fit);
        if (g > 32768) g = 32768;                            // the sort key holds 15 bits of guide index per delivery (and k_guide_classes 16)
        if (g < n_guides && g > SC_THREADS) g = g / SC_THREADS * SC_THREADS;
        return (uint32_t)g;
    };
    constexpr int EVC = 5;      // events per chunk
    while (ctx->ev_pool.size() < (size_t)EVC * n_chunks) {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        ctx->ev_pool.push_back(e);
    }
    // CTA size of k_score: one warp per 32 guides, at most SC_WARPS; a short tail (<= 8 guides) does not get a warp of its own
    // — it would idle most of the time and hold a warp slot (100 guides: 3 warps; the tail's 4-guide segments rotate over them)
    static const int fold_tail = getenv("VARSCOT_SCORE_FOLD_TAIL") ? atoi(getenv("VARSCOT_SCORE_FOLD_TAIL")) : 1;       // tuning knobs
    static const int rot_shift = getenv("VARSCOT_SCORE_ROT") ? atoi(getenv("VARSCOT_SCORE_ROT")) : 3;
    const auto score_cta = [](uint32_t ng) {
        if (ng >= (uint32_t)SC_THREADS) return (unsigned)SC_THREADS;
        const unsigned full = ng / 32, tail = ng % 32;
        return 32u * std::max(1u, full + ((tail > (fold_tail ? 8u : 0u) || full == 0) ? 1u : 0u));
    };
    unsigned score_ctas = (unsigned)ctx->n_sm * 32;         // persistent: a multiple of the SM count, about four waves of resident CTAs (16 / 32 / 64 per SM measured: 32 is 3 % faster than 16, 64 no better)
    if (const char *e = getenv("VARSCOT_SCORE_CTAS_PER_SM")) score_ctas = (unsigned)ctx->n_sm * (unsigned)std::max(1, atoi(e));   // tuning knob

    auto launch_extract = [&](uint32_t c) {
        const uint64_t c0 = plan[c], c1 = plan[c + 1];
        const unsigned tiles = (unsigned)((c1 - c0 + tile_words - 1) / tile_words);
        k_extract<<<tiles, EX_THREADS, 0, st>>>(ctx->d_bases, ctx->d_masks, c0, c1, tile_words, first_word * 32 - origin, pp,
                                                 ctx->d_planes[0], ctx->d_pos[0], ctx->d_planes[1], ctx->d_pos[1], ctx->blocks_cap, ctx->d_cnt);
        k_extract_mark<<<1, 32, 0, st>>>(ctx->d_cnt, d_rng + 4ull * c, d_all, ctx->d_planes[0], ctx->d_planes[1], ctx->blocks_cap);
        S.launches += 2;
    };
    auto launch_score = [&](const unsigned long long *rng, uint32_t g0, uint32_t ng) {
        ScoreArgs a;
        for (int s = 0; s < 2; ++s) { a.planes[s] = ctx->d_planes[s]; a.pos[s] = ctx->d_pos[s]; }
        a.rng = rng; a.cap = ctx->blocks_cap;
        a.n_guides = ng; a.guide_base = g0; a.pat_guides = n_guides; a.pat = ctx->d_pat;
        a.rot_shift = (uint32_t)rot_shift;
        a.hits = ctx->d_hits; a.n_hits = d_hitcnt; a.hit_cap = ctx->hits_cap;
        dispatch_score(k, a, score_ctas, score_cta(ng), st);
        S.launches++; S.score_launches++;
    };

    uint64_t total_out = 0;              // hits delivered so far (all super-chunks)
    bool out_overflow = false;
    uint32_t g0 = 0;
    bool first_pass = true;
    CK(cudaEventRecord(ctx->ev[0], st));
    CK(cudaMemcpyAsync(ctx->d_pat, ctx->h_pat, pat_entries * sizeof(uint16_t), cudaMemcpyHostToDevice, st));
    S.h2d_bytes += pat_entries * sizeof(uint16_t);
    const vs_text_view *source = src;
    bool derive_starts = false;
    while (g0 < n_guides) {
        uint32_t ng = std::min<uint32_t>(guides_per_pass(), n_guides - g0);
        uint64_t found = 0;
        for (int attempt = 0;; ++attempt) {
            if (attempt == 4) return fail(ctx, VS_ERR_CUDA, "vs_scan: device buffers still too small after regrowing");
            CK(cudaMemsetAsync(d_hitcnt, 0, sizeof(unsigned long long), st));
            if (ctx->idx_valid) {
                // the index is resident: one launch over the whole store
                CK(cudaEventRecord(ctx->ev[2], st));
                if (use_bk) {
                    const uint64_t need = 2ull * BK_N * ng;
                    if (need > ctx->perm_cap) {
                        CK(cudaStreamSynchronize(st));
                        cudaFree(ctx->d_perm); ctx->d_perm = nullptr; ctx->perm_cap = 0;
                        CK(cudaMalloc(&ctx->d_perm, need * sizeof(uint16_t)));
                        ctx->perm_cap = need;
                    }
                    // the keys of this pass's guides, strand by strand ([2][ng])
                    for (int s = 0; s < 2; ++s)
                        CK(cudaMemcpyAsync(ctx->d_gkey + (size_t)s * ng, ctx->h_gkey + (size_t)s * n_guides + g0, (size_t)ng * sizeof(uint16_t), cudaMemcpyHostToDevice, st));
                    S.h2d_bytes += 2ull * ng * sizeof(uint16_t);
                    k_guide_classes<<<dim3(BK_N, 2), 128, 0, st>>>(ctx->d_gkey, ng, pp, ctx->d_perm, ctx->d_cls);
                    BkScoreArgs b;
                    for (int s = 0; s < 2; ++s) { b.planes[s] = ctx->d_bk_planes[s]; b.pos[s] = ctx->d_bk_pos[s]; }
                    b.start = ctx->d_bk_ctl + 4 * BK_N;
                    b.n_guides = ng; b.guide_base = g0; b.pat_guides = n_guides; b.pat = ctx->d_pat;
                    b.perm = ctx->d_perm; b.cls = ctx->d_cls;
                    b.hits = ctx->d_hits; b.n_hits = d_hitcnt; b.hit_cap = ctx->hits_cap;
                    dispatch_score_bk(k, b, score_ctas, SC_THREADS, st);
                    S.launches += 2; S.score_launches++;
                } else {
                    launch_score(d_all, g0, ng);
                }
                CK(cudaEventRecord(ctx->ev[3], st));
                S.index_reused = first_pass && reuse ? (use_bk ? 2u : 1u) : S.index_reused;
            } else {
                CK(cudaMemsetAsync(ctx->d_cnt, 0, (4 + 4 * (ctx->cnt_chunks + 1) + 4) * sizeof(unsigned long long), st));
                CK(cudaEventRecord(ctx->ev[1], st));
                if (source) {
                    CK(cudaStreamWaitEvent(ctx->copy, ctx->ev[1], 0));
                    if ((r = begin_mask_source(ctx, source, n_words, ctx->ev[1])) != VS_OK) return abandon_upload(ctx, r);
                }
                uint64_t sparse_used = 0;
                for (uint32_t c = 0; c < n_chunks; ++c) {
                    cudaEvent_t *E = &ctx->ev_pool[(size_t)EVC * c];
                    if (source) {
                        cudaStream_t ready;
                        if ((r = enqueue_chunk_copy(ctx, source, first_word, plan[c], plan[c + 1], sparse_used, S.h2d_bytes, S.launches, ready)) != VS_OK)
                            return abandon_upload(ctx, r);
                        if (c + 1 == n_chunks && sp.usable && has_mask_source(source)) {
                            if ((r = enqueue_starts_from_plane(ctx, source, sp, first_word, n_words, origin, ctx->prep, S.launches)) != VS_OK) return abandon_upload(ctx, r);
                            derive_starts = true;
                            CK(cudaEventRecord(ctx->ev_starts, ctx->prep));
                        }
                        CK(cudaEventRecord(E[0], ready));
                        CK(cudaStreamWaitEvent(st, E[0], 0));
                    } else {
                        CK(cudaEventRecord(E[0], st));
                    }
                    CK(cudaEventRecord(E[1], st));
                    launch_extract(c);
                    CK(cudaEventRecord(E[2], st));
                    CK(cudaEventRecord(E[3], st));
                    launch_score(d_rng + 4ull * c, g0, ng);
                    CK(cudaEventRecord(E[4], st));
                }
                if (derive_starts) CK(cudaStreamWaitEvent(st, ctx->ev_starts, 0));
            }
            if (cudaGetLastError() != cudaSuccess) return abandon_upload(ctx, fail(ctx, VS_ERR_CUDA, "vs_scan: a kernel launch failed"));
            CK(cudaMemcpyAsync(ctx->h_cnt, ctx->d_cnt, cnt_words * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            if (cudaStreamSynchronize(st) != cudaSuccess) return abandon_upload(ctx, fail(ctx, VS_ERR_CUDA, std::string("vs_scan: ") + cudaGetErrorString(cudaGetLastError())));
            S.d2h_bytes += cnt_words * sizeof(unsigned long long);
            if (!ctx->idx_valid) {
                if (source) {                                // the text is resident from here on
                    if ((r = finish_contig_starts(ctx, source, sp, derive_starts, origin, S.h2d_bytes)) != VS_OK) return abandon_upload(ctx, r);
                    ctx->n_words = n_words; ctx->first_word = first_word; ctx->pos_origin = origin;
                    source = nullptr;
                }
                const uint64_t bf = ctx->h_cnt[2], br = ctx->h_cnt[3];
                if (std::max(bf, br) > ctx->blocks_cap) {    // the store overflowed (k_score skipped everything): regrow, extract again
                    uint64_t need = std::max(bf, br);
                    need = (need + need / 32 + 64ull * n_chunks + BLK_GROUP) / BLK_GROUP * BLK_GROUP;
                    if ((r = ensure_blocks(need)) != VS_OK) return r;
                    S.redo_chunks += n_chunks;
                    continue;
                }
                ctx->idx_valid = true; ctx->bk_valid = false; ctx->idx_pam = q.extra_pam; ctx->idx_chunks = n_chunks;
                ctx->idx_end[0] = bf; ctx->idx_end[1] = br;
                ctx->idx_cand[0] = ctx->h_cnt[0]; ctx->idx_cand[1] = ctx->h_cnt[1];
                ctx->idx_blocks[0] = 0; ctx->idx_blocks[1] = 0;
                for (uint32_t c = 0; c < n_chunks; ++c) { ctx->idx_blocks[0] += h_rng[4 * c + 2] - h_rng[4 * c]; ctx->idx_blocks[1] += h_rng[4 * c + 3] - h_rng[4 * c + 1]; }
                for (uint32_t c = 0; c < n_chunks; ++c) {
                    float a = 0.f, b = 0.f;
                    CK(cudaEventElapsedTime(&a, ctx->ev_pool[(size_t)EVC * c + 1], ctx->ev_pool[(size_t)EVC * c + 2]));
                    CK(cudaEventElapsedTime(&b, ctx->ev_pool[(size_t)EVC * c + 3], ctx->ev_pool[(size_t)EVC * c + 4]));
                    S.extract_ms += a; S.score_ms += b;
                }
                if (src) CK(cudaEventElapsedTime(&S.upload_ms, ctx->ev[1], ctx->ev_pool[(size_t)EVC * (n_chunks - 1)]));
            } else {
                float b = 0.f;
                CK(cudaEventElapsedTime(&b, ctx->ev[2], ctx->ev[3]));
                S.score_ms += b;
            }
            found = *h_hitcnt;
            if (found <= ctx->hits_cap) break;
            // device hit buffer too small: grow it (or halve the super-chunk once it is large) and repeat the pass over the index
            S.redo_chunks += n_chunks;
            if (found > (256ull << 20) && ng > 1) { ng = (ng + 1) / 2; continue; }
            if ((r = ensure_hits(found + found / 8 + 1024)) != VS_OK) return r;
        }
        S.guide_passes++;
        first_pass = false;
        // ---- deliver the super-chunk ----------------------------------------------------------------------
        CK(cudaEventRecord(ctx->ev[4], st));
        if (!q.resolved) {
            const uint64_t room = q.out_cap > total_out ? q.out_cap - total_out : 0, ncopy = std::min(found, room);
            if (q.out_raw && ncopy) CK(cudaMemcpyAsync(q.out_raw + total_out, ctx->d_hits, ncopy * sizeof(vs_hit), cudaMemcpyDeviceToHost, st));
            S.d2h_bytes += ncopy * sizeof(vs_hit);
            if (found > room) out_overflow = true;
        } else if (found) {
            if (found > ctx->loc_cap) {
                for (int s = 0; s < 2; ++s) { cudaFree(ctx->d_keys[s]); cudaFree(ctx->d_vals[s]); ctx->d_keys[s] = ctx->d_vals[s] = nullptr; }
                cudaFree(ctx->d_loc); ctx->d_loc = nullptr; ctx->loc_cap = 0;
                const uint64_t cap = std::max<uint64_t>(found + found / 8, 1u << 16);
                for (int s = 0; s < 2; ++s) { CK(cudaMalloc(&ctx->d_keys[s], cap * 8)); CK(cudaMalloc(&ctx->d_vals[s], cap * 8)); }
                CK(cudaMalloc(&ctx->d_loc, cap * sizeof(vs_loc_hit)));
                ctx->loc_cap = cap;
            }
            int guide_bits = 1;
            while ((1u << guide_bits) < ng) ++guide_bits;
            cub::DoubleBuffer<unsigned long long> dk(ctx->d_keys[0], ctx->d_keys[1]), dv(ctx->d_vals[0], ctx->d_vals[1]);
            size_t tmp = 0;
            CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp, dk, dv, (unsigned long long)found, 0, 49 + guide_bits, st));
            if (tmp > ctx->sort_tmp_bytes) {
                cudaFree(ctx->d_sort_tmp); ctx->d_sort_tmp = nullptr; ctx->sort_tmp_bytes = 0;
                CK(cudaMalloc(&ctx->d_sort_tmp, tmp + tmp / 4));
                ctx->sort_tmp_bytes = tmp + tmp / 4;
            }
            const unsigned gb = (unsigned)((found + 255) / 256);
            k_resolve_hits<<<gb, 256, 0, st>>>(ctx->d_hits, found, ctx->d_cstart, ctx->n_cstart, ctx->first_contig, g0, ctx->d_keys[0], ctx->d_vals[0]);
            tmp = ctx->sort_tmp_bytes;
            CK(cub::DeviceRadixSort::SortPairs(ctx->d_sort_tmp, tmp, dk, dv, (unsigned long long)found, 0, 49 + guide_bits, st));
            k_pack_loc_hits<<<gb, 256, 0, st>>>(dk.Current(), dv.Current(), found, ctx->d_loc);
            S.launches += 2 + 8;                              // + the radix sort's passes (CUB: histogram + one pass per 8 key bits)
            CK(cudaGetLastError());
            if (q.sink) {
                if (found > ctx->stage_cap) {
                    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
                    ctx->h_stage = nullptr; ctx->stage_cap = 0;
                    CK(cudaMallocHost(&ctx->h_stage, (found + found / 8) * sizeof(vs_loc_hit)));
                    ctx->stage_cap = found + found / 8;
                }
                CK(cudaMemcpyAsync(ctx->h_stage, ctx->d_loc, found * sizeof(vs_loc_hit), cudaMemcpyDeviceToHost, st));
                S.d2h_bytes += found * sizeof(vs_loc_hit);
            } else {
                const uint64_t room = q.out_cap > total_out ? q.out_cap - total_out : 0, ncopy = std::min(found, room);
                if (q.out_loc && ncopy) CK(cudaMemcpyAsync(q.out_loc + total_out, ctx->d_loc, ncopy * sizeof(vs_loc_hit), cudaMemcpyDeviceToHost, st));
                S.d2h_bytes += ncopy * sizeof(vs_loc_hit);
                if (found > room) out_overflow = true;
            }
        }
        CK(cudaEventRecord(ctx->ev[5], st));
        CK(cudaStreamSynchronize(st));
        { float a = 0.f; CK(cudaEventElapsedTime(&a, ctx->ev[4], ctx->ev[5])); S.resolve_ms += a; }
        if (q.resolved && q.sink && found) {
            if (q.sink(q.user, ctx->h_stage, found, g0, g0 + ng) != 0) return fail(ctx, VS_ERR_ARG, "vs_scan_resolved: the sink aborted the scan");
        }
        total_out += found;
        ctx->last_n_hits = found;                            // vs_scan_fetch serves the last super-chunk only (single-pass scans)
        g0 += ng;
    }
    CK(cudaEventRecord(ctx->ev[6], st));
    CK(cudaStreamSynchronize(st));
    CK(cudaEventElapsedTime(&S.total_ms, ctx->ev[0], ctx->ev[6]));
    S.n_cand_fwd = ctx->idx_cand[0]; S.n_cand_rev = ctx->idx_cand[1];
    S.n_blocks_fwd = ctx->idx_blocks[0]; S.n_blocks_rev = ctx->idx_blocks[1];
    S.n_hits = total_out;
    if (q.n_hits) *q.n_hits = total_out;
    if (!ctx->keep_index) { ctx->idx_valid = false; ctx->bk_valid = false; }
    if (q.stats) *q.stats = S;
    ctx->err.clear();
    if (out_overflow && !q.sink) {
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
    if (ctx->pos_origin) return fail(ctx, VS_ERR_ARG, LEGACY_BEYOND_4G);
    ScanReq q;
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
    ScanReq q;
    q.src = text; q.first_word = first_word; q.n_words = n_words;
    q.guides = guides; q.n_guides = n_guides; q.k = k; q.extra_pam = extra_pam;
    q.out_raw = out; q.out_cap = out_cap; q.n_hits = n_hits; q.stats = stats;
    return scan_engine(ctx, q);
}

extern "C" int vs_scan_resolved(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words,
                                const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                                vs_loc_hit *out, uint64_t out_cap, uint64_t *n_hits, vs_hit_sink sink, void *user, vs_scan_stats *stats)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_scan_resolved: ctx is NULL");
    if (text) {
        int r = check_view(ctx, text, first_word, n_words);
        if (r != VS_OK) return r;
    }
    ScanReq q;
    q.src = text; q.first_word = first_word; q.n_words = n_words;
    q.guides = guides; q.n_guides = n_guides; q.k = k; q.extra_pam = extra_pam;
    q.resolved = true; q.out_loc = out; q.out_cap = out_cap; q.n_hits = n_hits; q.sink = sink; q.user = user; q.stats = stats;
    return scan_engine(ctx, q);
}

extern "C" int vs_scan_fetch(vs_ctx *ctx, vs_hit *out, uint64_t out_cap, uint64_t *n_hits)
{
    if (!ctx) return fail(nullptr, VS_ERR_ARG, "vs_scan_fetch: ctx is NULL");
    if (ctx->pos_origin) return fail(ctx, VS_ERR_ARG, LEGACY_BEYOND_4G);
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
    uint32_t *d_out = nullptr;
    CK(cudaMalloc(&d_out, (size_t)grid * threads * sizeof(uint32_t)));
    cudaStream_t st = ctx->stream;
    float best_lop = 1e30f, best_lds = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        float ms = 0;
        CK(cudaEventRecord(ctx->ev[0], st));
        k_peak_lop3<<<grid, threads, 0, st>>>(d_out, iters);
        CK(cudaEventRecord(ctx->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
        if (rep && ms < best_lop) best_lop = ms;
        CK(cudaEventRecord(ctx->ev[0], st));
        k_peak_lds<<<grid, threads, 0, st>>>(d_out, iters);
        CK(cudaEventRecord(ctx->ev[1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
        if (rep && ms < best_lds) best_lds = ms;
    }
    CK(cudaGetLastError());
    cudaFree(d_out);
    const double nthreads = (double)grid * threads;
    if (lop3_per_s) *lop3_per_s = nthreads * iters * 64.0 / (best_lop * 1e-3);
    if (lds_words_per_s) *lds_words_per_s = nthreads * iters * 8.0 / (best_lds * 1e-3);
    return VS_OK;
}
