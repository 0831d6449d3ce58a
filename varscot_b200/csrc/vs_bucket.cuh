// varscot_b200/csrc/vs_bucket.cuh — the BUCKETED candidate index and the kernel that scores it (included by vs_kernels.cuh).
//
// Why: k_score is bound by the shared-memory pipe (one 32-bit word per lane, pattern position and candidate block:
// 19 LDS per 32-guide x 32-candidate tile at k = 6) and the alu pipe right behind it; the only way to go faster is
// to score fewer positions.  The candidates of a resident text are therefore regrouped by CONTENT: a bucket holds the
// candidates of one strand that share the PAM dinucleotide and the VS_KEYLEN - 2 bases next to it (VS_KEYLEN = 8, the default:
// six bases, window positions 15..22 on the forward pass, 0..7 on the reverse pass, 3 PAM kinds x 4096 buckets per strand;
// VS_KEYLEN = 6: four bases, positions 17..22 / 0..5, 3 x 256 buckets).  For a (bucket, guide) pair the mismatches c at
// those key positions are a constant, so
//   * the key positions are never loaded or counted,
//   * the remaining 23 - VS_KEYLEN positions are scored against the budget K' = K - c (K' < 0: the guide cannot hit in this
//     bucket at all — with six key bases and k = 6 that prunes every fifth pair of the GA buckets outright), and the
//     early-out test needs only PA'(K') = min(rest, 9 + 2 K') positions instead of PA(K) = 19: on uniform text E[c] = 4.5
//     (+ 1 in the buckets whose PAM differs from the guide's), i.e. 9..13 positions.
// The guides of a launch are sorted by c per bucket (k_guide_classes), the CTA that scores a batch of 32 blocks of the
// bucket walks the classes c = 0..K with the walk specialised on K'.  Everything else — block layout, expanded planes in
// shared memory, guide per lane, hit path, R4 — is k_score's; the reported mismatch count is count + c.
// The regrouping reads the PLAIN index (k_extract's output) and the resident text: it is built once per (text, PAM set)
// when a resident text is scanned repeatedly — the analogue of the reference building its FM index once
// (bidir_index.cpp:45-47) — and never on the streamed end-to-end path.
#pragma once

constexpr int BK_KINDS    = 3;                          // PAM kinds: GG, GA, -P XY (forward); their reverse complements (reverse)
constexpr int BK_KEYBITS  = 2 * (VS_KEYLEN - 2);        // key bits of the bases next to the PAM
constexpr int BK_PER_KIND = 1 << BK_KEYBITS;            // 256 (VS_KEYLEN 6) or 4096 (VS_KEYLEN 8) buckets per PAM kind
constexpr int BK_N        = BK_KINDS * BK_PER_KIND;     // buckets per strand
constexpr int BK_REST     = VS_GLEN - VS_KEYLEN;        // positions that are scored
constexpr int BK_PAD      = SC_NB * 32;                 // candidates per batch: a bucket is padded to whole batches
constexpr uint32_t BK_NOPOS = 0xFFFFFFFFu;              // padding slot of a bucket

// window position of key slot t of a strand; slots 0 .. VS_KEYLEN-3 are the bases next to the PAM, the last two the PAM itself
__host__ __device__ constexpr int key_position(int strand, int t)
{
    return strand ? (t < VS_KEYLEN - 2 ? 2 + t : t - (VS_KEYLEN - 2)) : VS_GLEN - VS_KEYLEN + t;
}
// key of a window / pattern: 2 bits (Dna code) per key slot, slot t at bits [2t, 2t+2)
__host__ __device__ inline uint32_t key_of_codes(int strand, const uint8_t *codes23)
{
    uint32_t k = 0;
    for (int t = 0; t < VS_KEYLEN; ++t) k |= (uint32_t)(codes23[key_position(strand, t)] & 3) << (2 * t);
    return k;
}
// bucket of a candidate key, or -1 if its PAM is none of the strand's kinds (cannot happen for an extracted candidate)
__host__ __device__ inline int bucket_of_key(int strand, uint32_t key, const PamParams &pp)
{
    const int x = (int)((key >> BK_KEYBITS) & 3), y = (int)((key >> (BK_KEYBITS + 2)) & 3);      // the PAM dinucleotide in window order
    for (int j = 0; j < pp.n; ++j)
        if (strand ? (x == pp.rx[j] && y == pp.ry[j]) : (x == pp.fx[j] && y == pp.fy[j])) return j * BK_PER_KIND + (int)(key & (BK_PER_KIND - 1));
    return -1;
}
// the key every candidate of a bucket has
__host__ __device__ inline uint32_t key_of_bucket(int strand, int bucket, const PamParams &pp)
{
    const int j = bucket / BK_PER_KIND;
    const uint32_t x = (uint32_t)(strand ? pp.rx[j] : pp.fx[j]), y = (uint32_t)(strand ? pp.ry[j] : pp.fy[j]);
    return (uint32_t)(bucket % BK_PER_KIND) | (x << BK_KEYBITS) | (y << (BK_KEYBITS + 2));
}
// mismatches between two keys (2 bits per position)
__host__ __device__ inline uint32_t key_mismatches(uint32_t a, uint32_t b)
{
    const uint32_t x = a ^ b, m = (x | (x >> 1)) & 0x5555u;
#if defined(__CUDA_ARCH__) && !defined(VS_HOST_UNIT_TEST)
    return (uint32_t)__popc(m);
#else
    return (uint32_t)__builtin_popcount(m);
#endif
}

// ---- index build ---------------------------------------------------------------------------------------------------
// the 32 candidate keys of one plain block, from its 2 x VS_KEYLEN key plane words (bit c of word = candidate c): a 32 x 32
// register transpose of which 12 / 16 rows are used
__device__ __forceinline__ void block_keys(const uint32_t *__restrict__ planes, uint64_t blk, int strand, uint32_t (&key)[32])
{
    const uint32_t *src = planes + plane_index(blk, 0);
#pragma unroll
    for (int i = 0; i < 32; ++i) key[i] = 0u;
#pragma unroll
    for (int t = 0; t < VS_KEYLEN; ++t) {
        const int p = key_position(strand, t);
        key[2 * t] = __ldg(src + (VS_GLEN + p) * BLK_GROUP);        // lo plane -> bit 2t
        key[2 * t + 1] = __ldg(src + p * BLK_GROUP);                // hi plane -> bit 2t + 1
    }
    transpose32(key);                                               // key[c] = the key of candidate c
}

#ifndef VS_HOST_UNIT_TEST
#define VS_BK_SMEM(name) extern __shared__ __align__(16) uint32_t vs_bk_dyn_smem[]; uint32_t *name = vs_bk_dyn_smem
#else
#define VS_BK_SMEM(name) static uint32_t name[BK_N]
#endif
constexpr int BK_HIST_SMEM = BK_N * 4;           // dynamic shared memory of k_bucket_hist / k_bucket_scatter
constexpr int BKB_THREADS = 256;                 // plain blocks per CTA of the histogram / scatter kernels (8192 candidates)

// k_bucket_hist: candidates per bucket.  grid.y = strand; one thread per plain block; CTA histogram in shared memory, then
// one global atomic per non-empty bin.  n_blocks[2] = blocks of the plain store per strand (device).
__global__ void __launch_bounds__(BKB_THREADS)
k_bucket_hist(const uint32_t *__restrict__ planes_f, const uint32_t *__restrict__ planes_r, const unsigned long long *__restrict__ rng_all,
              PamParams pp, unsigned long long *__restrict__ hist)
{
    VS_BK_SMEM(h);                                // uint32_t h[BK_N]: dynamic shared memory (48 KB for VS_KEYLEN 8)
    const int strand = blockIdx.y;
    const unsigned long long n_blocks = rng_all[2 + strand];
    const unsigned long long cta0 = (unsigned long long)blockIdx.x * BKB_THREADS;
    if (cta0 >= n_blocks) return;
    for (int i = threadIdx.x; i < BK_N; i += BKB_THREADS) h[i] = 0u;
    __syncthreads();
    const unsigned long long blk = cta0 + threadIdx.x;
    if (blk < n_blocks) {
        const uint32_t *planes = strand ? planes_r : planes_f;
        const uint32_t valid = __ldg(planes + plane_index(blk, BLK_VALID));
        if (valid) {
            uint32_t key[32];
            block_keys(planes, blk, strand, key);
#pragma unroll
            for (int c = 0; c < 32; ++c)
                if ((valid >> c) & 1u) {
                    const int b = bucket_of_key(strand, key[c], pp);
                    if (b >= 0) atomicAdd(&h[b], 1u);
                }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BK_N; i += BKB_THREADS)
        if (h[i]) atomicAdd(&hist[strand * BK_N + i], (unsigned long long)h[i]);
}

// k_bucket_scan (one CTA per strand, grid = 2): pads every bucket to whole batches, turns the counts into
//   start[s][b]  first BLOCK of bucket b in the bucketed store (start[s][BK_N] = total blocks), and
//   cursor[s][b] next free CANDIDATE slot of the bucket (= 32 * start), advanced by k_bucket_scatter.
__global__ void __launch_bounds__(1024)
k_bucket_scan(const unsigned long long *__restrict__ hist, unsigned long long *__restrict__ start, unsigned long long *__restrict__ cursor)
{
    __shared__ unsigned long long part[1024];
    const int s = blockIdx.x;
    constexpr int PER = (BK_N + 1023) / 1024;
    const int t0 = (int)threadIdx.x * PER, b0 = t0 < BK_N ? t0 : BK_N, b1 = b0 + PER < BK_N ? b0 + PER : BK_N;
    unsigned long long sum = 0;
    for (int b = b0; b < b1; ++b) sum += (hist[s * BK_N + b] + BK_PAD - 1) / BK_PAD * (BK_PAD / 32);
    part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int i = 0; i < 1024; ++i) { const unsigned long long v = part[i]; part[i] = run; run += v; }
        start[s * (BK_N + 1) + BK_N] = run;
    }
    __syncthreads();
    unsigned long long run = part[threadIdx.x];
    for (int b = b0; b < b1; ++b) {
        start[s * (BK_N + 1) + b] = run;
        cursor[s * BK_N + b] = run * 32;
        run += (hist[s * BK_N + b] + BK_PAD - 1) / BK_PAD * (BK_PAD / 32);
    }
}

// k_bucket_scatter: the positions of the plain index, regrouped by bucket.  Same traversal as k_bucket_hist; a CTA claims
// one range per non-empty bucket (one global atomic each) and its candidates take consecutive slots of it.  Slots that
// nobody writes (the padding of a bucket) keep BK_NOPOS (the array is pre-filled).
__global__ void __launch_bounds__(BKB_THREADS)
k_bucket_scatter(const uint32_t *__restrict__ planes_f, const uint32_t *__restrict__ planes_r, const uint32_t *__restrict__ pos_f,
                 const uint32_t *__restrict__ pos_r, const unsigned long long *__restrict__ rng_all, PamParams pp,
                 unsigned long long *__restrict__ cursor, uint32_t *__restrict__ out_f, uint32_t *__restrict__ out_r, uint64_t cap_f, uint64_t cap_r)
{
    VS_BK_SMEM(h);                                // uint32_t h[BK_N]: first the CTA's count per bucket, then the first slot of its range (slots fit 32 bits: a shard holds < 4 G bases)
    const int strand = blockIdx.y;
    const unsigned long long n_blocks = rng_all[2 + strand];
    const unsigned long long cta0 = (unsigned long long)blockIdx.x * BKB_THREADS;
    if (cta0 >= n_blocks) return;
    for (int i = threadIdx.x; i < BK_N; i += BKB_THREADS) h[i] = 0u;
    __syncthreads();
    const unsigned long long blk = cta0 + threadIdx.x;
    const uint32_t *planes = strand ? planes_r : planes_f;
    uint32_t valid = 0;
    uint32_t key[32];
    if (blk < n_blocks) valid = __ldg(planes + plane_index(blk, BLK_VALID));
    if (valid) {
        block_keys(planes, blk, strand, key);
#pragma unroll
        for (int c = 0; c < 32; ++c)
            if ((valid >> c) & 1u) {
                const int b = bucket_of_key(strand, key[c], pp);
                key[c] = b >= 0 ? ((uint32_t)b << 16) | atomicAdd(&h[b], 1u) : BK_NOPOS;        // bucket and rank inside the CTA's range
            }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BK_N; i += BKB_THREADS)
        if (h[i]) h[i] = (uint32_t)atomicAdd(&cursor[strand * BK_N + i], (unsigned long long)h[i]);
    __syncthreads();
    if (valid) {
        const uint32_t *pos = (strand ? pos_r : pos_f) + blk * 32;
        uint32_t *out = strand ? out_r : out_f;
        const uint64_t out_cap = strand ? cap_r : cap_f;
#pragma unroll
        for (int c = 0; c < 32; ++c)
            if (((valid >> c) & 1u) && key[c] != BK_NOPOS) {
                const unsigned long long slot = (unsigned long long)h[key[c] >> 16] + (key[c] & 0xFFFFu);
                if (slot < out_cap) out[slot] = __ldg(pos + c);
            }
    }
}

// k_bucket_gather: one thread per block of the bucketed store: the 23-base windows of its 32 positions are gathered from
// the resident text (funnel shifts over two words of each plane), transposed to the bit-sliced block layout of k_extract
// (48 words at plane_index) and written; padding slots get an empty valid bit.  first_base = position of the shard's word 0
// relative to the shard's origin, as the positions in `pos`.
__global__ void __launch_bounds__(64)
k_bucket_gather(const vs_bases *__restrict__ B, const vs_masks *__restrict__ M, uint64_t first_base, const uint32_t *__restrict__ pos,
                unsigned long long n_blocks, uint32_t *__restrict__ planes)
{
    const unsigned long long blk = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (blk >= n_blocks) return;
    uint32_t ah[32], al[32];
    uint32_t lastw = 0, valid = 0;
    const uint4 *p4 = reinterpret_cast<const uint4 *>(pos + blk * 32);
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
        const uint4 q = p4[c4];
        const uint32_t pp4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = c4 * 4 + u;
            const uint32_t p = pp4[u];
            if (p == BK_NOPOS) { ah[c] = 0u; al[c] = 0u; continue; }
            const uint64_t local = (uint64_t)p - first_base;
            const uint64_t w = local >> 5;
            const uint32_t b = (uint32_t)(local & 31);
            const vs_bases x = B[w], y = B[w + 1];
            ah[c] = __funnelshift_r(x.hi, y.hi, b) & 0x7FFFFFu;
            al[c] = __funnelshift_r(x.lo, y.lo, b) & 0x7FFFFFu;
            lastw |= ((M[w].lw >> b) & 1u) << c;
            valid |= 1u << c;
        }
    }
    uint32_t *pl_out = planes + plane_index(blk, 0);
    transpose32(ah);
#pragma unroll
    for (int i = 0; i < VS_GLEN; ++i) pl_out[i * BLK_GROUP] = ah[i];
    transpose32(al);
#pragma unroll
    for (int i = 0; i < VS_GLEN; ++i) pl_out[(VS_GLEN + i) * BLK_GROUP] = al[i];
    pl_out[BLK_LAST * BLK_GROUP] = lastw;
    pl_out[BLK_VALID * BLK_GROUP] = valid;
}

// ---- guide classes -----------------------------------------------------------------------------------------------
// k_guide_classes: for every (strand, bucket) the guides of the launch sorted by c = mismatches between the guide's key and
// the bucket's (a counting sort: VS_KEYLEN + 1 bins), as perm[strand][bucket][n_guides] (uint16 guide index) and the class starts
// cls[strand][bucket][VS_KEYLEN + 2] (cls[c] = first entry with c mismatches; cls[VS_KEYLEN + 1] = n_guides).  gkey[strand][g]
// = 2 * VS_KEYLEN-bit key of the pattern the strand's pass scores.  grid = (BK_N, 2), any CTA size; guides beyond 65535 per launch are
// not supported (the host splits the launch).
constexpr int BK_CLS = VS_KEYLEN + 2;
__global__ void __launch_bounds__(128)
k_guide_classes(const uint16_t *__restrict__ gkey, uint32_t n_guides, PamParams pp, uint16_t *__restrict__ perm, uint32_t *__restrict__ cls)
{
    __shared__ uint32_t cnt[BK_CLS], at[BK_CLS];
    const int bucket = blockIdx.x, strand = blockIdx.y;
    if (bucket / BK_PER_KIND >= pp.n) return;
    const uint32_t bkey = key_of_bucket(strand, bucket, pp);
    const uint16_t *gk = gkey + (size_t)strand * n_guides;
    if (threadIdx.x < BK_CLS) cnt[threadIdx.x] = 0u;
    __syncthreads();
    for (uint32_t g = threadIdx.x; g < n_guides; g += blockDim.x) atomicAdd(&cnt[key_mismatches(gk[g], bkey)], 1u);
    __syncthreads();
    uint32_t *c_out = cls + ((size_t)strand * BK_N + bucket) * BK_CLS;
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int c = 0; c <= VS_KEYLEN; ++c) { at[c] = run; c_out[c] = run; run += cnt[c]; }
        c_out[VS_KEYLEN + 1] = run;
    }
    __syncthreads();
    uint16_t *p_out = perm + ((size_t)strand * BK_N + bucket) * n_guides;
    // (the order inside a class is whatever the atomics give: every guide of a class is scored the same way)
    for (uint32_t g = threadIdx.x; g < n_guides; g += blockDim.x) p_out[atomicAdd(&at[key_mismatches(gk[g], bkey)], 1u)] = (uint16_t)g;
}

// ---- scoring -------------------------------------------------------------------------------------------------------
// slot order of the bucketed walk = the plain one (slot_position): its first BK_REST slots are exactly the positions
// outside the key on both strands.
// stage-A slots for the budget kp: two more than k_score's 7 + 2 k — here an iteration that survives stage A is rescanned by a
// routine of ~100 instructions instead of four more LDS, so it must be ten times rarer (about 1 % of the iterations)
__host__ __device__ constexpr int bk_walk_slots(int kp) { return 9 + 2 * kp < BK_REST ? 9 + 2 * kp : BK_REST; }
// The walks are specialised on the number of stage-A slots only — 9, 11, 13, 15 (VS_KEYLEN 6: also 17) — not on the budget: the budgets
// that share the longest walk share its code and pick their threshold at run time.  The instruction cache decides this: every
// batch runs every class, the SM's instruction cache holds 32 KB, and the first version of this kernel (one walk per budget
// and segment shape, unrolled 4 times with the rare path inlined: 130 KB) spent 17 of 18 issue cycles waiting for instructions.

// count <= kp for a warp-uniform budget kp in [LO, HI]
template <int LO, int HI>
__device__ __forceinline__ uint32_t le_runtime(const uint32_t (&b)[5], int kp)
{
    if constexpr (LO == HI) return le_k<LO>(b);
    else return kp == LO ? le_k<LO>(b) : le_runtime<LO + 1, HI>(b, kp);
}

// ---- the deal of a batch's segments to the CTA's warps ------------------------------------------------------------
// A batch is scored by the CTA's warps between two barriers, so it lasts as long as its most loaded warp.  Its work is, per
// class c = 0 .. min(K, VS_KEYLEN), one segment per 32 guides of the class and its tail in 4-guide segments (a 4-guide segment
// walks 8 blocks per iteration, so a class costs 32 * n / 32 iterations however it is cut).  At 100 guides a bucket's classes
// hold one 32-guide segment and a dozen or more 4-guide ones: dealt round robin by count, the warp that drew the 32-guide
// segment also drew its share of the small ones while the three others waited at the barrier for a third of the batch.
// The segments are therefore dealt longest first, each to the warp with the least cost dealt so far (LPT list scheduling:
// the most loaded warp carries at most 4/3 of the optimum).
// Cost of one segment in issue slots: set-up (perm and pattern loads, slot addresses) plus, per iteration, the walk's
// stage-A loads, its carry-save adder tree (2 LOP3 per adder, pa - popc(pa) adders), threshold, vote and half an address
// update per slot.  Only the ratios matter.
constexpr uint32_t BK_SEG_SETUP = 60;
__host__ __device__ inline uint32_t bk_segment_cost(int kp, uint32_t iters)
{
    const uint32_t pa = (uint32_t)bk_walk_slots(kp);
#if defined(__CUDA_ARCH__) && !defined(VS_HOST_UNIT_TEST)
    const uint32_t adders = pa - (uint32_t)__popc(pa);
#else
    const uint32_t adders = pa - (uint32_t)__builtin_popcount(pa);
#endif
    return BK_SEG_SETUP + iters * ((3u * pa) / 2u + 2u * adders + 4u);
}
// bk_deal: the deal of the segments of a bucket (class starts cls[0 .. BK_CLS)) to `warps` (<= SC_WARPS) warps, as RUNS: calls
// emit(v, at, nseg, c, L, last) once per run — nseg consecutive segments of 2^L guide lanes (L = 5: 32 guides, L = 2: 4 guides)
// of class c dealt to warp v, the first at perm entry `at`, the next 2^L entries further each, every one full but the last,
// which holds `last` guides.  Order: the 32-guide segments by class, then the 4-guide ones by class (c ascending = stage-A
// slots descending, so the cost never increases); ties go to the lowest warp.  The segments of one (class, shape) cost the
// same, so what the greedy decides for them is how many each warp gets: a warp takes a contiguous run of them, and a warp
// holds at most BK_RUNS runs.  It depends on the bucket only: k_score_bucketed computes it when its batches enter a new
// bucket (about 47 batches per bucket at 3.5 Gbases) and rotates the warps per batch.
constexpr int BK_RUNS = 2 * (VS_KEYLEN + 1);
template <int K, class F>
__host__ __device__ __forceinline__ void bk_deal(const uint32_t *cls, uint32_t warps, F &&emit)
{
    constexpr uint32_t CMAX = (uint32_t)(K < VS_KEYLEN ? K : VS_KEYLEN);   // a guide with c > K cannot hit in this bucket
    uint32_t load[SC_WARPS];                                               // cost dealt so far per warp
#pragma unroll
    for (int v = 0; v < SC_WARPS; ++v) load[v] = 0u;
#pragma unroll 1
    for (uint32_t pass = 0; pass < 2u; ++pass) {
#pragma unroll 1
        for (uint32_t c = 0; c <= CMAX; ++c) {
            const uint32_t c0 = cls[c], n = cls[c + 1] - c0, nfull = n & ~31u;
            const uint32_t L = pass ? 2u : 5u, base = pass ? nfull : 0u, units = pass ? (n - nfull + 3u) >> 2 : nfull >> 5;
            const uint32_t cost = bk_segment_cost(K - (int)c, pass ? 4u : 32u);
            uint32_t cnt[SC_WARPS];
#pragma unroll
            for (int v = 0; v < SC_WARPS; ++v) cnt[v] = 0u;
#pragma unroll 1
            for (uint32_t u = 0; u < units; ++u) {
                uint32_t best = 0u, least = load[0];
#pragma unroll
                for (uint32_t v = 1; v < (uint32_t)SC_WARPS; ++v)
                    if (v < warps && load[v] < least) { best = v; least = load[v]; }
#pragma unroll
                for (uint32_t v = 0; v < (uint32_t)SC_WARPS; ++v)
                    if (v == best) { load[v] += cost; ++cnt[v]; }
            }
            uint32_t i = base;
#pragma unroll
            for (uint32_t v = 0; v < (uint32_t)SC_WARPS; ++v)
                if (cnt[v]) {
                    const uint32_t end = i + (cnt[v] << L);
                    emit(v, c0 + i, cnt[v], c, L, min(1u << L, n - (end - (1u << L))));
                    i = end;
                }
        }
    }
}

struct BkScoreArgs {
    const uint32_t *planes[2];  // bucketed store per strand
    const uint32_t *pos[2];     // bucketed positions per strand
    const unsigned long long *start;    // [2][BK_N + 1] first block of every bucket (device)
    uint32_t n_guides, guide_base, pat_guides;
    const uint16_t *pat;        // pattern table as in ScoreArgs
    const uint16_t *perm;       // [2][BK_N][n_guides]
    const uint32_t *cls;        // [2][BK_N][BK_CLS]
    vs_hit *hits;
    unsigned long long *n_hits;
    uint64_t hit_cap;
};

// Rare path, ONE copy per kernel and nothing of the walk's register state: the walk only notes in `pend` which of its
// iterations had a lane within budget after stage A; afterwards this routine rescans those block rows exactly — every lane
// counts all scored slots of its guide (carry-save adder tree), compares with the budget, and appends its hits (count + c,
// R4 on last windows).  ~100 instructions per noted iteration, about 1 % of the iterations.
template <int K>
__device__ VS_COLD void bk_cold(const char *row0, uint32_t step_bytes, uint32_t pend, uint32_t step, uint32_t sub, const uint16_t *po, int kp, uint32_t c,
                                int strand, bool real, const uint32_t *lastm_s, const uint32_t *posb, uint32_t info, vs_hit *hits,
                                unsigned long long *n_hits, uint64_t hit_cap)
{
    const uint32_t zero5[5] = {0u, 0u, 0u, 0u, 0u};
    uint32_t off[BK_REST];
#pragma unroll
    for (int s = 0; s < BK_REST; ++s) off[s] = po[s];
    while (pend != 0) {
        const uint32_t it = (uint32_t)__ffs(pend) - 1u;
        pend &= pend - 1u;
        const char *row = row0 + it * step_bytes;
        uint32_t m[BK_REST], cnt[5];
#pragma unroll
        for (int s = 0; s < BK_REST; ++s) m[s] = *reinterpret_cast<const uint32_t *>(row + off[s]);
        popcount_planes<BK_REST, false>(m, zero5, cnt);
        // count <= kp, most significant bit first
        uint32_t gt = 0u, eq = ~0u;
#pragma unroll
        for (int w = 4; w >= 0; --w) {
            const uint32_t kb = ((kp >> w) & 1) ? ~0u : 0u;
            gt |= eq & cnt[w] & ~kb;
            eq &= ~(cnt[w] ^ kb);
        }
        const uint32_t le = ~gt;
        const uint32_t j = it * step + sub;
        if (le != 0 && real) score_hits_body<K>(row, po, strand, le, cnt, c, lastm_s[j], posb + (size_t)j * 32, info, hits, n_hits, hit_cap);
    }
}

template <int K>
__global__ void __launch_bounds__(SC_THREADS, score_min_blocks(K))
k_score_bucketed(BkScoreArgs a)
{
#ifndef VS_HOST_UNIT_TEST
    extern __shared__ __align__(16) uint32_t sm[];     // as k_score: planes, last-window masks, raw staging
#endif
    constexpr uint32_t ROW = SC_STRIDE * 4u;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned long long nbat_f = a.start[BK_N] / SC_NB, nbat = nbat_f + a.start[(BK_N + 1) + BK_N] / SC_NB;
    uint32_t *lastm_s = sm + SC_NB * SC_STRIDE;
    uint32_t *raw_s = lastm_s + SC_NB;
    const uint32_t zero5[5] = {0u, 0u, 0u, 0u, 0u};
    // every CTA takes a CONTIGUOUS run of batches: consecutive batches mostly belong to the same bucket
    const unsigned long long per = (nbat + gridDim.x - 1) / gridDim.x, bat0 = per * blockIdx.x, bat1 = min(nbat, bat0 + per);
    auto stage = [&](unsigned long long bat) {
        const uint32_t strand = bat >= nbat_f;
        const unsigned long long blk0 = (bat - (strand ? nbat_f : 0ull)) * SC_NB;
        const uint32_t *src = (strand ? a.planes[1] : a.planes[0]) + plane_index(blk0, 0);
#ifndef VS_HOST_UNIT_TEST
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(raw_s);
        for (uint32_t o = tid * 16u; o < BLK_WORDS * SC_NB * 4u; o += blockDim.x * 16u)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + o), "l"(reinterpret_cast<const char *>(src) + o));
        asm volatile("cp.async.commit_group;" ::: "memory");
#else
        for (uint32_t i = tid; i < BLK_WORDS * SC_NB; i += blockDim.x) raw_s[i] = src[i];
#endif
    };
    if (bat0 < bat1) stage(bat0);
    const uint32_t warps = blockDim.x >> 5;
    int bucket = -1, bucket_strand = -1;
    __shared__ uint2 runs_s[SC_WARPS][SC_WARPS][BK_RUNS];   // per warp: the current bucket's deal, BK_RUNS runs per dealt warp
    __shared__ uint32_t nrun_s[SC_WARPS][SC_WARPS];
    int deal_bucket = -1, deal_strand = -1;
    for (unsigned long long bat = bat0; bat < bat1; ++bat) {
    const uint32_t strand = bat >= nbat_f;
    const unsigned long long blk0 = (bat - (strand ? nbat_f : 0ull)) * SC_NB;
    const unsigned long long *st = a.start + (size_t)strand * (BK_N + 1);
    if (bucket_strand != (int)strand || blk0 >= st[bucket + 1]) {     // the batch's bucket: last one whose first block is <= blk0
        int lo = 0, hi = BK_N;                                         // invariant: st[lo] <= blk0 < st[hi]
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (st[mid] <= blk0) lo = mid; else hi = mid; }
        bucket = lo; bucket_strand = (int)strand;
    }
#ifndef VS_HOST_UNIT_TEST
    asm volatile("cp.async.wait_group 0;" ::: "memory");
#endif
    __syncthreads();
    if (deal_bucket != bucket || deal_strand != (int)strand) {
        // the bucket's deal, computed by every lane and kept by its warp in shared memory (each warp writes and reads only its
        // own copy; its lanes write the same values): recomputed when the batches enter a new bucket
        uint32_t nr[SC_WARPS];
#pragma unroll
        for (int u = 0; u < SC_WARPS; ++u) nr[u] = 0u;
        bk_deal<K>(a.cls + ((size_t)strand * BK_N + bucket) * BK_CLS, warps,
                   [&](uint32_t v, uint32_t at, uint32_t nseg, uint32_t c, uint32_t L, uint32_t last) {
#pragma unroll
                       for (uint32_t u = 0; u < (uint32_t)SC_WARPS; ++u)
                           if (u == v) runs_s[wid][u][nr[u]++] = uint2{at, nseg | (c << 16) | (L << 20) | (last << 24)};
                   });
#pragma unroll
        for (int u = 0; u < SC_WARPS; ++u) nrun_s[wid][u] = nr[u];
        deal_bucket = bucket; deal_strand = (int)strand;
    }
    {
        const uint32_t b = (uint32_t)lane;
        const uint32_t inv = ~raw_s[BLK_VALID * SC_NB + b];
        for (int p = wid; p < VS_GLEN; p += (int)warps) {
            const uint32_t h = raw_s[p * SC_NB + b], l = raw_s[(VS_GLEN + p) * SC_NB + b];
            *reinterpret_cast<uint4 *>(sm + b * SC_STRIDE + 4 * p) =
                make_uint4((h | l) | inv, (h | ~l) | inv, (~h | l) | inv, (~h | ~l) | inv);
        }
        if (wid == 0) lastm_s[b] = raw_s[BLK_LAST * SC_NB + b];
    }
    __syncthreads();
    if (bat + 1 < bat1) stage(bat + 1);
    const uint16_t *pat0 = a.pat + ((size_t)strand * a.pat_guides + a.guide_base) * PAT_STRIDE;
    const uint32_t *posb = (strand ? a.pos[1] : a.pos[0]) + blk0 * 32;
    const uint16_t *perm = a.perm + ((size_t)strand * BK_N + bucket) * a.n_guides;

    // The walk of one segment, stage A only: PA slots per iteration, (32 >> L) blocks per iteration.  Iterations in which some
    // lane is still within budget are noted in the returned mask and rescanned by bk_cold afterwards.  One copy of this code
    // per (PA, L) — 4 or 5 slot counts x {32-guide, 4-guide} segments — and nothing else inside: the kernel's hot code must
    // fit the SM's 32 KB instruction cache, every batch runs every variant.
    auto walk = [&](const char *(&adr)[BK_REST], int kp, auto pa_c, auto klo_c, auto khi_c, auto l_c) -> uint32_t {
        constexpr int PA = decltype(pa_c)::value, KLO = decltype(klo_c)::value, KHI = decltype(khi_c)::value;
        constexpr uint32_t L = decltype(l_c)::value, STEP = 32u >> L, UNR = 2u;
        uint32_t pend = 0u;
#pragma unroll 1
        for (uint32_t j0 = 0; j0 < (uint32_t)SC_NB; j0 += STEP * UNR) {
#pragma unroll
            for (uint32_t u = 0; u < UNR; ++u) {
                uint32_t m[PA], ca[5];
#pragma unroll
                for (int i = 0; i < PA; ++i) m[i] = *reinterpret_cast<const uint32_t *>(adr[i] + u * STEP * ROW);
                popcount_planes<PA, false>(m, zero5, ca);
                const uint32_t le = le_runtime<KLO, KHI>(ca, kp);
                if (__any_sync(0xffffffffu, le != 0)) pend |= 1u << (j0 / STEP + u);
            }
#pragma unroll
            for (int i = 0; i < PA; ++i) adr[i] += STEP * UNR * ROW;
        }
        return pend;
    };
    // one segment: guides perm[at .. at + GW) (GW = 32 or 4) of the class with c key mismatches, budget kp = K - c for the
    // other positions
    auto segment = [&](uint32_t at, uint32_t n_real, uint32_t c, uint32_t L) {
        const int kp = K - (int)c;
        const uint32_t gw = 1u << L, sub = (uint32_t)lane >> L, gl = (uint32_t)lane & (gw - 1u), step = 32u >> L;
        const bool real = gl < n_real;                     // padding lanes score the segment's first guide; their hits are dropped
        const uint32_t g = perm[at + (real ? gl : 0u)];
        const uint16_t *po = pat0 + (size_t)g * PAT_STRIDE;
        const char *smb = reinterpret_cast<const char *>(sm) + sub * ROW;
        const char *adr[BK_REST];
        {
            const uint4 *q = reinterpret_cast<const uint4 *>(po);
            uint32_t w[12];
#pragma unroll
            for (int i = 0; i < 3; ++i) { const uint4 v = q[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
#pragma unroll
            for (int i = 0; i < BK_REST; ++i) adr[i] = smb + ((w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu);
        }
        uint32_t pend = 0u;
        const int pa = bk_walk_slots(kp);
        auto go = [&](auto l_c) {
            // 9 / 11 / 13 (/ 15) slots for the budgets 0 / 1 / 2 (/ 3), every scored position (one stage, exact) for the budgets above
            using I0 = std::integral_constant<int, 0>;
            if (pa == BK_REST) {
                constexpr int KLO = (BK_REST - 9) / 2 < K ? (BK_REST - 9) / 2 : K;
                pend = walk(adr, kp, std::integral_constant<int, BK_REST>{}, std::integral_constant<int, KLO>{}, std::integral_constant<int, K>{}, l_c);
            } else if (pa == 9) pend = walk(adr, kp, std::integral_constant<int, 9>{}, I0{}, I0{}, l_c);
            else if (pa == 11) { if constexpr (K >= 1) pend = walk(adr, kp, std::integral_constant<int, 11>{}, std::integral_constant<int, 1>{}, std::integral_constant<int, 1>{}, l_c); }
            else if (pa == 13) { if constexpr (K >= 2) pend = walk(adr, kp, std::integral_constant<int, 13>{}, std::integral_constant<int, 2>{}, std::integral_constant<int, 2>{}, l_c); }
            else { if constexpr (K >= 3 && BK_REST > 15) pend = walk(adr, kp, std::integral_constant<int, 15>{}, std::integral_constant<int, 3>{}, std::integral_constant<int, 3>{}, l_c); }
        };
        if (L == 5u) go(std::integral_constant<uint32_t, 5>{}); else go(std::integral_constant<uint32_t, 2>{});
        if (pend) bk_cold<K>(smb, step * ROW, pend, step, sub, po, kp, c, (int)strand, real, lastm_s, posb,
                             ((a.guide_base + g) << 8) | (strand << 7), a.hits, a.n_hits, a.hit_cap);
    };
    // the segments of the batch: the bucket's deal (bk_deal), its warps rotated by one for every batch and CTA so that no warp
    // (and SM sub-partition) keeps the heavy share
    const uint32_t v = (uint32_t)(wid + bat + blockIdx.x) % warps;
    const uint32_t nrun = nrun_s[wid][v];
#pragma unroll 1
    for (uint32_t r = 0; r < nrun; ++r) {
        const uint2 e = runs_s[wid][v][r];
        const uint32_t nseg = e.y & 0xFFFFu, c = (e.y >> 16) & 0xFu, L = (e.y >> 20) & 0xFu, last = e.y >> 24;
#pragma unroll 1
        for (uint32_t j = 0; j < nseg; ++j) segment(e.x + (j << L), j + 1u < nseg ? 1u << L : last, c, L);
    }
    }
}
