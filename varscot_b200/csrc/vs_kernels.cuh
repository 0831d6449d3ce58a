// varscot_b200/csrc/vs_kernels.cuh — hand-written sm_100a kernels of the off-target scan.
//
// What they replace: the inner loops of VARSCOT_pipeline/read_mapping/bidir_mapping.cpp —
// SeqAn's find<0,K>(delegate, index, half, HammingDistance()) (:129-146) plus the verify
// delegate (:34-127) — restated as a dense, PAM-first Hamming scan (rules R1-R4 of SURVEY.md 8a).
//
// Pipeline per scan, per pipeline chunk of the text (8 Mi words), all on one stream:
//   k_extract  : per tile of ~240 words (7680 window starts), find the PAM-valid / scannable windows of each strand
//                (bit-parallel on the packed planes and the precomputed window masks), compact them into blocks of 32
//                candidates and store each block bit-sliced ACROSS candidates (per-thread 32x32 register
//                transposes): 48 words per block = hi_0..hi_22, lo_0..lo_22, last-window mask, valid mask; + 32 positions
//   k_score<K> : one thread per candidate block, both strands in one launch; the 46 planes are expanded into 92
//                "mismatch if the guide base at position i is b" planes in shared memory; per guide the select is one
//                LDS per position at a warp-uniform offset from constant memory, the count a bit-sliced carry-save
//                adder tree (2 LOP3 per full adder), the threshold 2 LOP3; two stages with a warp-uniform early out.
//                Hits (rare): count read from the bit-sliced counter, R4 check on last windows, atomic append.
// Integer pipe + shared-memory bound; no tensor cores (nothing here is a dense contraction worth a GEMM:
// the bit-sliced form costs ~1.1 ALU ops per (window, guide) pair, below one op per output element).
#pragma once
#include <cstdint>
#include <type_traits>
#ifndef VS_HOST_UNIT_TEST          // tests/cpu_kernel_units.cpp and tests/cpu_scan_emulator.cpp compile this header with g++ and run the
                                   // kernels on the host (k_extract with one OS thread per CUDA thread, the others thread by thread)
#include <cuda_runtime.h>
#endif
#include "../../include/varscot_scan.h"

namespace vs {

constexpr int BLK_WORDS    = 48;                  // words per candidate block
constexpr int BLK_GROUP    = 32;                  // blocks per layout group: word w of block b sits at plane_index(b, w), so that
                                                  // the 32 lanes of a warp (32 consecutive blocks) touch 128 contiguous bytes per word
constexpr int BLK_LAST     = 46;                  // word index of the last-window mask
constexpr int BLK_VALID    = 47;                  // word index of the valid mask

__host__ __device__ __forceinline__ uint64_t plane_index(uint64_t blk, int w)
{
    return (blk / BLK_GROUP) * (uint64_t)(BLK_WORDS * BLK_GROUP) + (uint64_t)w * BLK_GROUP + (blk % BLK_GROUP);
}

struct PamParams {
    int n;            // number of forward dinucleotides (2 or 3)
    int fx[3], fy[3]; // forward: W[21] == fx && W[22] == fy
    int rx[3], ry[3]; // reverse: W[0]  == rx && W[1]  == ry   (reverse complement of the forward list)
};

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t eq_plane(uint32_t h, uint32_t l, int code)
{
    uint32_t mh = (code & 2) ? 0u : ~0u;   // XNOR masks: ~(h ^ H) = h ^ ~H
    uint32_t ml = (code & 1) ? 0u : ~0u;
    return (h ^ mh) & (l ^ ml);
}

// Candidate masks for the 32 window starts of one word (a = its bases, b = next word's bases, m = its masks).
//   m.iv (precomputed by the packer): start is invalid — the window holds an N, runs over a contig end or past the
//         text (R1, R3);  m.lw: the window ends exactly at a contig end (R4, bidir_mapping.cpp:51)
//   R2: PAM on the genome: forward W[21..22], reverse W[0..1]   (bidir_mapping.cpp:70-76, :240-247)
__device__ __forceinline__ void cand_masks(const vs_bases &a, const vs_bases &b, const vs_masks &m, const PamParams &pp,
                                           uint32_t &fwd, uint32_t &rev)
{
    const uint32_t h21 = __funnelshift_r(a.hi, b.hi, 21), h22 = __funnelshift_r(a.hi, b.hi, 22);
    const uint32_t l21 = __funnelshift_r(a.lo, b.lo, 21), l22 = __funnelshift_r(a.lo, b.lo, 22);
    const uint32_t h0 = a.hi, l0 = a.lo, h1 = __funnelshift_r(a.hi, b.hi, 1), l1 = __funnelshift_r(a.lo, b.lo, 1);
    uint32_t f = 0, r = 0;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        if (j < pp.n) {
            f |= eq_plane(h21, l21, pp.fx[j]) & eq_plane(h22, l22, pp.fy[j]);
            r |= eq_plane(h0, l0, pp.rx[j]) & eq_plane(h1, l1, pp.ry[j]);
        }
    }
    fwd = f & ~m.iv;
    rev = r & ~m.iv;
}

// ------------------------------------------------------------------------------------------------
// 32 x 32 bit-matrix transpose in registers (LSB-first): out[i] bit c = in[c] bit i.
// Stages 16 and 8 move whole bytes (2 PRMT per pair), stages 4, 2, 1 are masked swaps (5 ops per pair);
// ptxas drops the swaps that only feed unused outputs.
__device__ __forceinline__ void transpose32(uint32_t (&a)[32])
{
#pragma unroll
    for (int k = 0; k < 16; ++k) {                       // 16-bit halves: a[k].hi <-> a[k+16].lo
        const uint32_t x = a[k], y = a[k + 16];
        a[k] = __byte_perm(x, y, 0x5410);
        a[k + 16] = __byte_perm(x, y, 0x7632);
    }
#pragma unroll
    for (int k = 0; k < 32; k = ((k | 8) + 1) & ~8) {    // bytes: odd bytes of a[k] <-> even bytes of a[k+8]
        const uint32_t x = a[k], y = a[k | 8];
        a[k] = __byte_perm(x, y, 0x6240);
        a[k | 8] = __byte_perm(x, y, 0x7351);
    }
    uint32_t m = 0x0F0F0F0Fu;
#pragma unroll
    for (int j = 4; j; j >>= 1, m ^= m << j) {
#pragma unroll
        for (int k = 0; k < 32; k = ((k | j) + 1) & ~j) {
            const uint32_t t = ((a[k] >> j) ^ a[k | j]) & m;
            a[k | j] ^= t;
            a[k] ^= t << j;
        }
    }
}

constexpr int EX_THREADS   = 64;                  // threads per extraction CTA
constexpr int EX_MAX_WORDS = 256;                 // words per tile (<=); the host picks the tile so that it holds ~60 blocks

// k_extract: one 64-thread CTA per tile of `tile_words` words.  global_base = position of device word 0 (relative to the
// shard's position origin: the 32-bit positions it writes are global - origin).
//   phase 1 (bit-parallel, 32 starts per word): candidate masks per strand -> shared memory + exclusive rank prefix;
//   phase 2 (one THREAD per 32-candidate block): walk the masks from the block's first candidate, gather the 23-base
//            windows (funnel shifts on the staged planes), transpose 32 x 23 bits twice in registers, write
//            48 plane words + 32 positions.
// Block ranges are claimed with one atomicAdd per strand per tile on cnt[2], cnt[3] (layout order is not
// deterministic; hit resolution sorts).  If a claim runs past the capacity nothing is written for that tile; k_score
// then skips the whole chunk and the host, which reads the counters back, regrows the stores and redoes the chunk.
// Block layout (48 words): hi_0..hi_22, lo_0..lo_22, last-window mask, valid mask; word w of block b at plane_index(b, w).
// (Measured on B200 and dropped in round 2: one thread per HALF block — two 16-row transposes, half the registers, twice
// the resident warps — extracts config 3 in 1.04 ms per 0.25-scale pass against 0.98 ms for this form.)
#ifndef VS_EX_MINBLOCKS
#define VS_EX_MINBLOCKS 10
#endif
__global__ void __launch_bounds__(EX_THREADS, VS_EX_MINBLOCKS)
k_extract(const vs_bases *__restrict__ B, const vs_masks *__restrict__ M, uint64_t w_begin, uint64_t w_end, uint32_t tile_words,
          uint64_t global_base, PamParams pp,
          uint32_t *__restrict__ planes_f, uint32_t *__restrict__ pos_f,
          uint32_t *__restrict__ planes_r, uint32_t *__restrict__ pos_r, uint64_t cap,
          unsigned long long *__restrict__ cnt)
{
    __shared__ __align__(16) uint2 s_hl[EX_MAX_WORDS + 2];   // bases {hi, lo} per word (+ halo, + one word read under the sentinel)
    __shared__ uint32_t s_m[2][EX_MAX_WORDS + 1];      // candidate masks per strand
    __shared__ uint32_t s_p[2][EX_MAX_WORDS + 1];      // exclusive rank prefix per word (+ total at [nw])
    __shared__ __align__(16) uint2 s_mk[EX_MAX_WORDS + 2];   // window masks {iv, lw} per word (+ one word read under the sentinel)
    __shared__ uint32_t wsum[2][EX_MAX_WORDS / EX_THREADS][EX_THREADS / 32];
    __shared__ unsigned long long base[2];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint64_t w0 = w_begin + (uint64_t)blockIdx.x * tile_words;
    const uint32_t nw = (uint32_t)min((uint64_t)tile_words, w_end - w0);      // words of this tile
    // phase 1a: the tile's bases (+ halo word) and window masks are staged into shared memory with cp.async (LDGSTS):
    // coalesced 128-bit copies when the tile starts on a 16-byte boundary (always, except for odd test chunk sizes),
    // 64-bit copies otherwise; nothing passes through registers and every copy of the tile is in flight at once.
#ifndef VS_HOST_UNIT_TEST
    {
        const uint32_t sb = (uint32_t)__cvta_generic_to_shared(s_hl), smk = (uint32_t)__cvta_generic_to_shared(s_mk);
        const char *gb = reinterpret_cast<const char *>(B + w0), *gm = reinterpret_cast<const char *>(M + w0);
        const uint32_t nb_bytes = (nw + 1) * 8u, nm_bytes = nw * 8u;        // B[w_end] is the halo / pad word, always readable
        if (((w0 & 1) == 0)) {
            for (uint32_t o = tid * 16u; o + 16u <= nb_bytes; o += EX_THREADS * 16u)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sb + o), "l"(gb + o));
            for (uint32_t o = tid * 16u; o + 16u <= nm_bytes; o += EX_THREADS * 16u)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smk + o), "l"(gm + o));
            if (tid == 0 && (nb_bytes & 8u)) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sb + nb_bytes - 8u), "l"(gb + nb_bytes - 8u));
            if (tid == 1 && (nm_bytes & 8u)) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smk + nm_bytes - 8u), "l"(gm + nm_bytes - 8u));
        } else {
            for (uint32_t o = tid * 8u; o < nb_bytes; o += EX_THREADS * 8u)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sb + o), "l"(gb + o));
            for (uint32_t o = tid * 8u; o < nm_bytes; o += EX_THREADS * 8u)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smk + o), "l"(gm + o));
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
#else       // host emulation (tests/cpu_kernel_units.cpp): plain copies
    for (uint32_t i = tid; i < nw + 1; i += EX_THREADS) s_hl[i] = uint2{B[w0 + i].hi, B[w0 + i].lo};
    for (uint32_t i = tid; i < nw; i += EX_THREADS) s_mk[i] = uint2{M[w0 + i].iv, M[w0 + i].lw};
#endif
    __syncthreads();
    constexpr int EX_ITERS = EX_MAX_WORDS / EX_THREADS;
    // phase 1b: candidate masks and their rank prefix (word order: thread t owns words t, t+64, t+128, t+192)
    uint32_t cf[EX_ITERS], cr[EX_ITERS], xf[EX_ITERS], xr[EX_ITERS];
#pragma unroll
    for (int it = 0; it < EX_ITERS; ++it) {
        const uint32_t i = it * EX_THREADS + tid;
        uint32_t fwd = 0, rev = 0;
        if (i < nw) {
            const uint2 cur = s_hl[i], nx = s_hl[i + 1], mk = s_mk[i];
            cand_masks(vs_bases{cur.x, cur.y}, vs_bases{nx.x, nx.y}, vs_masks{mk.x, mk.y}, pp, fwd, rev);
            s_m[0][i] = fwd; s_m[1][i] = rev;
        }
        cf[it] = __popc(fwd); cr[it] = __popc(rev);
        uint32_t a = cf[it], b = cr[it];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t p = __shfl_up_sync(0xffffffffu, a, o), q = __shfl_up_sync(0xffffffffu, b, o);
            if (lane >= o) { a += p; b += q; }
        }
        xf[it] = a; xr[it] = b;
        if (lane == 31) { wsum[0][it][wid] = a; wsum[1][it][wid] = b; }
    }
    __syncthreads();
    uint32_t run_f = 0, run_r = 0;                     // candidates before the current group of 64 words
#pragma unroll
    for (int it = 0; it < EX_ITERS; ++it) {
        const uint32_t i = it * EX_THREADS + tid;
        const uint32_t w0f = wsum[0][it][0], w0r = wsum[1][it][0], w1f = wsum[0][it][1], w1r = wsum[1][it][1];
        if (i < nw) {
            s_p[0][i] = run_f + (wid ? w0f : 0u) + xf[it] - cf[it];
            s_p[1][i] = run_r + (wid ? w0r : 0u) + xr[it] - cr[it];
        }
        run_f += w0f + w1f; run_r += w0r + w1r;
    }
    const uint32_t nf = run_f, nr = run_r;
    const uint32_t nbf = (nf + 31) >> 5, nbr = (nr + 31) >> 5;
    if (tid == 0) {
        s_p[0][nw] = nf; s_p[1][nw] = nr;
        s_m[0][nw] = ~0u; s_m[1][nw] = ~0u;              // sentinel: ends the mask walk of a partial block (see phase 2)
        base[0] = atomicAdd(&cnt[2], (unsigned long long)nbf);
        base[1] = atomicAdd(&cnt[3], (unsigned long long)nbr);
        if (nf) atomicAdd(&cnt[0], (unsigned long long)nf);
        if (nr) atomicAdd(&cnt[1], (unsigned long long)nr);
    }
    __syncthreads();
    const uint32_t gbase = (uint32_t)(global_base + w0 * 32);      // device word 0 sits at global_base
    for (uint32_t j = tid; j < nbf + nbr; j += EX_THREADS) {
#include "vs_extract_block.inc"
    }
}

// k_scatter_masks: expand the sparse form of the window masks (only words with a non-zero mask travel over PCIe).
__global__ void __launch_bounds__(256)
k_scatter_masks(const vs_mask_entry *__restrict__ e, uint64_t n, uint64_t word_base, vs_masks *__restrict__ M)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        vs_mask_entry x = e[i];
        M[x.word - word_base] = vs_masks{x.iv, x.lw};
    }
}

// ------------------------------------------------------------------------------------------------
// Window masks on the device, from the compact mask source of a view (include/varscot_scan.h).
// k_fill_runs: plane[word - word_base + i] = value for the part of every run {word, count, value} that lies inside
// [lo, hi) (global word indices).  Warp (blockIdx.x * 8 + warp) owns a run, blockIdx.y selects a segment of FILL_SEG
// words of it, so that a long run (an N stretch of a chromosome is 10^5 words) is filled by many warps.
constexpr uint32_t FILL_SEG = 1024;
__global__ void __launch_bounds__(256)
k_fill_runs(const vs_plane_run *__restrict__ runs, uint64_t n_runs, uint64_t lo, uint64_t hi, uint64_t word_base, uint32_t *__restrict__ plane)
{
    const uint64_t r = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= n_runs) return;
    const vs_plane_run x = runs[r];
    const uint64_t a = max((uint64_t)x.word, lo) + (uint64_t)blockIdx.y * FILL_SEG;
    const uint64_t b = min(min((uint64_t)x.word + x.count, hi), a + FILL_SEG);
    for (uint64_t w = a + (threadIdx.x & 31); w < b; w += 32) plane[w - word_base] = x.value;
}

// k_expand_em_code: contig-end plane words from their one-byte codes, for the words of blocks that travel coded
// (code = index of the only set bit, VS_EM_NONE = no single bit; words with several bits arrive as runs afterwards).
// code / out point at the first word of the range (global word index g0), dense at block 0 of the text.
__global__ void __launch_bounds__(256)
k_expand_em_code(const uint8_t *__restrict__ code, const uint8_t *__restrict__ dense, uint64_t g0, uint64_t n, uint32_t *__restrict__ out)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !dense[(g0 + i) / VS_EM_BLOCK]) return;
    const uint32_t c = code[i];
    out[i] = c < 32u ? 1u << c : 0u;
}

// k_masks_from_planes: the device twin of masks_of() in vs_host.cpp.  nm / em point at the first word of the range and
// hold n + 1 words (the last one is the halo);
//   iv: any N in [p, p+23)  or  any contig end in [p, p+22)   (R1, R3)
//   lw: the window is valid and its last base (p+22) is a contig end   (R4)
__global__ void __launch_bounds__(256)
k_masks_from_planes(const uint32_t *__restrict__ nm, const uint32_t *__restrict__ em, uint64_t n, vs_masks *__restrict__ out)
{
    const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n) return;
    const uint64_t N = ((uint64_t)nm[w + 1] << 32) | nm[w], E = ((uint64_t)em[w + 1] << 32) | em[w];
    uint64_t t = N | (N >> 1); t |= t >> 2; t |= t >> 4; t |= t >> 8;      // OR over 16 consecutive
    const uint64_t n23 = t | (t >> 7);                                       // OR over 23
    uint64_t e = E | (E >> 1); e |= e >> 2; e |= e >> 4; e |= e >> 8;
    const uint64_t e22 = e | (e >> 6);                                       // OR over 22
    vs_masks m;
    m.iv = (uint32_t)(n23 | e22);
    m.lw = (uint32_t)(E >> 22) & ~m.iv;
    out[w] = m;
}

// ------------------------------------------------------------------------------------------------
// Scoring.
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c)
{
#ifndef VS_HOST_UNIT_TEST
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(c), "n"(LUT));
    return r;
#else       // the instruction's definition: bit (4a + 2b + c) of the table, per bit position
    uint32_t r = 0;
    for (int i = 0; i < 8; ++i)
        if ((LUT >> i) & 1) r |= ((i & 4) ? a : ~a) & ((i & 2) ? b : ~b) & ((i & 1) ? c : ~c);
    return r;
#endif
}

// Bit-sliced population count of N one-bit planes (plus optional planes `init[w]` already carrying weight 2^w):
// column compression with full adders (2 LOP3 each: XOR3 0x96, MAJ3 0xE8) taken from the front of a queue so the
// tree stays balanced.  Written as template recursion so that every index is a compile-time constant and all
// planes live in registers.
template <int HEAD, int TAIL, int NN>
struct CsaColumn {
    static constexpr int LEFT = TAIL - HEAD;
    using Next = CsaColumn<(LEFT >= 3 ? HEAD + 3 : HEAD + 2), TAIL + 1, NN + 1>;
    static __device__ __forceinline__ void run(uint32_t *col, uint32_t *nxt)
    {
        if constexpr (LEFT >= 3) {
            const uint32_t x = col[HEAD], y = col[HEAD + 1], z = col[HEAD + 2];
            col[TAIL] = lop3<0x96>(x, y, z);
            nxt[NN] = lop3<0xE8>(x, y, z);
            Next::run(col, nxt);
        } else if constexpr (LEFT == 2) {
            const uint32_t x = col[HEAD], y = col[HEAD + 1];
            col[TAIL] = x ^ y;
            nxt[NN] = x & y;
            Next::run(col, nxt);
        }
    }
    static __host__ __device__ constexpr int final_head() { if constexpr (LEFT >= 2) return Next::final_head(); else return HEAD; }
    static __host__ __device__ constexpr int final_left() { if constexpr (LEFT >= 2) return Next::final_left(); else return LEFT; }
    static __host__ __device__ constexpr int final_nn() { if constexpr (LEFT >= 2) return Next::final_nn(); else return NN; }
};

template <int W, int N_IN, bool HAS_INIT>
struct CsaWeights {
    static __device__ __forceinline__ void run(uint32_t *col, const uint32_t *init, uint32_t *bit)
    {
        constexpr int T0 = N_IN + (HAS_INIT ? 1 : 0);
        if constexpr (HAS_INIT) col[N_IN] = init[W];
        using C = CsaColumn<0, T0, 0>;
        uint32_t nxt[T0 + 2];
        C::run(col, nxt);
        if constexpr (C::final_left() == 1) bit[W] = col[C::final_head()]; else bit[W] = 0u;
        if constexpr (W < 4) {
            constexpr int NN = C::final_nn();
            uint32_t col2[2 * NN + 4];
#pragma unroll
            for (int i = 0; i < NN; ++i) col2[i] = nxt[i];
            CsaWeights<W + 1, NN, HAS_INIT>::run(col2, init, bit);
        }
    }
};

template <int N, bool HAS_INIT>
__device__ __forceinline__ void popcount_planes(const uint32_t (&in)[N], const uint32_t (&init)[5], uint32_t (&bit)[5])
{
    uint32_t col[2 * N + 4];
#pragma unroll
    for (int i = 0; i < N; ++i) col[i] = in[i];
    CsaWeights<0, N, HAS_INIT>::run(col, init, bit);
}

// count <= K on a 5-bit bit-sliced count (K <= 8): two LOP3 with compile-time LUTs
template <int K>
__device__ __forceinline__ uint32_t le_k(const uint32_t (&b)[5])
{
    constexpr int LUT_F = (K < 8) ? ((1 << (K + 1)) - 1) : 0x01;   // f(b2,b1,b0): low3 <= K      (K = 8: low3 == 0)
    constexpr int LUT_G = (K < 8) ? 0x02 : 0x0B;                   // g(b4,b3,f): ~b4 & ~b3 & f   (K = 8: ~b4 & (~b3 | f))
    const uint32_t f = lop3<LUT_F>(b[2], b[1], b[0]);
    return lop3<LUT_G>(b[4], b[3], f);
}

// Number of pattern slots scored before the early-out test: with uniform-random text, after PA(K) informative
// positions fewer than ~12 % of the warp iterations (1024 window x guide pairs) still hold a pair with <= K mismatches, so
// the remaining slots (the PAM positions come last in the slot order) are loaded only for those.
__host__ __device__ constexpr int stage_a_slots(int k) { return k >= 8 ? VS_GLEN : 7 + 2 * k; }

// ---- k_score: "guide per lane" ------------------------------------------------------------------------------------
// One CTA scores one BATCH of SC_NB consecutive candidate blocks (one layout group: 6 KB of contiguous plane words)
// of one strand against every guide of the launch.
//   expand : the CTA turns the 46 raw planes of each block into the 92 planes "mismatch if the pattern base at position
//            i is b" in shared memory, block-major: word (4 i + b) of block j at s_planes[j * SC_STRIDE + 4 i + b]
//            (one 16-byte store per position).  Invalid lanes of a partial block mismatch everywhere.
//   score  : LANE = GUIDE.  A warp takes 32 guides (or, for the tail of the guide list, GW = 16 / 8 / 4 guides x 32 / GW
//            blocks at a time); each lane holds the byte offsets of ITS pattern's planes in registers — loaded once per
//            (batch, guide segment) from the pattern table in global memory — and walks the blocks of the batch:
//            per block PA(K) x [LDS at lane offset + uniform block base], a bit-sliced carry-save adder tree over the 32
//            candidates of the block (2 LOP3 per full adder), a 2-LOP3 threshold and a warp vote; the few iterations that
//            pass score the remaining slots and, on a hit (rare), read the exact count out of the bit-sliced counter,
//            apply R4 and append.
// Compared with one-candidate-block-per-lane this needs no per-guide uniform loads in the hot loop (the offsets live
// in registers), 12 KB of shared memory per CTA instead of 43 KB (occupancy is set by registers alone), reads every
// block from HBM once per launch whatever the number of guides, and keeps the pattern table per context in global
// memory (no __constant__ symbol shared by the contexts of a device).
// Shared-memory banks: the lanes of a warp read at most 4 words per block (one per pattern base), (32 / GW) blocks at a
// time; SC_STRIDE = 92 = 4 (mod 8) puts the 4-word groups of up to 8 consecutive blocks in distinct banks, and lanes
// reading the same word are served by broadcast, so every LDS is a single wavefront.
#ifndef VS_SCORE_WARPS
#define VS_SCORE_WARPS 4
#endif
#ifndef VS_SCORE_UNROLL
#define VS_SCORE_UNROLL 8              // block iterations per trip of the walk
#endif
constexpr int SC_UNROLL = VS_SCORE_UNROLL;
constexpr int SC_WARPS   = VS_SCORE_WARPS;
constexpr int SC_THREADS = 32 * SC_WARPS;         // guides per pass of a CTA over its batch
constexpr int SC_NB      = BLK_GROUP;             // blocks per batch
constexpr int SC_STRIDE  = 4 * VS_GLEN;           // words per block in shared memory
static_assert(SC_STRIDE % 8 == 4, "block stride must be 4 mod 8 words: conflict-free reads of up to 8 blocks at a time");
constexpr int SC_SMEM_BYTES = (SC_NB * SC_STRIDE + SC_NB + BLK_WORDS * SC_NB) * 4;      // planes + last-window masks + raw staging (18 KB)
constexpr int PAT_STRIDE = 24;                    // uint16 per pattern (23 slot offsets + pad; 48 bytes = 3 x 16)

// key of the bucketed index (vs_bucket.cuh): the PAM dinucleotide + the VS_KEYLEN - 2 bases next to it
#ifndef VS_KEYLEN
#define VS_KEYLEN 8
#endif
static_assert(VS_KEYLEN == 6 || VS_KEYLEN == 8, "key of 4 or 6 bases + the PAM dinucleotide");
// position scored by slot j of a strand's slot order: the PAM dinucleotide last, before it the bases next to it
// (forward 0..22; reverse VS_KEYLEN..22, 2..VS_KEYLEN-1, 0, 1) — so that the first 23 - VS_KEYLEN slots are exactly the positions
// outside the key of the bucketed index, and the first PA(K) slots never hold the PAM
__host__ __device__ constexpr int slot_position(int strand, int j)
{
    return !strand ? j : (j < VS_GLEN - VS_KEYLEN ? j + VS_KEYLEN : (j < VS_GLEN - 2 ? j - (VS_GLEN - VS_KEYLEN) + 2 : j - (VS_GLEN - 2)));
}
// table entry of slot j for pattern base b (0..3): byte offset of plane (4 position + b) inside a block's shared-memory row
__host__ __device__ constexpr uint16_t pat_slot(int strand, int j, int b) { return (uint16_t)((4 * slot_position(strand, j) + b) * 4); }
// inverse of pat_slot
__host__ __device__ __forceinline__ void pat_decode(int strand, int j, uint32_t e, int &i, int &b)
{
    i = slot_position(strand, j);
    b = (int)((e >> 2) & 3u);
}
__host__ __device__ constexpr int score_min_blocks(int k)
{
#ifdef VS_SCORE_MINBLOCKS
    return VS_SCORE_MINBLOCKS;          // tuning override: only steers the register allocation
#endif
    // registers: PA offsets + PA loaded planes + adder temporaries; 64 per thread for k <= 6, 80 above
    return (k <= 6 ? 1024 : 768) / SC_THREADS;
}

struct ScoreArgs {
    const uint32_t *planes[2];  // per strand: candidate blocks, word w of block b at plane_index(b, w)
    const uint32_t *pos[2];     // per strand: [n_blocks][32] global positions
    const unsigned long long *rng;  // device: {lo_fwd, lo_rev, hi_fwd, hi_rev} block range to score (written by k_extract_mark)
    uint64_t cap;               // capacity of each candidate store; a range that ran past it is skipped (the host redoes the pass)
    uint32_t n_guides;          // guides of this launch: rows [guide_base, guide_base + n_guides) of the table
    uint32_t guide_base;
    uint32_t pat_guides;        // rows per strand of the table
    uint32_t rot_shift;         // the guide slices of the warps rotate every 2^rot_shift batches (>= 32: never)
    const uint16_t *pat;        // [2][pat_guides][PAT_STRIDE] slot offsets (pat_slot), 16-byte aligned rows
    vs_hit *hits;
    unsigned long long *n_hits;
    uint64_t hit_cap;
};

// (One atomicAdd per hit on purpose: a warp-aggregated append measured slower on B200 in every config, including the
// dense one, because the whole warp then walks the slow path.)
// Slow path (rare): for every candidate of the lane's block that passed the threshold read its exact count out of the
// bit-sliced counter, apply R4 to last-window candidates (H over positions 11..22 must be <= floor(K/2),
// bidir_mapping.cpp:48-53) and append the hit.  `row` = the block's expanded planes in shared memory, `po` = the lane's
// pattern in the global table.
#if defined(VS_SCORE_NOINLINE_HITS) && !defined(VS_HOST_UNIT_TEST)
#define VS_NOINLINE __noinline__          // tuning variant: smaller unrolled walk, at the price of spills around the call
#else
#define VS_NOINLINE __forceinline__
#endif
// `extra` = mismatches already known outside the counted slots (the key positions of a bucket; 0 for the plain index).
template <int K>
__device__ __forceinline__ void score_hits_body(const char *row, const uint16_t *po, int strand, uint32_t le, const uint32_t (&cnt)[5], uint32_t extra,
                                                uint32_t lastm, const uint32_t *pos, uint32_t info, vs_hit *hits,
                                                unsigned long long *n_hits, uint64_t hit_cap)
{
    while (le != 0) {
        const int c = __ffs(le) - 1;
        le &= le - 1;
        const uint32_t mm = extra + (((cnt[0] >> c) & 1u) | (((cnt[1] >> c) & 1u) << 1) | (((cnt[2] >> c) & 1u) << 2) |
                                     (((cnt[3] >> c) & 1u) << 3) | (((cnt[4] >> c) & 1u) << 4));
        if ((lastm >> c) & 1u) {                                             // R4: last window of its contig
            uint32_t h2 = 0;
#pragma unroll 1
            for (int j = 0; j < VS_GLEN; ++j)
                if (slot_position(strand, j) >= 11) h2 += (*reinterpret_cast<const uint32_t *>(row + po[j]) >> c) & 1u;
            if (h2 > (uint32_t)(K / 2)) continue;
        }
        const unsigned long long idx = atomicAdd(n_hits, 1ull);
        if (idx < hit_cap) {
            vs_hit hrec;
            hrec.pos = pos[c];
            hrec.info = info | mm;
            hits[idx] = hrec;
        }
    }
}
template <int K>
__device__ VS_NOINLINE void score_hits(const char *row, const uint16_t *po, int strand, uint32_t le, const uint32_t (&cnt)[5],
                                       uint32_t lastm, const uint32_t *pos, uint32_t info, vs_hit *hits, unsigned long long *n_hits, uint64_t hit_cap)
{
    score_hits_body<K>(row, po, strand, le, cnt, 0u, lastm, pos, info, hits, n_hits, hit_cap);
}
// the same out of line (k_score_bucketed instantiates its walk once per class: the rare path must not be copied into each)
#ifndef VS_HOST_UNIT_TEST
#define VS_COLD __noinline__
#else
#define VS_COLD
#endif
template <int K>
__device__ VS_COLD void score_hits_cold(const char *row, const uint16_t *po, int strand, uint32_t le, const uint32_t (&cnt)[5], uint32_t extra,
                                        uint32_t lastm, const uint32_t *pos, uint32_t info, vs_hit *hits, unsigned long long *n_hits, uint64_t hit_cap)
{
    score_hits_body<K>(row, po, strand, le, cnt, extra, lastm, pos, info, hits, n_hits, hit_cap);
}

template <int K>
__global__ void __launch_bounds__(SC_THREADS, score_min_blocks(K))
k_score(ScoreArgs a)
{
#ifndef VS_HOST_UNIT_TEST       // (the host emulation declares vs::sm itself)
    extern __shared__ __align__(16) uint32_t sm[];     // [SC_NB][SC_STRIDE] planes, [SC_NB] last-window masks, [BLK_WORDS][SC_NB] raw staging
#endif
    constexpr int PA = stage_a_slots(K), PB = VS_GLEN - PA;
    constexpr uint32_t ROW = SC_STRIDE * 4u;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (max(a.rng[2], a.rng[3]) > a.cap) return;          // the candidate store overflowed: the host regrows it and redoes the pass
    // persistent CTAs: batches of the forward range first, then of the reverse range, strided over the grid — the grid does
    // not depend on the block counts, which only the device knows while a pass is in flight
    const unsigned long long nbat_f = (a.rng[2] - a.rng[0] + SC_NB - 1) / SC_NB, nbat = nbat_f + (a.rng[3] - a.rng[1] + SC_NB - 1) / SC_NB;
    uint32_t *lastm_s = sm + SC_NB * SC_STRIDE;
    uint32_t *raw_s = lastm_s + SC_NB;                      // the batch's 48 raw words per block, as they lie in the store (6 KB)
    const uint32_t zero5[5] = {0u, 0u, 0u, 0u, 0u};
    auto batch_of = [&](unsigned long long bat, uint32_t &strand, unsigned long long &blk0, uint32_t &nb) {
        strand = bat >= nbat_f;
        blk0 = a.rng[strand] + (bat - (strand ? nbat_f : 0ull)) * SC_NB;
        nb = (uint32_t)min((unsigned long long)SC_NB, a.rng[2 + strand] - blk0);
    };
    // stage the raw words of a batch: one layout group = BLK_WORDS * SC_NB contiguous words (ranges start on group boundaries
    // and the store's capacity is a whole number of groups, so the copy never leaves the allocation); cp.async, so the next
    // batch's words arrive while this one is scored
    auto stage = [&](unsigned long long bat) {
        uint32_t strand, nb; unsigned long long blk0;
        batch_of(bat, strand, blk0, nb);
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
    if ((unsigned long long)blockIdx.x < nbat) stage(blockIdx.x);
    // a warp whose 32 guides are the same for every batch (the launch has no more guides than the CTA has lanes) keeps the
    // addresses of its pattern's planes in registers across batches; they change only with the strand
    // The warps of a CTA sit on different SM sub-partitions (warp id mod 4).  When the guides do not fill every warp (100
    // guides: three full warps and one that works an eighth of the time) the light role must not always fall on the same
    // sub-partition: the guide slice of a warp rotates every 8 batches (and starts at the CTA index).
    const uint32_t warps = blockDim.x >> 5;
    const char *adr_keep[PA];
    int kept_strand = -1;                                   // strand and role the kept addresses belong to
    uint32_t iter = 0;
    for (unsigned long long bat = blockIdx.x; bat < nbat; bat += gridDim.x, ++iter) {
    const uint32_t role = ((uint32_t)wid + (a.rot_shift < 32u ? blockIdx.x + (iter >> a.rot_shift) : 0u)) % warps;
    // the role has exactly one full 32-guide segment in the whole guide list: its plane addresses can stay in registers
    const bool fixed_guides = 32u * role + 32u <= a.n_guides && 32u * warps + 32u * role + 32u > a.n_guides;
    uint32_t strand, nb; unsigned long long blk0;
    batch_of(bat, strand, blk0, nb);
#ifndef VS_HOST_UNIT_TEST
    asm volatile("cp.async.wait_group 0;" ::: "memory");
#endif
    __syncthreads();
    // expand: thread -> (block tid % 32, positions tid / 32, tid / 32 + warps, ...); rows past the range mismatch everywhere
    {
        const uint32_t b = (uint32_t)lane;
        const uint32_t inv = b < nb ? ~raw_s[BLK_VALID * SC_NB + b] : ~0u;
        for (int p = wid; p < VS_GLEN; p += (int)(blockDim.x >> 5)) {
            const uint32_t h = raw_s[p * SC_NB + b], l = raw_s[(VS_GLEN + p) * SC_NB + b];
            *reinterpret_cast<uint4 *>(sm + b * SC_STRIDE + 4 * p) =
                make_uint4((h | l) | inv, (h | ~l) | inv, (~h | l) | inv, (~h | ~l) | inv);     // pattern base A, C, G, T
        }
        if (wid == 0) lastm_s[b] = b < nb ? raw_s[BLK_LAST * SC_NB + b] : 0u;
    }
    __syncthreads();
    if (bat + gridDim.x < nbat) stage(bat + gridDim.x);    // the staging area is free again: fetch the next batch
    const uint16_t *pat0 = a.pat + ((size_t)strand * a.pat_guides + a.guide_base) * PAT_STRIDE;
    const uint32_t *posb = (strand ? a.pos[1] : a.pos[0]) + blk0 * 32;

    // one guide segment: GW = 2^L guides [seg, seg + GW) x (32 / GW) blocks per warp iteration.  The walk always covers the
    // SC_NB rows of the batch (rows past the range mismatch everywhere), so its trip count and the block offsets are
    // compile-time constants: every LDS is [address register + immediate], no address arithmetic inside a trip.
    auto segment = [&](uint32_t seg, auto gw_log2_c, auto keep_c) {
        constexpr uint32_t L = decltype(gw_log2_c)::value, GW = 1u << L, STEP = 32u >> L;
        constexpr bool KEEP = decltype(keep_c)::value;      // walk with the kept address registers (restored after the walk)
        const uint32_t sub = (uint32_t)lane >> L;
        const uint32_t g = seg + ((uint32_t)lane & (GW - 1u));
        const bool real = g < a.n_guides;                  // padding lanes score the segment's first guide; their hits are dropped
        const uint16_t *po = pat0 + (size_t)(real ? g : seg) * PAT_STRIDE;
        const char *smb = reinterpret_cast<const char *>(sm) + sub * ROW;     // the lane's first block row
        const char *adr_local[KEEP ? 1 : PA];
        const char *(&adr)[KEEP ? PA : (KEEP ? 1 : PA)] = *reinterpret_cast<const char *(*)[PA]>(KEEP ? (void *)adr_keep : (void *)adr_local);   // the lane's stage-A planes in that row
        if (!KEEP || kept_strand != (int)(strand * 64u + role)) {
            const uint4 *q = reinterpret_cast<const uint4 *>(po);
            uint32_t w[12];
#pragma unroll
            for (int i = 0; i < 3; ++i) { const uint4 v = q[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
#pragma unroll
            for (int i = 0; i < PA; ++i) adr[i] = smb + ((w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu);
            if (KEEP) kept_strand = (int)(strand * 64u + role);
        }
        // UNR iterations per trip with compile-time offsets; the address registers advance once per trip
        constexpr uint32_t UNR = (uint32_t)SC_UNROLL < (uint32_t)SC_NB / STEP ? (uint32_t)SC_UNROLL : (uint32_t)SC_NB / STEP;
#pragma unroll 1
        for (uint32_t j0 = 0; j0 < (uint32_t)SC_NB; j0 += STEP * UNR) {
#pragma unroll
            for (uint32_t u = 0; u < UNR; ++u) {
                const uint32_t j = j0 + u * STEP;              // first block of the iteration
                uint32_t m[PA], ca[5];
#pragma unroll
                for (int i = 0; i < PA; ++i) m[i] = *reinterpret_cast<const uint32_t *>(adr[i] + u * STEP * ROW);
                popcount_planes<PA, false>(m, zero5, ca);
                uint32_t le = le_k<K>(ca);
                // warp-uniform early out: if no pair of the iteration can still be within K, the remaining slots are never scored
                if (PB == 0 ? (le != 0) : __any_sync(0xffffffffu, le != 0)) {
                    const char *row = smb + j * ROW;
                    if constexpr (PB > 0) {
                        uint32_t mb[PB], cb[5];
#pragma unroll
                        for (int i = 0; i < PB; ++i) mb[i] = *reinterpret_cast<const uint32_t *>(row + po[PA + i]);
                        popcount_planes<PB, true>(mb, ca, cb);
                        le = le_k<K>(cb);
#pragma unroll
                        for (int w = 0; w < 5; ++w) ca[w] = cb[w];
                    }
                    if (le != 0 && real)
                        score_hits<K>(row, po, (int)strand, le, ca, lastm_s[j + sub], posb + (size_t)(j + sub) * 32,
                                      ((a.guide_base + g) << 8) | (strand << 7), a.hits, a.n_hits, a.hit_cap);
                }
            }
#pragma unroll
            for (int i = 0; i < PA; ++i) adr[i] += STEP * UNR * ROW;
        }
        if (KEEP) {
#pragma unroll
            for (int i = 0; i < PA; ++i) adr[i] -= SC_NB * ROW;
        }
    };
    for (uint32_t gc = 0; gc < a.n_guides; gc += 32u * warps) {
        const uint32_t g_w = gc + 32u * role;
        if (g_w >= a.n_guides) break;
        const uint32_t n = min(32u, a.n_guides - g_w);
        // tail of the guide list: pad to a multiple of 4 and split into 16 / 8 / 4 guides x 2 / 4 / 8 blocks per iteration; a tail
        // of 29..31 guides pads to a full segment (its padding lanes score the segment's first guide, their hits are dropped)
        const uint32_t np = (n + 3u) & ~3u;
        if (np == 32u) {
            if (fixed_guides && n == 32u) segment(g_w, std::integral_constant<uint32_t, 5>{}, std::true_type{});
            else segment(g_w, std::integral_constant<uint32_t, 5>{}, std::false_type{});
            continue;
        }
        uint32_t seg = g_w;
        if (np & 16u) { segment(seg, std::integral_constant<uint32_t, 4>{}, std::false_type{}); seg += 16u; }
        if (np & 8u) { segment(seg, std::integral_constant<uint32_t, 3>{}, std::false_type{}); seg += 8u; }
        if (np & 4u) { segment(seg, std::integral_constant<uint32_t, 2>{}, std::false_type{}); }
    }
    // (the barrier at the top of the next batch keeps its expansion from overwriting planes that are still being scored)
    }
}

// k_extract_mark: closes the block range of one pipeline chunk.  cnt[2], cnt[3] are the running block claims of the two
// strands; the chunk's range {lo, hi} goes to rng[0..3], the claims are rounded up to a whole layout group (so that the
// next chunk — and every batch of k_score — starts on a 4 KB boundary of the store), the padding blocks get an empty valid
// mask, the next chunk's lo is written to rng[4..5] and the whole-store range {0, 0, end, end} to all[0..3].
__global__ void __launch_bounds__(32)
k_extract_mark(unsigned long long *cnt, unsigned long long *rng, unsigned long long *all, uint32_t *planes_f, uint32_t *planes_r, uint64_t cap)
{
    const int s = threadIdx.x;                             // one thread per strand (at most 31 padding blocks each)
    if (s > 1) return;
    const unsigned long long hi = cnt[2 + s], end = (hi + BLK_GROUP - 1) / BLK_GROUP * BLK_GROUP;
    uint32_t *pl = s ? planes_r : planes_f;
    for (unsigned long long b = hi; b < end && b < cap; ++b) { pl[plane_index(b, BLK_VALID)] = 0u; pl[plane_index(b, BLK_LAST)] = 0u; }
    rng[2 + s] = hi;
    rng[4 + s] = end;
    all[s] = 0ull; all[2 + s] = end;
    cnt[2 + s] = end;
}

// ---- hit resolution on the device ---------------------------------------------------------------------------------------
// k_contig_starts_*: the start positions of the contigs that overlap the shard, from the shard's contig-end plane
// (em, one bit per base, set on the last base of a contig): starts[0] = first_start (given by the host: the contig that
// holds the shard's first base), starts[r + 1] = position after the r-th end bit.  Three steps: bits per tile of
// CS_TILE words, exclusive scan of the tile counts (one CTA), scatter.  Positions are relative to the shard's origin
// (first_base = position of device word 0); first_start may lie before the origin and is then stored modulo 2^32.
constexpr int CS_TILE = 2048;              // words per CTA of 256 threads (8 per thread)
__global__ void __launch_bounds__(256)
k_contig_starts_count(const uint32_t *__restrict__ em, uint64_t n_words, uint32_t *__restrict__ tile_cnt)
{
    __shared__ uint32_t s_c[256];
    const uint64_t w0 = (uint64_t)blockIdx.x * CS_TILE + (uint64_t)threadIdx.x * 8;
    uint32_t c = 0;
    for (int i = 0; i < 8; ++i) if (w0 + i < n_words) c += __popc(em[w0 + i]);
    s_c[threadIdx.x] = c;
    __syncthreads();
    if (threadIdx.x < 32) {                                // the bit count of a tile is small work: 8 adds per lane, 32 by lane 0
        uint32_t t = 0;
        for (int i = 0; i < 8; ++i) t += s_c[threadIdx.x * 8 + i];
        s_c[threadIdx.x * 8] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int i = 0; i < 32; ++i) t += s_c[i * 8]; tile_cnt[blockIdx.x] = t; }
}
// exclusive scan of n tile counts in place (single CTA of 1024 threads), total to *total
__global__ void __launch_bounds__(1024)
k_contig_starts_scan(uint32_t *tile_cnt, uint32_t n, uint32_t *total)
{
    __shared__ uint32_t part[1024];
    const uint32_t per = (n + 1023) / 1024, a = min(n, threadIdx.x * per), b = min(n, a + per);
    uint32_t sum = 0;
    for (uint32_t i = a; i < b; ++i) sum += tile_cnt[i];
    part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t run = 0; for (int i = 0; i < 1024; ++i) { const uint32_t v = part[i]; part[i] = run; run += v; } *total = run; }
    __syncthreads();
    uint32_t run = part[threadIdx.x];
    for (uint32_t i = a; i < b; ++i) { const uint32_t v = tile_cnt[i]; tile_cnt[i] = run; run += v; }
}
__global__ void __launch_bounds__(256)
k_contig_starts_scatter(const uint32_t *__restrict__ em, uint64_t n_words, const uint32_t *__restrict__ tile_off, uint64_t first_base,
                        uint32_t first_start, uint32_t *__restrict__ starts)
{
    __shared__ uint32_t s_c[256 + 32];
    const uint64_t w0 = (uint64_t)blockIdx.x * CS_TILE + (uint64_t)threadIdx.x * 8;
    uint32_t c = 0;
    for (int i = 0; i < 8; ++i) if (w0 + i < n_words) c += __popc(em[w0 + i]);
    s_c[threadIdx.x] = c;
    __syncthreads();
    if (threadIdx.x < 32) { uint32_t t = 0; for (int i = 0; i < 8; ++i) t += s_c[threadIdx.x * 8 + i]; s_c[256 + threadIdx.x] = t; }
    __syncthreads();
    // end bits of the tile before this thread's words: whole groups of 8 threads, then the threads of its own group
    uint32_t r = tile_off[blockIdx.x];
    for (uint32_t i = 0; i < threadIdx.x / 8; ++i) r += s_c[256 + i];
    for (uint32_t i = threadIdx.x & ~7u; i < threadIdx.x; ++i) r += s_c[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) starts[0] = first_start;
    for (int i = 0; i < 8; ++i) {
        if (w0 + i >= n_words) break;
        uint32_t m = em[w0 + i];
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            starts[++r] = (uint32_t)(first_base + (w0 + i) * 32 + b + 1);
        }
    }
}

// k_resolve_hits: hit {position, info} -> sort key + payload.  The contig is the last one whose start is <= the
// position (binary search over the shard's n_starts contig starts; contig id = first_contig + index);
// positions and starts are relative to the shard's origin.  starts[0] is never compared (every probe has mid >= 1): the
// first contig may begin before the origin, its start is then stored modulo 2^32, and pos - starts[0] wraps to the exact
// position in the contig (a contig holds at most 2^32 bases).
//   key = (guide - guide_lo) << 49 | strand << 48 | (contig & 0xFFFF) << 32 | pos in contig     (the std::map order of
//         bidir_mapping.cpp:13,154 inside the pass order of :285-295)
//   val = contig << 32 | info
__global__ void __launch_bounds__(256)
k_resolve_hits(const vs_hit *__restrict__ hits, uint64_t n, const uint32_t *__restrict__ starts, uint32_t n_starts, uint32_t first_contig,
               uint32_t guide_lo, unsigned long long *__restrict__ keys, unsigned long long *__restrict__ vals)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const vs_hit h = hits[i];
    uint32_t lo = 0, hi = n_starts;                        // invariant: starts[lo] <= pos < starts[hi] (starts[n_starts] = +inf)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (starts[mid] <= h.pos) lo = mid; else hi = mid;
    }
    const uint32_t contig = first_contig + lo, pos = h.pos - starts[lo];
    const unsigned long long guide = (h.info >> 8) - guide_lo, strand = (h.info >> 7) & 1u;
    keys[i] = (guide << 49) | (strand << 48) | ((unsigned long long)(contig & 0xFFFFu) << 32) | pos;
    vals[i] = ((unsigned long long)contig << 32) | h.info;
}
// sorted {key, val} pairs -> vs_loc_hit records
__global__ void __launch_bounds__(256)
k_pack_loc_hits(const unsigned long long *__restrict__ keys, const unsigned long long *__restrict__ vals, uint64_t n, vs_loc_hit *__restrict__ out)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    vs_loc_hit r;
    r.key = keys[i]; r.contig = (uint32_t)(vals[i] >> 32); r.info = (uint32_t)vals[i];
    out[i] = r;
}

#include "vs_bucket.cuh"

// ------------------------------------------------------------------------------------------------
// Microbenchmarks for the roofline denominators (alu-pipe LOP3 issue rate, shared-memory LDS rate).
#ifndef VS_HOST_UNIT_TEST
__global__ void __launch_bounds__(256)
k_peak_lop3(uint32_t *out, int iters)
{
    uint32_t a0 = threadIdx.x, a1 = a0 * 3 + 1, a2 = a0 * 5 + 2, a3 = a0 * 7 + 3, a4 = a0 * 11 + 4, a5 = a0 * 13 + 5, a6 = a0 * 17 + 6, a7 = a0 * 19 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = lop3<0x96>(a0, a1, a2); a1 = lop3<0xE8>(a1, a2, a3); a2 = lop3<0x96>(a2, a3, a4); a3 = lop3<0xE8>(a3, a4, a5);
            a4 = lop3<0x96>(a4, a5, a6); a5 = lop3<0xE8>(a5, a6, a7); a6 = lop3<0x96>(a6, a7, a0); a7 = lop3<0xE8>(a7, a0, a1);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}

__global__ void __launch_bounds__(256)
k_peak_lds(uint32_t *out, int iters)
{
    __shared__ uint32_t s[256 * 8];
    for (int i = threadIdx.x; i < 256 * 8; i += 256) s[i] = i * 2654435761u;
    __syncthreads();
    uint32_t acc = 0;
    const volatile uint32_t *p = s + threadIdx.x;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) acc ^= p[u * 256];
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}

#endif  // VS_HOST_UNIT_TEST

}  // namespace vs
