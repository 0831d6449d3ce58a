// tests/cpu_deal_units.cpp — TEST INFRASTRUCTURE: the deal of a batch's guide segments to the warps of k_score_bucketed
// (vs::bk_deal in varscot_b200/csrc/vs_bucket.cuh), compiled for the HOST with g++ under tests/cuda_on_host.h.
//  * every segment of every class is dealt exactly once, to a warp in range, in the shape the kernel walks (32 guides while a
//    whole 32 fit, then 4-guide segments over the tail), as runs of consecutive segments;
//  * the most loaded warp stays within the longest-first bound 1.25 x LB for 4 warps, where LB is a lower bound of the best
//    possible deal: the mean load, the largest segment, and (j + 1) x the (4 j + 1)-th largest segment (4 j + 1 segments on
//    4 warps put j + 1 of them on one warp);
//  * a warp holds at most BK_RUNS runs of segments (what k_score_bucketed keeps per warp in shared memory).
// Class counts: guides 1..32768 whose keys meet a bucket key as the bench's guides do (PAM GG against GG / GA buckets, uniform
// bases next to it), and uniformly random splits; K = 0..8.  Nothing in the product uses this file.  Built and run by
// tests/test_bucketed_deal.py.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <random>
#include <vector>

#include "cuda_on_host.h"
#include "../varscot_b200/csrc/vs_kernels.cuh"

namespace vs { uint32_t sm[SC_SMEM_BYTES / 4] __attribute__((aligned(16))); }
using namespace vs;

static int failures = 0;
#define CHECK(cond)                                                                     \
    do {                                                                                \
        if (!(cond)) { ++failures; fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); } \
    } while (0)

static std::mt19937_64 rng(2026);
static double worst_ratio = 0.0;

// the deal of one batch for K, checked; returns the largest warp load over LB
template <int K>
static double check_deal(const uint32_t (&cls)[BK_CLS], uint32_t warps)
{
    constexpr uint32_t CMAX = K < VS_KEYLEN ? K : VS_KEYLEN;
    std::vector<uint32_t> owner(cls[VS_KEYLEN + 1], ~0u);               // per guide entry: the warp that scores it
    std::vector<uint64_t> load(warps, 0);
    std::vector<uint64_t> costs;
    std::vector<uint32_t> runs(warps, 0);
    bk_deal<K>(cls, warps, [&](uint32_t w, uint32_t at0, uint32_t nseg, uint32_t c, uint32_t L, uint32_t last) {
        CHECK(w < warps && nseg >= 1);
        ++runs[w < warps ? w : 0];
        for (uint32_t j = 0; j < nseg; ++j) {
            const uint32_t at = at0 + (j << L), n_real = j + 1 < nseg ? 1u << L : last;
            CHECK(c <= CMAX && (L == 5u || L == 2u));
            CHECK(at >= cls[c] && at + n_real <= cls[c + 1] && n_real >= 1 && n_real <= (1u << L));
            const uint32_t i = at - cls[c], n = cls[c + 1] - cls[c];
            // the kernel's shape: 32-guide segments at multiples of 32 while a whole one fits, the tail in 4-guide segments
            if (L == 5u) CHECK(i % 32u == 0 && i + 32u <= n && n_real == 32u);
            else CHECK(i >= (n & ~31u) && (i - (n & ~31u)) % 4u == 0 && n_real == std::min(4u, n - i));
            for (uint32_t g = at; g < at + n_real && g < owner.size(); ++g) {
                CHECK(owner[g] == ~0u);
                owner[g] = w;
            }
            const uint64_t cost = bk_segment_cost(K - (int)c, L == 5u ? 32u : 4u);
            load[w < warps ? w : 0] += cost;
            costs.push_back(cost);
        }
    });
    for (uint32_t w = 0; w < warps; ++w) CHECK(runs[w] <= (uint32_t)BK_RUNS);          // what the kernel keeps per warp
    for (uint32_t g = cls[0]; g < cls[CMAX + 1]; ++g) CHECK(owner[g] != ~0u);          // every guide of a class c <= K
    for (uint32_t g = cls[CMAX + 1]; g < cls[VS_KEYLEN + 1]; ++g) CHECK(owner[g] == ~0u);  // and none beyond
    if (costs.empty()) return 0.0;
    std::sort(costs.rbegin(), costs.rend());
    uint64_t total = 0;
    for (uint64_t x : costs) total += x;
    double lb = std::max((double)total / warps, (double)costs[0]);
    for (size_t j = 1; j * warps < costs.size(); ++j) lb = std::max(lb, (double)(j + 1) * (double)costs[j * warps]);
    const double ratio = (double)*std::max_element(load.begin(), load.end()) / lb;
    if (warps == (uint32_t)SC_WARPS) {
        CHECK(ratio <= 1.25 + 1e-9);
        if (ratio > 1.25 + 1e-9) {
            fprintf(stderr, "  K=%d cls:", K);
            for (int c = 0; c < BK_CLS; ++c) fprintf(stderr, " %u", cls[c]);
            fprintf(stderr, "  ratio %.3f\n", ratio);
        }
    }
    worst_ratio = std::max(worst_ratio, warps == (uint32_t)SC_WARPS ? ratio : 0.0);
    return ratio;
}

static void check_any_k(int K, const uint32_t (&cls)[BK_CLS], uint32_t warps)
{
    switch (K) {
    case 0: check_deal<0>(cls, warps); break;
    case 1: check_deal<1>(cls, warps); break;
    case 2: check_deal<2>(cls, warps); break;
    case 3: check_deal<3>(cls, warps); break;
    case 4: check_deal<4>(cls, warps); break;
    case 5: check_deal<5>(cls, warps); break;
    case 6: check_deal<6>(cls, warps); break;
    case 7: check_deal<7>(cls, warps); break;
    default: check_deal<8>(cls, warps); break;
    }
}

static void starts_of(const uint32_t (&cnt)[VS_KEYLEN + 1], uint32_t (&cls)[BK_CLS])
{
    uint32_t run = 0;
    for (int c = 0; c <= VS_KEYLEN; ++c) { cls[c] = run; run += cnt[c]; }
    cls[VS_KEYLEN + 1] = run;
}

// class counts of n guides with PAM GG in a bucket of kind GG or GA, as k_guide_classes computes them
static void bench_like(uint32_t n, uint32_t (&cls)[BK_CLS])
{
    const uint32_t pam_gg = (2u << BK_KEYBITS) | (2u << (BK_KEYBITS + 2)), pam_ga = 2u << BK_KEYBITS;
    const uint32_t bkey = (uint32_t)(rng() & (BK_PER_KIND - 1)) | ((rng() & 1) ? pam_gg : pam_ga);
    uint32_t cnt[VS_KEYLEN + 1] = {};
    for (uint32_t g = 0; g < n; ++g) ++cnt[key_mismatches((uint32_t)(rng() & (BK_PER_KIND - 1)) | pam_gg, bkey)];
    starts_of(cnt, cls);
}

static void random_split(uint32_t n, uint32_t (&cls)[BK_CLS])
{
    uint32_t cnt[VS_KEYLEN + 1] = {};
    const uint32_t used = 1 + (uint32_t)(rng() % (VS_KEYLEN + 1));      // classes that get guides
    for (uint32_t g = 0; g < n; ++g) ++cnt[rng() % used];
    starts_of(cnt, cls);
}

int main()
{
    // the cost is monotone in the shape and the slot count: the deal order (32-guide segments, then 4-guide ones, c ascending)
    // is longest first
    for (int kp = 0; kp < 8; ++kp) {
        CHECK(bk_segment_cost(kp, 32u) >= bk_segment_cost(kp + 1, 4u) && bk_segment_cost(8, 4u) <= bk_segment_cost(0, 32u));
        CHECK(bk_segment_cost(kp, 32u) <= bk_segment_cost(kp + 1, 32u) && bk_segment_cost(kp, 4u) <= bk_segment_cost(kp + 1, 4u));
    }
    uint64_t cases = 0;
    const uint32_t small[] = {1, 2, 3, 4, 5, 9, 31, 32, 33, 36, 63, 64, 65, 100, 127, 128, 129, 255, 256, 1000, 4096};
    for (int K = 0; K <= 8; ++K)
        for (uint32_t n : small)
            for (int rep = 0; rep < 40; ++rep) {
                uint32_t cls[BK_CLS];
                if (rep & 1) random_split(n, cls); else bench_like(n, cls);
                for (uint32_t w = 1; w <= (uint32_t)SC_WARPS; ++w) { check_any_k(K, cls, w); ++cases; }
            }
    for (int it = 0; it < 4000; ++it) {
        const int K = (int)(rng() % 9);
        const uint32_t n = 1 + (uint32_t)(rng() % (it % 4 == 0 ? 32768 : 600));
        uint32_t cls[BK_CLS];
        if (it & 1) random_split(n, cls); else bench_like(n, cls);
        check_any_k(K, cls, SC_WARPS);
        ++cases;
    }
    printf("%llu deals, largest warp load / lower bound <= %.3f\n", (unsigned long long)cases, worst_ratio);
    if (failures) { fprintf(stderr, "%d check(s) failed\n", failures); return 1; }
    printf("deal units ok\n");
    return 0;
}
