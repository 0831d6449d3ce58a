// tests/cpu_beyond_4g_units.cpp — TEST INFRASTRUCTURE for texts beyond 4 Gbases: the device code that places positions
// (k_contig_starts_*, k_resolve_hits, k_extract, k_bucket_gather, compiled from vs_kernels.cuh under tests/cuda_on_host.h)
// run on the host with shard-relative positions, and the shard plan of the library (vs::shard_plan, linked from
// libvarscot_scan.so).  Built with -fvisibility=hidden so that the library's own kernel launch stubs stay bound to the
// library.  Nothing in the product uses this file.  Built and run by tests/test_zz_beyond_4g.py.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <random>
#include <vector>

#include "cuda_on_host.h"
#include "../varscot_b200/csrc/vs_kernels.cuh"
#include "../varscot_b200/csrc/vs_internal.h"

namespace vs { uint32_t sm[SC_SMEM_BYTES / 4] __attribute__((aligned(16))); }
using namespace vs;

static int failures = 0;
#define CHECK(cond)                                                                     \
    do {                                                                                \
        if (!(cond)) { ++failures; fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); } \
    } while (0)

static std::mt19937_64 rng(4242);
static uint32_t r32() { return (uint32_t)rng(); }

// ---- contig starts and hit resolution of a shard whose origin lies above 2^32 ---------------------------------------------
// The shard [W0, W0 + n_words) of a text longer than 4 Gbases has origin W0 * 32.  As vs_device.cu does: the starts come
// from the shard's contig-end plane (no empty contig in the range) or are the host's offsets minus the origin (modulo 2^32:
// the first contig may begin before the origin); k_resolve_hits must give the (contig, pos) of a 64-bit linear search.
static void check_shard(const std::vector<uint64_t> &off, uint64_t W0, uint64_t n_words)
{
    const uint64_t origin = W0 * 32, b0 = origin, b1 = std::min<uint64_t>(off.back(), (W0 + n_words) * 32);
    const uint32_t n_contigs = (uint32_t)(off.size() - 1);
    // plan_contig_starts: the last contig starting at or before the first / last base of the shard
    const uint32_t c_first = (uint32_t)(std::upper_bound(off.begin(), off.end(), b0) - off.begin() - 1);
    const uint32_t c_last = (uint32_t)(std::upper_bound(off.begin(), off.end(), b1 - 1) - off.begin() - 1);
    std::vector<uint32_t> em(n_words + 1, 0);
    bool any_empty = false;
    for (uint32_t c = c_first; c <= c_last; ++c) {
        any_empty |= off[c + 1] == off[c];
        const uint64_t last = off[c + 1] - 1;
        if (off[c + 1] > off[c] && last >= origin && last < (W0 + n_words) * 32) em[(last - origin) >> 5] |= 1u << (last & 31);
    }
    em[n_words] = ~0u;                                       // the halo word does not count
    const uint32_t n_starts = c_last - c_first + 1;
    std::vector<uint32_t> host(n_starts);                    // finish_contig_starts' fallback
    for (uint32_t i = 0; i < n_starts; ++i) host[i] = (uint32_t)(off[c_first + i] - origin);
    std::vector<std::vector<uint32_t>> forms{host};
    if (!any_empty) {                                        // the derivation from the plane (enqueue_starts_from_plane)
        const unsigned tiles = (unsigned)((n_words + CS_TILE - 1) / CS_TILE);
        std::vector<uint32_t> tile(tiles + 1, 0), starts(n_starts + 4, 0xDEADBEEFu);
        uint32_t total = 0;
        launch_cta(tiles, 256, [&] { k_contig_starts_count(em.data(), n_words, tile.data()); });
        launch_cta(1, 1024, [&] { k_contig_starts_scan(tile.data(), tiles, &total); });
        launch_cta(tiles, 256, [&] {
            k_contig_starts_scatter(em.data(), n_words, tile.data(), W0 * 32 - origin, (uint32_t)(off[c_first] - origin), starts.data());
        });
        const uint32_t expect_bits = c_last - c_first + (off[c_last + 1] - 1 < (W0 + n_words) * 32 ? 1u : 0u);
        CHECK(total == expect_bits);
        for (uint32_t i = 0; i < n_starts; ++i) CHECK(starts[i] == host[i]);
        starts.resize(n_starts);
        forms.push_back(starts);
    }
    // hits at random window starts of the shard, plus the first and the last base of every contig of the range
    std::vector<uint64_t> gpos;
    for (int i = 0; i < 400; ++i) gpos.push_back(b0 + rng() % (b1 - b0));
    for (uint32_t c = c_first; c <= c_last; ++c)
        if (off[c + 1] > off[c])
            for (uint64_t g : {off[c], off[c + 1] - 1}) if (g >= b0 && g < b1) gpos.push_back(g);
    const uint64_t n = gpos.size();
    std::vector<vs_hit> hits(n);
    for (uint64_t i = 0; i < n; ++i) {
        hits[i].pos = (uint32_t)(gpos[i] - origin);
        CHECK(gpos[i] - origin < (1ull << 32) - 8192);
        hits[i].info = ((7 + r32() % 50) << 8) | ((r32() & 1) << 7) | (r32() % 9);
    }
    for (const auto &starts : forms) {
        std::vector<unsigned long long> keys(n), vals(n);
        launch((unsigned)((n + 255) / 256), 1, 256, [&] { k_resolve_hits(hits.data(), n, starts.data(), n_starts, c_first, 7, keys.data(), vals.data()); });
        for (uint64_t i = 0; i < n; ++i) {
            uint32_t c = 0;                                  // 64-bit linear search: the last contig starting at or before the base
            for (uint32_t x = 0; x < n_contigs; ++x) if (off[x] <= gpos[i]) c = x;
            const uint64_t pos = gpos[i] - off[c];
            CHECK((uint32_t)(vals[i] >> 32) == c && (uint32_t)vals[i] == hits[i].info);
            CHECK((keys[i] & 0xFFFFFFFFull) == pos && ((keys[i] >> 32) & 0xFFFF) == (c & 0xFFFF));
        }
    }
}

static void test_starts_and_resolve_beyond_4g()
{
    const uint64_t W0 = ((5ull << 32) + (1ull << 30)) / 32;     // the shard starts at 5.25 Gbases
    for (int rep = 0; rep < 12; ++rep) {
        const uint64_t n_words = rep == 0 ? 1 : 200 + r32() % (3 * CS_TILE);
        const uint64_t origin = W0 * 32, end = (W0 + n_words) * 32;
        std::vector<uint64_t> off{0};
        // contig 0 ends somewhere far below; then the contig holding the shard's first base: it starts before the origin
        // (by up to almost 2^32 bases: starts[0] then wraps), or exactly on it
        off.push_back(1000);
        const uint64_t back = rep % 3 == 0 ? 0 : rep % 3 == 1 ? 1 + r32() % 100000 : (1ull << 32) - 50 - r32() % 1000;
        off.push_back(origin - back);
        uint64_t at = origin - back;
        while (at < end) {
            const uint32_t kind = r32() % 8;
            uint64_t len = kind == 0 ? 0 : kind == 1 ? 23 + r32() % 30 : kind == 2 ? 1 + r32() % 22 : 30 + r32() % 3000;
            if (rep % 2 == 0 && kind == 0) len = 45;              // every second rep has no empty contig: the plane path runs
            if (at < origin && at + len <= origin) len = origin - at + r32() % 40;     // the first contig reaches into the shard
            at += len;
            off.push_back(at);
        }
        if (rep % 4 == 1) off.back() = end;                           // a contig that ends exactly on the shard border
        if (rep % 4 == 3) { off.back() = end; off.push_back(end); off.push_back(end + 77); }   // ... followed by an empty one
        else off.push_back(off.back() + 500);
        check_shard(off, W0, n_words);
    }
}

// ---- k_extract and k_bucket_gather with a non-zero position base: the same windows, positions moved by the base -----------
static void test_extract_and_gather_with_base()
{
    const uint64_t n_words = 3000;
    std::vector<vs_bases> B(n_words + 1);
    std::vector<vs_masks> M(n_words);
    for (uint64_t w = 0; w < n_words; ++w) {
        B[w] = vs_bases{r32(), r32()};
        M[w] = vs_masks{r32() & r32() & r32(), 0};
        M[w].lw = r32() & r32() & ~M[w].iv;
    }
    B[n_words] = vs_bases{0, 0};
    PamParams pp;
    pp.n = 2;
    pp.fx[0] = 2; pp.fy[0] = 2; pp.fx[1] = 2; pp.fy[1] = 0; pp.fx[2] = 0; pp.fy[2] = 0;
    for (int j = 0; j < 3; ++j) { pp.rx[j] = 3 - pp.fy[j]; pp.ry[j] = 3 - pp.fx[j]; }
    const uint32_t tile_words = 160;
    const uint64_t cap = (n_words + n_words / tile_words + 64) / BLK_GROUP * BLK_GROUP + BLK_GROUP;      // at most 32 candidates per word
    struct Store { std::vector<uint32_t> pl[2], pos[2]; std::vector<unsigned long long> cnt; };
    auto extract = [&](uint64_t base, Store &st) {
        for (int s = 0; s < 2; ++s) { st.pl[s].assign(cap * BLK_WORDS, 0xDEADBEEFu); st.pos[s].assign(cap * 32, 0xDEADBEEFu); }
        st.cnt.assign(8, 0);
        const unsigned tiles = (unsigned)((n_words + tile_words - 1) / tile_words);
        launch_cta(tiles, EX_THREADS, [&] {
            k_extract(B.data(), M.data(), 0, n_words, tile_words, base, pp, st.pl[0].data(), st.pos[0].data(), st.pl[1].data(), st.pos[1].data(), cap, st.cnt.data());
        });
    };
    // a shard at word 0 of a text within 4 Gbases (base 0); a shard of such a text at a later word (origin 0: base = its
    // first base); a shard of a longer text (origin = its first base: base 0 again, tested above by equality with the first)
    const uint64_t bases_to_try[] = {0, 123456789ull * 32, ((1ull << 32) - 8192) - n_words * 32};
    Store ref;
    extract(0, ref);
    CHECK(ref.cnt[0] > 1000 && ref.cnt[1] > 1000 && ref.cnt[2] <= cap && ref.cnt[3] <= cap);
    for (uint64_t base : bases_to_try) {
        Store st;
        extract(base, st);
        CHECK(st.cnt == ref.cnt);
        for (int s = 0; s < 2; ++s) {
            CHECK(st.pl[s] == ref.pl[s]);
            const uint64_t nb = ref.cnt[2 + s];
            for (uint64_t b = 0; b < nb; ++b) {
                const uint32_t valid = ref.pl[s][plane_index(b, BLK_VALID)];
                for (int c = 0; c < 32; ++c)
                    if ((valid >> c) & 1) CHECK(st.pos[s][b * 32 + c] == (uint32_t)(ref.pos[s][b * 32 + c] + base));
            }
        }
        // the bucketed store's gather: the extracted positions (with BK_NOPOS padding slots in between) read back the same
        // windows from the text at that base
        for (int s = 0; s < 2; ++s) {
            const uint64_t nb = 2 * BLK_GROUP;                         // whole layout groups (plane_index)
            std::vector<uint32_t> pos_ref(nb * 32, BK_NOPOS), pos_b(nb * 32, BK_NOPOS);
            for (uint64_t i = 0; i < nb * 32; ++i)
                if (r32() % 5) {
                    const uint64_t j = r32() % (ref.cnt[2 + s] * 32);   // some slot of the plain store
                    const uint64_t b = j / 32, c = j % 32;
                    if (!((ref.pl[s][plane_index(b, BLK_VALID)] >> c) & 1)) continue;
                    pos_ref[i] = ref.pos[s][j];
                    pos_b[i] = st.pos[s][j];
                }
            std::vector<uint32_t> g_ref(nb * BLK_WORDS, 0), g_b(nb * BLK_WORDS, 1);
            launch((unsigned)((nb + 63) / 64), 1, 64, [&] { k_bucket_gather(B.data(), M.data(), 0, pos_ref.data(), nb, g_ref.data()); });
            launch((unsigned)((nb + 63) / 64), 1, 64, [&] { k_bucket_gather(B.data(), M.data(), base, pos_b.data(), nb, g_b.data()); });
            CHECK(g_ref == g_b);
            uint64_t filled = 0;
            for (uint64_t b = 0; b < nb; ++b) filled += __builtin_popcount(g_ref[plane_index(b, BLK_VALID)]);
            CHECK(filled > nb * 16);
        }
    }
}

// ---- the shard plan of vs_map_records and the executables --------------------------------------------------------------
static void test_shard_plan()
{
    for (double gbases : {3.9, 4.0, 4.3, 9.0, 17.0})
        for (int nd : {1, 2, 3, 8}) {
            const uint64_t n_words = ((uint64_t)(gbases * 1e9) + 31) / 32;
            const std::vector<uint64_t> b = shard_plan(n_words, nd);
            const uint64_t ns = b.size() - 1;
            const bool beyond = n_words * 32 > (1ull << 32);
            const uint64_t fewest = (n_words + VS_MAX_SHARD_WORDS - 1) / VS_MAX_SHARD_WORDS;
            const uint64_t want = beyond ? (std::max<uint64_t>(nd, fewest) + nd - 1) / nd * nd : (uint64_t)nd;
            CHECK(ns == want);
            CHECK(ns % (uint64_t)nd == 0);
            if (!beyond) CHECK(b == shard_bounds(n_words, nd));       // texts within 4 Gbases: one shard per device, as before
            CHECK(b.front() == 0 && b.back() == n_words);
            uint64_t lo = ~0ull, hi = 0;
            for (uint64_t s = 0; s < ns; ++s) {
                const uint64_t n = b[s + 1] - b[s];
                CHECK(b[s] % 256 == 0 && b[s] < b[s + 1]);
                if (beyond) CHECK(n <= VS_MAX_SHARD_WORDS);
                lo = std::min(lo, n); hi = std::max(hi, n);
            }
            CHECK(hi - lo <= 2 * 256);                                  // shards differ by a tile (and the clipped tail)
            std::vector<uint64_t> dev((size_t)nd, 0);                   // device i scans shards [i, i + 1) * ns / nd
            for (uint64_t s = 0; s < ns; ++s) dev[s / (ns / nd)] += b[s + 1] - b[s];
            CHECK(*std::max_element(dev.begin(), dev.end()) - *std::min_element(dev.begin(), dev.end()) <= 2 * 256 * (ns / nd));
        }
}

int main()
{
    test_starts_and_resolve_beyond_4g();
    test_extract_and_gather_with_base();
    test_shard_plan();
    if (failures) { fprintf(stderr, "%d check(s) failed\n", failures); return 1; }
    printf("beyond 4G units ok\n");
    return 0;
}
