// tests/cpu_window_units.cpp — TEST INFRASTRUCTURE for the genome windows of streamed records:
//   * k_loc_windows (compiled from vs_kernels.cuh under tests/cuda_on_host.h) against a naive gather from a text packed by
//     the library (vs_pack_text_planes), on a shard with origin 0 and first word > 0, and on a shard whose origin is its first
//     base (beyond 2^32) with a first contig that starts before the origin (its start stored modulo 2^32); hits in the first
//     word, in the last word, and windows that end in the halo word;
//   * vs_md_from_window against vs_md_string, both MD styles and both strands, at every window start of random texts with
//     planted near-matches of the guides.
// Built with -fvisibility=hidden so that the library's own kernel launch stubs stay bound to the library.  Nothing in the
// product uses this file.  Built and run by tests/test_record_stream.py.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <random>
#include <string>
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

static std::mt19937_64 rng(2323);
static const char ACGT[4] = {'A', 'C', 'G', 'T'};

static int code_of(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : 3; }

// The shard [W0, W0 + n_words) of a text whose bases are known only there (+ the halo word): `ascii` holds bases W0 * 32 ..
// (W0 + n_words + 1) * 32.  off: contig offsets of the whole text (global); origin: the shard's position origin.
static void check_shard(uint64_t W0, uint64_t n_words, uint64_t origin, const std::vector<uint64_t> &off)
{
    const uint64_t b0 = W0 * 32, n_local = (n_words + 1) * 32;
    std::string ascii(n_local, 'A');
    for (char &c : ascii) c = ACGT[rng() & 3];
    std::vector<vs_bases> B(n_words + 2);
    std::vector<uint32_t> nm(n_words + 2), em(n_words + 2);
    const uint64_t one[2] = {0, n_local};
    CHECK(vs_pack_text_planes(ascii.data(), n_local, one, 1, B.data(), nm.data(), em.data()) == VS_OK);
    // the contigs overlapping the shard, and their starts relative to the origin (modulo 2^32), as the upload stores them
    const uint32_t c_first = (uint32_t)(std::upper_bound(off.begin(), off.end(), b0) - off.begin() - 1);
    const uint32_t c_last = (uint32_t)(std::upper_bound(off.begin(), off.end(), b0 + n_words * 32 - 1) - off.begin() - 1);
    std::vector<uint32_t> starts;
    for (uint32_t c = c_first; c <= c_last; ++c) starts.push_back((uint32_t)(off[c] - origin));
    // window starts: the whole first word, the whole last word (its windows end in the halo word), random ones between
    std::vector<uint64_t> gpos;
    for (uint64_t i = 0; i < 32; ++i) { gpos.push_back(b0 + i); gpos.push_back(b0 + (n_words - 1) * 32 + i); }
    for (int i = 0; i < 300; ++i) gpos.push_back(b0 + rng() % (n_words * 32));
    const uint64_t n = gpos.size();
    std::vector<vs_loc_hit> hits(n);
    for (uint64_t i = 0; i < n; ++i) {
        const uint32_t c = (uint32_t)(std::upper_bound(off.begin(), off.end(), gpos[i]) - off.begin() - 1);
        const uint64_t pos = gpos[i] - off[c];
        hits[i].contig = c;
        hits[i].info = (uint32_t)(rng() & 0xFFFFFFu);
        hits[i].key = ((uint64_t)(rng() & 0x7FFF) << 49) | ((uint64_t)(c & 0xFFFF) << 32) | pos;
    }
    std::vector<uint64_t> win(n, 0);
    launch((unsigned)((n + 255) / 256), 1, 256, [&] {
        k_loc_windows(hits.data(), n, starts.data(), c_first, B.data(), W0 * 32 - origin, win.data());
    });
    for (uint64_t i = 0; i < n; ++i) {
        uint64_t want = 0;
        for (int j = 0; j < VS_GLEN; ++j) want |= (uint64_t)code_of(ascii[gpos[i] - b0 + (uint64_t)j]) << (2 * j);
        CHECK(win[i] == want);
        if (win[i] != want) { fprintf(stderr, "  gpos %llu: %llx vs %llx\n", (unsigned long long)gpos[i], (unsigned long long)win[i], (unsigned long long)want); break; }
    }
}

static void test_windows()
{
    for (int rep = 0; rep < 6; ++rep) {
        const uint64_t n_words = 1 + rng() % 300;
        // origin 0: a shard that starts at word W0 > 0 of a text within 4 Gbases; contigs of every length, one reaching into the shard
        {
            const uint64_t W0 = 1000 + rng() % 100000;
            std::vector<uint64_t> off{0, W0 * 32 - 1 - rng() % 500};
            while (off.back() < (W0 + n_words + 2) * 32) off.push_back(off.back() + 23 + rng() % 400);
            check_shard(W0, n_words, 0, off);
        }
        // origin = the shard's first base, beyond 2^32; the first contig starts before it (by up to almost 2^32 bases), or on it
        {
            const uint64_t W0 = ((5ull << 32) + (1ull << 30)) / 32, origin = W0 * 32;
            const uint64_t back = rep % 3 == 0 ? 0 : rep % 3 == 1 ? 1 + rng() % 100000 : (1ull << 32) - 50 - rng() % 1000;
            std::vector<uint64_t> off{0, 1000, origin - back};
            while (off.back() < (W0 + n_words + 2) * 32) off.push_back(std::max(off.back() + 23 + rng() % 400, origin + 1));
            check_shard(W0, n_words, origin, off);
        }
    }
}

// ---- vs_md_from_window against vs_md_string at every window start -----------------------------------------------------------
static void test_md()
{
    for (int rep = 0; rep < 4; ++rep) {
        const uint64_t n = 3000;
        std::string ascii(n, 'A');
        for (char &c : ascii) c = ACGT[rng() & 3];
        std::vector<std::vector<uint8_t>> guides(3, std::vector<uint8_t>(VS_GLEN));
        for (auto &g : guides) for (uint8_t &b : g) b = (uint8_t)(rng() & 3);
        // near-matches of the guides (0..8 substitutions), forward and reverse complement
        for (int p = 0; p + VS_GLEN <= (int)n; p += 40 + (int)(rng() % 60)) {
            std::vector<uint8_t> w = guides[rng() % 3];
            for (int m = (int)(rng() % 9); m > 0; --m) w[rng() % VS_GLEN] = (uint8_t)(rng() & 3);
            const bool rev = rng() & 1;
            for (int j = 0; j < VS_GLEN; ++j) ascii[(size_t)p + j] = ACGT[rev ? 3 - w[VS_GLEN - 1 - j] : w[j]];
        }
        const uint64_t nw = (n + 31) / 32, off[2] = {0, n};
        std::vector<vs_bases> B(nw + 1);
        std::vector<uint32_t> nm(nw + 1), em(nw + 1);
        CHECK(vs_pack_text_planes(ascii.data(), n, off, 1, B.data(), nm.data(), em.data()) == VS_OK);
        for (uint64_t p = 0; p + VS_GLEN <= n; ++p) {
            uint64_t w = 0;
            for (int j = 0; j < VS_GLEN; ++j) w |= (uint64_t)code_of(ascii[p + j]) << (2 * j);
            for (const auto &g : guides)
                for (int strand = 0; strand < 2; ++strand)
                    for (int style : {VS_MD_SEQAN, VS_MD_SAMTOOLS}) {
                        char a[64], b[64];
                        CHECK(vs_md_string(B.data(), p, g.data(), strand, style, a) == VS_OK);
                        CHECK(vs_md_from_window(w, g.data(), strand, style, b) == VS_OK);
                        CHECK(strcmp(a, b) == 0);
                    }
        }
    }
}

int main()
{
    test_windows();
    test_md();
    if (failures) { fprintf(stderr, "%d failures\n", failures); return 1; }
    printf("window units ok\n");
    return 0;
}
