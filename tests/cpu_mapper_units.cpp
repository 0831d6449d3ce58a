// tests/cpu_mapper_units.cpp — TEST INFRASTRUCTURE for the memory check of the resident mapper (vs_mapper_create): the
// per-shard estimate vs::resident_shard_bytes and the plan check vs::resident_plan_check, linked from libvarscot_scan.so and
// run on the host — the refusal for lack of device memory is tested here, never by filling a device.  Nothing in the product
// uses this file.  Built and run by tests/test_resident_mapper.py.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <vector>

#include "../varscot_b200/csrc/vs_internal.h"

static int failures = 0;
#define CHECK(cond)                                                                     \
    do {                                                                                \
        if (!(cond)) { ++failures; fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); } \
    } while (0)

static uint64_t words_of(double gbases) { return (uint64_t)(gbases * 1e9 / 32.0); }

// the shapes of a plan: every non-empty shard with a handful of contigs and staged runs per 1000 words
static std::vector<vs::ShardShape> shapes_of(const std::vector<uint64_t> &b)
{
    std::vector<vs::ShardShape> s(b.size() - 1);
    for (size_t i = 0; i + 1 < b.size(); ++i)
        if (b[i + 1] > b[i]) s[i] = vs::ShardShape{b[i + 1] - b[i], 25, (b[i + 1] - b[i]) / 1000};
    return s;
}

// the largest need of any device for a text of `gbases` on nd devices; need per device in *need
static uint64_t max_need(double gbases, int nd, std::vector<uint64_t> *need_out = nullptr)
{
    const uint64_t nw = words_of(gbases);
    const std::vector<uint64_t> b = vs::shard_plan(nw, nd);
    std::vector<uint64_t> need, unlimited((size_t)nd, ~0ull);
    CHECK(vs::resident_plan_check(shapes_of(b), nw, unlimited, need) == -1);
    if (need_out) *need_out = need;
    return *std::max_element(need.begin(), need.end());
}

int main()
{
    // ---- the estimate grows with the shard's words and with the PAM density ----
    {
        uint64_t prev = 0;
        for (uint64_t w : {1ull << 10, 1ull << 16, 1ull << 20, 1ull << 24, 1ull << 27}) {
            const vs::ShardShape s{w, 1, 0};
            const uint64_t b2 = vs::resident_shard_bytes(s, w, 2), b3 = vs::resident_shard_bytes(s, w, 3);
            CHECK(b2 > prev);
            CHECK(b3 > b2);
            // at least the text (bases + masks, 16 B a word) and both candidate stores (plain + bucketed, 2 strands, 320 B a
            // block of 32 candidates) at the expected density
            CHECK(b3 >= w * 16 + (uint64_t)(4.0 * 320.0 * (double)w * 3.0 / 16.0));
            prev = b3;
        }
        const vs::ShardShape a{1ull << 24, 1, 0}, more_contigs{1ull << 24, 1000000, 0}, more_runs{1ull << 24, 1, 1000000};
        CHECK(vs::resident_shard_bytes(more_contigs, 1ull << 24, 3) > vs::resident_shard_bytes(a, 1ull << 24, 3));
        CHECK(vs::resident_shard_bytes(more_runs, 1ull << 24, 3) > vs::resident_shard_bytes(a, 1ull << 24, 3));
    }
    // ---- a device's need is the sum over its contiguous run of shards ----
    for (int nd : {1, 3, 8})
        for (double g : {1.0, 5.0, 17.0}) {
            const uint64_t nw = words_of(g);
            const std::vector<uint64_t> b = vs::shard_plan(nw, nd);
            const std::vector<vs::ShardShape> sh = shapes_of(b);
            std::vector<uint64_t> need;
            max_need(g, nd, &need);
            const size_t per = sh.size() / (size_t)nd;
            for (int i = 0; i < nd; ++i) {
                uint64_t sum = 0;
                for (size_t s = (size_t)i * per; s < (size_t)(i + 1) * per; ++s)
                    if (sh[s].words) sum += vs::resident_shard_bytes(sh[s], nw, 3);
                CHECK(need[(size_t)i] == sum);
            }
        }
    // ---- 1-8 devices, 1-20 Gbases: accepted exactly when every device's need fits its free bytes ----
    const uint64_t B200 = 180000000000ull;
    for (int nd = 1; nd <= 8; ++nd)
        for (int g = 1; g <= 20; ++g) {
            const uint64_t nw = words_of(g);
            const std::vector<vs::ShardShape> sh = shapes_of(vs::shard_plan(nw, nd));
            std::vector<uint64_t> need;
            const uint64_t top = max_need(g, nd);
            CHECK(vs::resident_plan_check(sh, nw, std::vector<uint64_t>((size_t)nd, top), need) == -1);       // just fits
            CHECK(vs::resident_plan_check(sh, nw, std::vector<uint64_t>((size_t)nd, top - 1), need) >= 0);    // one byte short
            // one device short of its own need: that device is the one refused
            std::vector<uint64_t> free_b = need;
            const int victim = (g * 7 + nd) % nd;
            if (need[(size_t)victim]) {
                free_b[(size_t)victim] -= 1;
                CHECK(vs::resident_plan_check(sh, nw, free_b, need) == victim);
            }
            // a fixed budget of 180 GB per device
            const int r = vs::resident_plan_check(sh, nw, std::vector<uint64_t>((size_t)nd, B200), need);
            CHECK((r == -1) == (top <= B200));
            // more devices never need more per device
            if (nd > 1) CHECK(top <= max_need(g, nd - 1));
        }
    // ---- anchors: a 17-Gbase genome (wheat) is four resident shards on one 180 GB device; 30 Gbases are not ----
    {
        const uint64_t nw17 = words_of(17), nw30 = words_of(30);
        CHECK(vs::shard_plan(nw17, 1).size() - 1 == 4);
        std::vector<uint64_t> need;
        CHECK(vs::resident_plan_check(shapes_of(vs::shard_plan(nw17, 1)), nw17, {B200}, need) == -1);
        printf("17 Gbases on one device: %.1f GB planned\n", need[0] / 1e9);
        CHECK(vs::resident_plan_check(shapes_of(vs::shard_plan(nw30, 1)), nw30, {B200}, need) == 0);
        printf("30 Gbases on one device: %.1f GB planned\n", need[0] / 1e9);
        CHECK(vs::resident_plan_check(shapes_of(vs::shard_plan(nw30, 2)), nw30, {B200, B200}, need) == -1);
    }
    if (failures) { fprintf(stderr, "%d failures\n", failures); return 1; }
    printf("mapper units ok\n");
    return 0;
}
