// tests/cpu_stream_units.cpp — TEST INFRASTRUCTURE for the guide-range streaming driver of vs_mapper_map_stream and
// vs_map_records_stream (vs::stream_ranges + vs::deliver_pieces, linked from libvarscot_scan.so) run on the host over FAKE
// shards: every shard is a sorted vs_loc_hit list as the device emits it, and a range scan returns its slice of whole guides with
// guide ids made relative to the range.  Checked against one vs_merge_resolved over the whole lists:
//   * the concatenated deliveries are the same records, byte for byte, and the key16 collision counts add up to the same total;
//   * ranges are ascending and contiguous and cover [0, n), no guide is split, every delivery keeps to the budget unless it
//     holds a single guide, and range sizing is deterministic;
//   * record guide ids are absolute, and every window (here: contig << 32 | pos) follows its record through the merge;
//   * a sink that returns non-zero gets no further call.
// 1-8 shards, empty shards, guides without hits, a single guide, budgets from 1 record to unlimited.  Nothing in the product
// uses this file.  Built and run by tests/test_record_stream.py.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "../varscot_b200/csrc/vs_internal.h"

static int failures = 0;
#define CHECK(cond)                                                                     \
    do {                                                                                \
        if (!(cond)) { ++failures; fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); } \
    } while (0)

static std::mt19937_64 rng(9001);

static uint64_t win_of(const vs_loc_hit &h) { return ((uint64_t)h.contig << 32) | (uint32_t)h.key; }
static uint64_t win_of(const vs_record &r) { return ((uint64_t)r.contig << 32) | r.pos; }

// shard lists for n guides: per shard ascending in (guide, strand, contig & 0xFFFF, pos) as the device sorts them, ties on that
// key (contigs 2^16 apart) in any order; some guides get no hits at all, some shards are empty
static std::vector<std::vector<vs_loc_hit>> fake_shards(int n_shards, uint32_t n_guides, int density)
{
    std::vector<std::vector<vs_loc_hit>> L((size_t)n_shards);
    for (int s = 0; s < n_shards; ++s) {
        if (n_shards > 1 && rng() % 5 == 0) continue;                       // an empty shard
        for (uint32_t g = 0; g < n_guides; ++g) {
            if (rng() % 4 == 0) continue;                                   // a guide without hits on this shard
            const int n = (int)(rng() % (uint64_t)(2 * density + 1)) * (rng() % 10 == 0 ? 8 : 1);
            for (int i = 0; i < n; ++i) {
                vs_loc_hit h;
                const uint32_t strand = (uint32_t)(rng() & 1), contig = (uint32_t)(s * 10 + rng() % 3), pos = (uint32_t)(rng() % 64);
                h.contig = contig;
                h.info = (g << 8) | (strand << 7) | (uint32_t)(rng() % 9);
                h.key = ((uint64_t)strand << 48) | ((uint64_t)(contig & 0xFFFF) << 32) | pos;
                L[(size_t)s].push_back(h);
                if (rng() % 16 == 0) {                                      // a uint16 key collision: same key, contig + 2^16
                    vs_loc_hit t = h;
                    t.contig = contig + 65536;
                    t.info = (h.info & ~0x7Fu) | (uint32_t)(rng() % 9);
                    L[(size_t)s].push_back(t);
                }
            }
        }
        std::shuffle(L[(size_t)s].begin(), L[(size_t)s].end(), rng);
        std::stable_sort(L[(size_t)s].begin(), L[(size_t)s].end(), [](const vs_loc_hit &a, const vs_loc_hit &b) {
            const uint64_t pa = a.info >> 7, pb = b.info >> 7;
            return pa != pb ? pa < pb : (a.key & ((1ull << 49) - 1)) < (b.key & ((1ull << 49) - 1));
        });
    }
    return L;
}

struct Delivery {
    uint32_t lo, hi;
    uint64_t n;
};

struct Run {
    int rc = VS_OK;
    std::vector<vs_record> rec;
    std::vector<uint64_t> win;
    std::vector<Delivery> del;
    std::vector<std::pair<uint32_t, uint32_t>> scanned;
    uint64_t coll = 0;
    bool windows_ok = true;
};

// the driver over the fake shards; abort_at: the sink returns 1 on that delivery (0-based), -1 never
static Run stream(const std::vector<std::vector<vs_loc_hit>> &L, uint32_t n_guides, uint64_t target, double first_per_guide, bool windows,
                  int abort_at = -1)
{
    Run run;
    const vs::RangeScan scan = [&](uint32_t lo, uint32_t hi, vs::RangeLists &out, vs_scan_stats *st, std::string &) {
        run.scanned.push_back({lo, hi});
        out.hits.assign(L.size(), {});
        out.win.assign(L.size(), {});
        for (size_t s = 0; s < L.size(); ++s)
            for (const vs_loc_hit &h : L[s]) {
                const uint32_t g = h.info >> 8;
                if (g < lo || g >= hi) continue;
                vs_loc_hit r = h;
                r.info -= lo << 8;                                           // guide ids relative to the range, as a scan of the sub-array
                out.hits[s].push_back(r);
                if (windows) out.win[s].push_back(win_of(h));
            }
        st->n_hits = out.total();
        st->guide_passes = 1;
        return (int)VS_OK;
    };
    std::vector<vs_record> rec;
    std::vector<uint64_t> win;
    struct Ctx { Run *run; bool windows; int abort_at; } ctx{&run, windows, abort_at};
    vs_record_sink sink = [](void *user, const vs_record *r, const uint64_t *w, uint64_t n, uint32_t lo, uint32_t hi) -> int {
        Ctx *c = static_cast<Ctx *>(user);
        c->run->del.push_back({lo, hi, n});
        if ((w != nullptr) != c->windows) c->run->windows_ok = false;
        c->run->rec.insert(c->run->rec.end(), r, r + n);
        if (w) {
            c->run->win.insert(c->run->win.end(), w, w + n);
            for (uint64_t i = 0; i < n; ++i) if (w[i] != win_of(r[i])) c->run->windows_ok = false;
        }
        return (int)c->run->del.size() - 1 == c->abort_at ? 1 : 0;
    };
    const vs::RangeDeliver deliver = [&](const vs::RangeLists &lists, uint32_t lo, uint32_t hi, std::string &err) {
        const int r = vs::deliver_pieces(lists, lo, hi, target, windows, 3, sink, &ctx, rec, win, &run.coll);
        if (r == vs::SINK_ABORTED) { err = "the sink aborted"; return (int)VS_ERR_ARG; }
        return r;
    };
    vs_scan_stats st;
    std::string err;
    run.rc = vs::stream_ranges(n_guides, target, first_per_guide, scan, deliver, &st, err);
    return run;
}

static void check_case(int n_shards, uint32_t n_guides, int density, uint64_t target, bool windows)
{
    const auto L = fake_shards(n_shards, n_guides, density);
    std::vector<const vs_loc_hit *> ptr;
    std::vector<uint64_t> cnt;
    uint64_t total = 0;
    for (const auto &l : L) { ptr.push_back(l.data()); cnt.push_back(l.size()); total += l.size(); }
    std::vector<vs_record> want(total);
    uint64_t want_coll = 0;
    CHECK(vs_merge_resolved(ptr.data(), cnt.data(), (int)ptr.size(), want.data(), &want_coll, 2) == VS_OK);
    const double first = 1.0 + (double)(rng() % 40);                        // a first estimate that may be far off
    const Run run = stream(L, n_guides, target, first, windows);
    CHECK(run.rc == VS_OK);
    CHECK(run.rec.size() == total);
    CHECK(run.rec.size() == total && (total == 0 || memcmp(run.rec.data(), want.data(), total * sizeof(vs_record)) == 0));
    CHECK(run.coll == want_coll);
    CHECK(run.windows_ok);
    CHECK(!windows || run.win.size() == total);
    // deliveries: ascending, contiguous, covering [0, n), within budget unless a single guide
    uint32_t at = 0;
    for (const Delivery &d : run.del) {
        CHECK(d.lo == at && (d.hi > d.lo || n_guides == 0));
        CHECK(d.n <= target || d.hi - d.lo == 1);
        at = d.hi;
    }
    CHECK(at == n_guides);
    // scanned ranges: whole guides, contiguous; every delivery lies inside one of them
    at = 0;
    for (auto [lo, hi] : run.scanned) { CHECK(lo == at); at = hi; }
    CHECK(at == n_guides);
    for (const Delivery &d : run.del) {
        bool inside = false;
        for (auto [lo, hi] : run.scanned) inside |= d.lo >= lo && d.hi <= hi;
        CHECK(inside);
    }
    // the same inputs give the same ranges
    const Run again = stream(L, n_guides, target, first, windows);
    CHECK(again.scanned == run.scanned && again.del.size() == run.del.size());
}

int main()
{
    for (int n_shards = 1; n_shards <= 8; ++n_shards)
        for (uint32_t n_guides : {1u, 2u, 7u, 40u, 300u})
            for (uint64_t target : {(uint64_t)1, (uint64_t)2, (uint64_t)17, (uint64_t)100, (uint64_t)5000, (uint64_t)UINT64_MAX})
                check_case(n_shards, n_guides, (int)(rng() % 6), target, (n_shards + n_guides + target) % 2 == 0);
    check_case(3, 0, 2, 10, true);                                              // no guides: one empty delivery
    // guide ids beyond one range: 2 ranges at least, every record's guide absolute
    {
        const auto L = fake_shards(4, 200, 3);
        const Run run = stream(L, 200, 50, 1.0, true);
        CHECK(run.rc == VS_OK && run.scanned.size() >= 2);
        for (size_t i = 1; i < run.rec.size(); ++i) CHECK(run.rec[i].guide >= run.rec[i - 1].guide);
        for (const Delivery &d : run.del) CHECK(d.hi <= 200);
    }
    // an abort on the second delivery: no third call, VS_ERR_ARG
    {
        const auto L = fake_shards(3, 120, 4);
        const Run run = stream(L, 120, 20, 4.0, false, 1);
        CHECK(run.rc == VS_ERR_ARG);
        CHECK(run.del.size() == 2);
        const Run first = stream(L, 120, 20, 4.0, false, 0);
        CHECK(first.rc == VS_ERR_ARG && first.del.size() == 1);
    }
    // range sizing: the target over the expected, then over the observed hits per guide; at least one guide, never more than left
    CHECK(vs::next_range_guides(100, 10.0, 1000) == 10);
    CHECK(vs::next_range_guides(5, 10.0, 1000) == 1);
    CHECK(vs::next_range_guides(100, 0.5, 7) == 7);
    CHECK(vs::next_range_guides(UINT64_MAX, 10.0, 1000) == 1000);
    if (failures) { fprintf(stderr, "%d failures\n", failures); return 1; }
    printf("stream units ok\n");
    return 0;
}
