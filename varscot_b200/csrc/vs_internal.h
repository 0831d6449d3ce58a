// varscot_b200/csrc/vs_internal.h — helpers shared by the host and device halves of libvarscot_scan.
#pragma once
#include "../../include/varscot_scan.h"
#include <functional>
#include <string>
#include <vector>

void vs_set_last_error(const char *msg);

// Start creating the CUDA primary context of `device` (driver + module initialisation, 0.3-4 s on a cold box); the
// executables call it from a helper thread while they read their input files.
void vs_warmup_device(int device);

namespace vs {

// Why the guides, mismatch count and extra PAM of a scan are rejected, or nullptr when they are valid.  Callers check them
// before touching any device or resident state and prefix the reason with their own name.
const char *scan_arg_error(const uint8_t *guides, uint32_t n_guides, int k, int extra_pam);

// Scan a packed text on one or several devices (text sharded by word ranges as shard_plan, one host thread and one
// context per device, no collective) and return all hits, unordered.  devices empty -> device 0.
int scan_text_sharded(const vs_text_view &text, const std::vector<int> &devices,
                      const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                      std::vector<vs_hit> &hits, vs_scan_stats *agg, std::string &err);

// vs_scan_resolved with the genome window of every hit (k_loc_windows) when `windows` is set: the sink receives each
// super-chunk's sorted hits and, with windows, one uint64_t per hit (the format of vs_record_sink); NULL otherwise.
typedef int (*loc_sink)(void *user, const vs_loc_hit *hits, const uint64_t *windows, uint64_t n, uint32_t guide_lo, uint32_t guide_hi);
int scan_resolved_ex(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words,
                     const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                     vs_loc_hit *out, uint64_t out_cap, uint64_t *n_hits, bool windows, loc_sink sink, void *user, vs_scan_stats *stats);

// Expected hits per guide and text base on uniform-random text at k mismatches and the PAM set of extra_pam (what a scan
// sizes its hit buffer with).
double expected_hits_per_base(int k, int extra_pam);

// ---- guide-range streaming (vs_mapper_map_stream, vs_map_records_stream, and with one unlimited range vs_mapper_map and
// vs_map_records) ----
// The sorted lists of one guide range, one per shard, as vs_scan_resolved delivers them: guide ids (info >> 8) relative to the
// range's first guide; win[s] holds one window per hit of hits[s] when windows were asked for, and is empty otherwise.
struct RangeLists {
    std::vector<std::vector<vs_loc_hit>> hits;
    std::vector<std::vector<uint64_t>> win;
    uint64_t total() const;
};
// Scan guides [lo, hi) on every shard into `out` (cleared by the callee), counting into *stats; err names a failure.
using RangeScan = std::function<int(uint32_t lo, uint32_t hi, RangeLists &out, vs_scan_stats *stats, std::string &err)>;
// A scanned range handed to the host: called on the calling thread, ranges in ascending order.  A code other than VS_OK stops
// the stream and is returned, with the reason in err.
using RangeDeliver = std::function<int(const RangeLists &lists, uint32_t lo, uint32_t hi, std::string &err)>;
// deliver_pieces: the sink returned non-zero
constexpr int SINK_ABORTED = -1;

// Default target of records per delivery (records_per_delivery == 0).
constexpr uint64_t DEFAULT_RECORDS_PER_DELIVERY = 32ull << 20;

// Guides of the next range: target / the expected hits per guide (the last range's hits per guide once one was scanned),
// at least 1, at most `left`.  target == UINT64_MAX: all of them.
uint32_t next_range_guides(uint64_t target, double per_guide, uint32_t left);

// The streaming driver: guide ranges [lo, hi) of whole guides in ascending order, sized by next_range_guides from
// first_per_guide and then from each scanned range; while deliver() runs on range c on the calling thread, another thread
// scans range c + 1 (a pipeline of depth two).  Stats are summed over the ranges.  Every thread is joined before it returns.
int stream_ranges(uint32_t n_guides, uint64_t target, double first_per_guide, const RangeScan &scan, const RangeDeliver &deliver,
                  vs_scan_stats *stats, std::string &err);

// Merge of one range's lists (vs_merge_resolved) into records, guide ids offset by guide_base; with win_out, each record's window
// travels through the same permutation.  Records of guides [g_lo, g_hi) (relative to the range) only.
int merge_range(const RangeLists &lists, uint32_t g_lo, uint32_t g_hi, uint32_t guide_base, vs_record *out, uint64_t *win_out,
                uint64_t *key16_collisions, int n_threads);
// Records of guides [g_lo, g_hi) of the range (relative) in lists: sum over the shards.
uint64_t range_count(const RangeLists &lists, uint32_t g_lo, uint32_t g_hi);

// One range's deliveries to a vs_record_sink: split at guide borders into pieces of at most `target` records (a single guide
// denser than that goes alone), each merged with guide ids offset by lo and handed to the sink; SINK_ABORTED when it returned
// non-zero (no further call is made).  A range without records is one delivery with n = 0.
int deliver_pieces(const RangeLists &lists, uint32_t lo, uint32_t hi, uint64_t target, bool windows, int n_threads,
                   vs_record_sink sink, void *user, std::vector<vs_record> &rec, std::vector<uint64_t> &win, uint64_t *key16_collisions);

// Split [0, n_words) into n contiguous shards of (almost) equal size, tile-aligned.
std::vector<uint64_t> shard_bounds(uint64_t n_words, int n);

// Shards of a text scanned on n_devices devices: shard_bounds with n_devices shards for a text within 4 Gbases; beyond,
// max(n_devices, the fewest shards of at most VS_MAX_SHARD_WORDS words) shards, rounded up to a multiple of n_devices
// (device i scans shards [i, i + 1) * count / n_devices one after the other).
std::vector<uint64_t> shard_plan(uint64_t n_words, int n_devices);

// ---- device memory of resident shards (vs_mapper) ----
// Bytes of device memory a context holds now: the sum of its buffer capacities.
uint64_t ctx_device_bytes(const vs_ctx *ctx);

// A shard as the memory estimate sees it: its words, the contigs that overlap it, and the run (or sparse mask) entries its
// upload stages on the device.
struct ShardShape {
    uint64_t words = 0, contigs = 0, staged = 0;
};
// Scan scratch the estimate allows every context: a pass that keeps up to this many hits, of up to this many guides.  A denser
// scan grows its buffers beyond the estimate (and fails with VS_ERR_CUDA when the device has no room left).
constexpr uint64_t RESIDENT_SCRATCH_HITS = 16ull << 20;
constexpr uint64_t RESIDENT_SCRATCH_GUIDES = 4096;
// Upper bound of the device memory of a context that holds the shard resident with both candidate stores (plain and bucketed)
// for n_pam PAM dinucleotides per strand and scans with the scratch above.  The stores are sized for the expected candidate
// density + 15 %, as the scan sizes them; a text far from uniform may regrow them beyond it.
uint64_t resident_shard_bytes(const ShardShape &shard, uint64_t text_words, int n_pam);
// The shards of a plan dealt to free_bytes.size() devices in contiguous runs, as for_each_shard deals them: need[i] = the bytes
// device i's shards take at the densest PAM set (GG, GA and a -P dinucleotide: 3 of 16 per strand).  Returns the first device
// whose need exceeds its free bytes, or -1 when every device has room.
int resident_plan_check(const std::vector<ShardShape> &shards, uint64_t text_words, const std::vector<uint64_t> &free_bytes,
                        std::vector<uint64_t> &need);
// free device memory (cudaMemGetInfo) of a device
int device_free_bytes(int device, uint64_t *free_bytes);

}  // namespace vs
