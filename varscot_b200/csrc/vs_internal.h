// varscot_b200/csrc/vs_internal.h — helpers shared by the host and device halves of libvarscot_scan.
#pragma once
#include "../../include/varscot_scan.h"
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

// The same with every shard's hits resolved to (contig, pos) and sorted on its device (vs_scan_resolved): one list per
// shard, in shard order, ready for vs_merge_resolved.
int scan_text_sharded_resolved(const vs_text_view &text, const std::vector<int> &devices,
                               const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                               std::vector<std::vector<vs_loc_hit>> &lists, vs_scan_stats *agg, std::string &err);

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
