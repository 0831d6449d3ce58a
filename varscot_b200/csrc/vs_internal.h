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

}  // namespace vs
