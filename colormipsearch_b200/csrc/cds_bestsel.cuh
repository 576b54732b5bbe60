// cds_bestsel.cuh -- ColorMIPProcessUtils.selectBestMatches on the device (SURVEY.md 8f, row f1): the per-mask selection of the
// top lines, samples and matches out of a device list of passing pairs, computed by radix sorts and segmented scans instead of
// the host's hash maps (csrc/cds_select.cpp defines the order; include/cdsgpu.h restates it).
#ifndef CDS_BESTSEL_CUH
#define CDS_BESTSEL_CUH

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "cds_runtime.h"

namespace cds {

// bytes per pair of the per-device list of passing pairs (topk key + mask)
constexpr int64_t kBestPairBytes = 12;

// The group keys of cds_target_groups copied to one device (freed through its pool by release()).
struct DevGroups {
    int32_t *line = nullptr, *sample = nullptr, *line_hash = nullptr, *sample_hash = nullptr;
    void release(DevState &ds);
};

// Host-side checks of `g` for n_targets targets (NULL pointers, ids outside [0, n_lines) / [0, n_samples)); "" when fine.
std::string check_target_groups(const cds_target_groups *g, int64_t n_targets);
cds_status upload_target_groups(cds_ctx *ctx, DevState &ds, const cds_target_groups *g, int64_t n_targets, DevGroups &out);

// keys of a resident library carry shard-local target indices: make them global (block-cyclic, kLibBlock targets)
void launch_bestsel_globalize(uint64_t *keys, int64_t n, int dev, int n_dev, cudaStream_t s);

// Keeps, of the n pairs in keys / masks (any order), the first top_matches (> 0) of every (mask, line, sample) in key order,
// packed at the front of the same arrays; *counter and n receive the new count.  Blocks the host until it is known.  The keys'
// targets are shard `dev`'s local indices of a library over n_dev devices (the groups are indexed globally); 0, 1 = already global.
cds_status bestsel_compact(cds_ctx *ctx, DevState &ds, uint64_t *keys, int32_t *masks, int64_t &n, unsigned long long *counter,
                           const DevGroups &groups, int32_t top_matches, int dev, int n_dev);

// Where the selected pairs go: the fields of a search (mask, target, score, mirrored) or, for the test hook, positions in the list.
struct BestSelOut {
    int64_t capacity = 0;
    int32_t *mask = nullptr;
    int64_t *target = nullptr;
    int32_t *score = nullptr;
    uint8_t *mirrored = nullptr;
    int64_t *selected = nullptr;
    int64_t *count = nullptr;
};

// The selection over the n pairs of keys / masks on device ds for masks 0 .. n_masks - 1.  `presorted`: the list is already in
// (mask, key) order (the test hook); otherwise it is sorted first.  Only the selected entries and their count reach the host;
// CDS_ERR_CAPACITY (nothing written, *out.count set) when more than out.capacity are selected.
cds_status bestsel_select(cds_ctx *ctx, DevState &ds, const uint64_t *keys, const int32_t *masks, int64_t n, int32_t n_masks, bool presorted,
                          const DevGroups &groups, int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                          const BestSelOut &out);

}  // namespace cds
#endif
