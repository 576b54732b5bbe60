// cds_bestsel.cu -- the reference's best-matches selection (ColorMIPProcessUtils.selectBestMatches,
// colormipsearch-tools/.../cmd/cdsprocess/ColorMIPProcessUtils.java:12-34; two nested ItemsHandling.selectTopRankedElements,
// colormipsearch-api/.../results/ItemsHandling.java:80-109) on the device, over the list of passing pairs a search collected.
//
// csrc/cds_select.cpp is the host restatement this file reproduces bit for bit.  Its hash maps become sorts: with the pairs of a
// mask in encounter order (position p = score descending, target ascending), a group (line of a mask, or sample of a kept line)
// is ranked by (best score desc, HashMap bucket asc, first position asc), where best / first come from the group's first pair and
// the bucket from the Java hash of its key and the table size the number of distinct groups of its parent implies.  Per level:
//   - stable radix sort of the pairs by (parent, group id, p) and run heads -> one record per group, and its parent's group count;
//   - two stable radix sorts of the records by (bucket, first), then (parent, best desc) -> the rank of every group in its parent;
// and at the end the kept pairs sorted by (sample slot, p), which is the reference's output order.  No host pass over the list.
#include <cub/cub.cuh>

#include <algorithm>
#include <climits>
#include <cstdio>
#include <string>
#include <vector>

#include "cds_bestsel.cuh"
#include "cds_topk.cuh"

using namespace cds;

#define CDS_TRY(expr) do { cds_status _s = (expr); if (_s != CDS_OK) return _s; } while (0)
#define CDS_CUDA(ctx, expr) CDS_TRY((ctx)->check((expr), #expr))

namespace {

constexpr int kThreads = 256;
constexpr uint64_t kNone = ~0ull;        // sorts behind every real key

inline unsigned grid_for(int64_t n) { return (unsigned) std::max<int64_t>(1, (n + kThreads - 1) / kThreads); }

__device__ __forceinline__ int32_t key_score(uint64_t k) { return 0x3FFFFFFF - (int32_t) (k >> 34); }
__device__ __forceinline__ int64_t key_target(uint64_t k) { return (int64_t) ((k >> 1) & ((1ull << 33) - 1)); }

// java.util.HashMap after n_keys insertions into a default table: capacity 16, doubled while size > 0.75 * capacity;
// bucket = spread(hash) & (capacity - 1)
__device__ __forceinline__ uint32_t hashmap_bucket(int32_t hash, int64_t n_keys)
{
    uint64_t cap = 16;
    while ((uint64_t) n_keys * 4 > cap * 3) cap <<= 1;
    const uint32_t h = (uint32_t) hash;
    return (uint32_t) ((uint64_t) (h ^ (h >> 16)) & (cap - 1));
}

// one atomic per warp: slot of this lane's item among those appended by the warp
__device__ __forceinline__ unsigned long long warp_append(unsigned long long *counter, bool pass)
{
    const unsigned bal = __ballot_sync(0xffffffffu, pass);
    const int lane = threadIdx.x & 31;
    if (bal == 0) return 0;
    const int leader = __ffs((int) bal) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(counter, (unsigned long long) __popc(bal));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (unsigned long long) __popc(bal & ((1u << lane) - 1u));
}

// global index of target `local` of shard `dev` of a library spread block-cyclically over n_dev devices (cds_library::global_of);
// dev 0 of 1 is the identity, for lists that already hold global indices
__device__ __forceinline__ int64_t global_target(int64_t local, int dev, int n_dev)
{
    return ((local / kLibBlock) * n_dev + dev) * kLibBlock + local % kLibBlock;
}

__global__ void bestsel_globalize_kernel(uint64_t *keys, int64_t n, int dev, int n_dev)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = keys[i];
    const int64_t g = global_target(key_target(k), dev, n_dev);
    keys[i] = (k & ~(((1ull << 33) - 1) << 1)) | ((uint64_t) g << 1);
}

// level 1 input: (mask << 32 | line of the target) of every position, value = position
__global__ void bestsel_line_keys_kernel(const uint64_t *__restrict__ K, const int32_t *__restrict__ Mk, int64_t n,
                                         const int32_t *__restrict__ line, uint64_t *__restrict__ key_out, int32_t *__restrict__ val_out)
{
    const int64_t p = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (p >= n) return;
    key_out[p] = ((uint64_t) (uint32_t) Mk[p] << 32) | (uint32_t) line[key_target(K[p])];
    val_out[p] = (int32_t) p;
}

__global__ void bestsel_heads_kernel(const uint64_t *__restrict__ keys, int64_t n, int32_t *__restrict__ flags)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = keys[i];
    flags[i] = k != kNone && (i == 0 || keys[i - 1] != k);
}

// one record per run of equal keys (key = parent << 32 | group id, value = position): parent, id, first position, index of the
// run's head, best score; count[parent] = number of groups of the parent
__global__ void bestsel_groups_kernel(const uint64_t *__restrict__ keys, const int32_t *__restrict__ vals, const int32_t *__restrict__ flags,
                                      const int32_t *__restrict__ seg, int64_t n, const uint64_t *__restrict__ K,
                                      int32_t *__restrict__ g_parent, int32_t *__restrict__ g_id, int32_t *__restrict__ g_first,
                                      int32_t *__restrict__ g_start, int32_t *__restrict__ g_best, int32_t *__restrict__ count)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n || !flags[i]) return;
    const int gi = seg[i] - 1;
    const uint64_t k = keys[i];
    const int32_t parent = (int32_t) (k >> 32);
    const int32_t p = vals[i];
    g_parent[gi] = parent;
    g_id[gi] = (int32_t) (uint32_t) k;
    g_first[gi] = p;
    g_start[gi] = (int32_t) i;
    g_best[gi] = key_score(K[p]);
    atomicAdd(&count[parent], 1);
}

// first ranking pass: (HashMap bucket, first position); records past the group count sort last
__global__ void bestsel_rank_key1_kernel(const int32_t *__restrict__ n_groups, int64_t n, const int32_t *__restrict__ g_parent,
                                         const int32_t *__restrict__ g_id, const int32_t *__restrict__ g_first, const int32_t *__restrict__ count,
                                         const int32_t *__restrict__ hash, uint64_t *__restrict__ key, int32_t *__restrict__ val)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    val[i] = (int32_t) i;
    if (i >= *n_groups) { key[i] = kNone; return; }
    const uint32_t bucket = hashmap_bucket(hash[g_id[i]], count[g_parent[i]]);
    key[i] = ((uint64_t) bucket << 32) | (uint32_t) g_first[i];
}

// second (stable) ranking pass: (parent, best score descending)
__global__ void bestsel_rank_key2_kernel(const int32_t *__restrict__ n_groups, int64_t n, const int32_t *__restrict__ perm,
                                         const int32_t *__restrict__ g_parent, const int32_t *__restrict__ g_best, uint64_t *__restrict__ key)
{
    const int64_t j = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (j >= n) return;
    if (j >= *n_groups) { key[j] = kNone; return; }
    const int gi = perm[j];
    key[j] = ((uint64_t) (uint32_t) g_parent[gi] << 32) | (uint32_t) (0x3FFFFFFF - g_best[gi]);
}

// slot of a group = its place in the ranked order of all groups when it is among the first `limit` of its parent, else -1
__global__ void bestsel_slots_kernel(const int32_t *__restrict__ n_groups, int64_t n, const int32_t *__restrict__ order,
                                     const int32_t *__restrict__ g_parent, const int32_t *__restrict__ off, int32_t limit, int32_t *__restrict__ slot)
{
    const int64_t r = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (r >= n || r >= *n_groups) return;
    const int gi = order[r];
    const int64_t rank = r - off[g_parent[gi]];
    slot[gi] = (limit <= 0 || rank < limit) ? (int32_t) r : -1;
}

// pairs in (mask, line, position) order -> level 2 input by position: (line slot << 32 | sample) for the pairs of kept lines
__global__ void bestsel_sample_keys_kernel(const int32_t *__restrict__ vals, const int32_t *__restrict__ seg, int64_t n,
                                           const int32_t *__restrict__ slot, const uint64_t *__restrict__ K, const int32_t *__restrict__ sample,
                                           uint64_t *__restrict__ key_out, int32_t *__restrict__ val_out)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int32_t p = vals[i];
    const int32_t ls = slot[seg[i] - 1];
    key_out[p] = ls >= 0 ? (((uint64_t) (uint32_t) ls << 32) | (uint32_t) sample[key_target(K[p])]) : kNone;
    val_out[p] = p;
}

// pairs in (line slot, sample, position) order -> (sample slot << 32 | position) of the selected ones; *n_sel counts them
__global__ void bestsel_final_keys_kernel(const uint64_t *__restrict__ keys, const int32_t *__restrict__ vals, const int32_t *__restrict__ seg,
                                          int64_t n, const int32_t *__restrict__ slot, const int32_t *__restrict__ g_start, int32_t top_matches,
                                          uint64_t *__restrict__ out, unsigned long long *__restrict__ n_sel)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    bool keep = false;
    if (i < n) {
        if (keys[i] != kNone) {
            const int gi = seg[i] - 1;
            const int32_t ss = slot[gi];
            keep = ss >= 0 && (top_matches <= 0 || i - g_start[gi] < top_matches);
            out[i] = keep ? (((uint64_t) (uint32_t) ss << 32) | (uint32_t) vals[i]) : kNone;
        } else {
            out[i] = kNone;
        }
    }
    const int kept = __syncthreads_count(keep);
    if (threadIdx.x == 0 && kept) atomicAdd(n_sel, (unsigned long long) kept);
}

__global__ void bestsel_output_kernel(const uint64_t *__restrict__ fk, const unsigned long long *__restrict__ n_sel, const uint64_t *__restrict__ K,
                                      const int32_t *__restrict__ Mk, int32_t *__restrict__ o_mask, int64_t *__restrict__ o_target,
                                      int32_t *__restrict__ o_score, uint8_t *__restrict__ o_mir, int64_t *__restrict__ o_pos)
{
    const int64_t j = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if ((unsigned long long) j >= *n_sel) return;
    const int32_t p = (int32_t) (uint32_t) fk[j];
    if (o_pos) { o_pos[j] = p; return; }
    const uint64_t k = K[p];
    o_mask[j] = Mk[p];
    o_target[j] = key_target(k);
    o_score[j] = key_score(k);
    o_mir[j] = (uint8_t) (k & 1);
}

// compaction: the sample of every pair (keys in key order), value = index
__global__ void bestsel_cmp_sample_kernel(const uint64_t *__restrict__ Ks, int64_t n, const int32_t *__restrict__ sample, int dev, int n_dev,
                                          uint32_t *__restrict__ key_out, int32_t *__restrict__ val_out)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    key_out[i] = (uint32_t) sample[global_target(key_target(Ks[i]), dev, n_dev)];
    val_out[i] = (int32_t) i;
}

__global__ void bestsel_cmp_mask_line_kernel(const int32_t *__restrict__ perm, const uint64_t *__restrict__ Ks, const int32_t *__restrict__ Ms,
                                             int64_t n, const int32_t *__restrict__ line, int dev, int n_dev, uint64_t *__restrict__ key_out)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int32_t q = perm[i];
    key_out[i] = ((uint64_t) (uint32_t) Ms[q] << 32) | (uint32_t) line[global_target(key_target(Ks[q]), dev, n_dev)];
}

// (mask, line, sample, key) order: head flags of the (mask, line, sample) runs
__global__ void bestsel_cmp_heads_kernel(const int32_t *__restrict__ perm, const uint64_t *__restrict__ ml, const uint64_t *__restrict__ Ks,
                                         int64_t n, const int32_t *__restrict__ sample, int dev, int n_dev, int32_t *__restrict__ flags)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    flags[i] = i == 0 || ml[i] != ml[i - 1] ||
               sample[global_target(key_target(Ks[perm[i]]), dev, n_dev)] != sample[global_target(key_target(Ks[perm[i - 1]]), dev, n_dev)];
}

__global__ void bestsel_cmp_start_kernel(const int32_t *__restrict__ flags, const int32_t *__restrict__ seg, int64_t n, int32_t *__restrict__ start)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    if (i < n && flags[i]) start[seg[i] - 1] = (int32_t) i;
}

__global__ void bestsel_cmp_keep_kernel(const int32_t *__restrict__ perm, const int32_t *__restrict__ seg, const int32_t *__restrict__ start, int64_t n,
                                        int32_t top_matches, const uint64_t *__restrict__ Ks, const int32_t *__restrict__ Ms,
                                        uint64_t *__restrict__ keys_out, int32_t *__restrict__ masks_out, unsigned long long *__restrict__ counter)
{
    const int64_t i = (int64_t) blockIdx.x * kThreads + threadIdx.x;
    const bool keep = i < n && i - start[seg[i] - 1] < top_matches;
    const unsigned long long slot = warp_append(counter, keep);
    if (keep) {
        const int32_t q = perm[i];
        keys_out[slot] = Ks[q];
        masks_out[slot] = Ms[q];
    }
}

// Device scratch of one selection / compaction, taken from the device's pool and returned to it at the end, once the work queued on
// ds.stream (kernels, copies out of the scratch) is done.
struct Work {
    cds_ctx *ctx;
    DevState &ds;
    std::vector<void *> blocks;
    void *temp = nullptr;
    size_t temp_bytes = 0;
    Work(cds_ctx *c, DevState &d) : ctx(c), ds(d) {}
    ~Work()
    {
        cudaSetDevice(ds.dev);
        cudaStreamSynchronize(ds.stream);
        for (void *b : blocks) ds.pool.free(b);
    }
    template <class T> cds_status get(T *&p, int64_t count)
    {
        void *v = nullptr;
        CDS_CUDA(ctx, ds.pool.alloc(&v, (size_t) std::max<int64_t>(count, 1) * sizeof(T)));
        blocks.push_back(v);
        p = (T *) v;
        return CDS_OK;
    }
    cds_status temp_for(size_t bytes)
    {
        if (bytes <= temp_bytes) return CDS_OK;
        uint8_t *t = nullptr;
        CDS_TRY(get(t, (int64_t) bytes));
        temp = t;
        temp_bytes = bytes;
        return CDS_OK;
    }
    // stable LSD radix sorts (cub)
    template <class K, class V> cds_status sort_pairs(const K *kin, K *kout, const V *vin, V *vout, int64_t n)
    {
        size_t bytes = 0;
        CDS_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, bytes, kin, kout, vin, vout, (int) n, 0, (int) sizeof(K) * 8, ds.stream));
        CDS_TRY(temp_for(bytes));
        CDS_CUDA(ctx, cub::DeviceRadixSort::SortPairs(temp, bytes, kin, kout, vin, vout, (int) n, 0, (int) sizeof(K) * 8, ds.stream));
        return CDS_OK;
    }
    cds_status sort_keys(const uint64_t *kin, uint64_t *kout, int64_t n)
    {
        size_t bytes = 0;
        CDS_CUDA(ctx, cub::DeviceRadixSort::SortKeys(nullptr, bytes, kin, kout, (int) n, 0, 64, ds.stream));
        CDS_TRY(temp_for(bytes));
        CDS_CUDA(ctx, cub::DeviceRadixSort::SortKeys(temp, bytes, kin, kout, (int) n, 0, 64, ds.stream));
        return CDS_OK;
    }
    cds_status inclusive_sum(const int32_t *in, int32_t *out, int64_t n)
    {
        size_t bytes = 0;
        CDS_CUDA(ctx, cub::DeviceScan::InclusiveSum(nullptr, bytes, in, out, (int) n, ds.stream));
        CDS_TRY(temp_for(bytes));
        CDS_CUDA(ctx, cub::DeviceScan::InclusiveSum(temp, bytes, in, out, (int) n, ds.stream));
        return CDS_OK;
    }
    cds_status exclusive_sum(const int32_t *in, int32_t *out, int64_t n)
    {
        size_t bytes = 0;
        CDS_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, (int) n, ds.stream));
        CDS_TRY(temp_for(bytes));
        CDS_CUDA(ctx, cub::DeviceScan::ExclusiveSum(temp, bytes, in, out, (int) n, ds.stream));
        return CDS_OK;
    }
};

// Device bytes per pair of the scratch of a selection (bestsel_select: sorted list 12, sort buffers 24, one ranking level 84, cub's
// alternate sort buffers and scan storage ~16) and of a compaction (bestsel_compact: 72 + cub ~16), with some slack.
constexpr int64_t kSelectBytesPerPair = 144;
constexpr int64_t kCompactBytesPerPair = 96;

// Fails with CDS_ERR_OOM naming the bytes needed when the scratch for n pairs cannot fit in what the device has free.
cds_status check_room(cds_ctx *ctx, DevState &ds, int64_t n, int64_t bytes_per_pair, const char *what)
{
    size_t free_b = 0, total_b = 0;
    CDS_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
    const uint64_t need = (uint64_t) n * (uint64_t) bytes_per_pair + ((uint64_t) 64 << 20);
    const uint64_t have = (uint64_t) free_b + (uint64_t) ds.pool.cached_bytes;
    if (need <= have) return CDS_OK;
    char buf[300];
    snprintf(buf, sizeof buf, "best matches: the %s of %lld pairs needs about %llu bytes of device memory, %llu are available; "
             "a smaller \"best_list_bytes\" with a per-sample limit keeps the list shorter", what, (long long) n,
             (unsigned long long) need, (unsigned long long) have);
    return ctx->fail(CDS_ERR_OOM, buf);
}

// The arrays of one ranking level, sized for n pairs (a level has at most n groups and, at level 2, at most n parents).
struct Level {
    int32_t *flags, *seg, *g_parent, *g_id, *g_first, *g_start, *g_best, *count, *off, *v1, *v1s, *order, *slot;
    uint64_t *k1, *k1s, *k2, *k2s;
    cds_status alloc(Work &w, int64_t n, int64_t n_parents)
    {
        for (int32_t **p : {&flags, &seg, &g_parent, &g_id, &g_first, &g_start, &g_best, &v1, &v1s, &order, &slot}) CDS_TRY(w.get(*p, n));
        CDS_TRY(w.get(count, n_parents));
        CDS_TRY(w.get(off, n_parents));
        for (uint64_t **p : {&k1, &k1s, &k2, &k2s}) CDS_TRY(w.get(*p, n));
        return CDS_OK;
    }
};

// Groups the n pairs given in (parent, group id, position) order (keys / vals), ranks the groups inside their parents and sets
// lv.slot[group] (-1 = cut by `limit`); lv.seg[i] - 1 = group of entry i, lv.g_start[group] = its first entry.
cds_status rank_level(Work &w, Level &lv, const uint64_t *keys, const int32_t *vals, int64_t n, int64_t n_parents, const uint64_t *K,
                      const int32_t *hash, int32_t limit)
{
    cudaStream_t s = w.ds.stream;
    const unsigned g = grid_for(n);
    bestsel_heads_kernel<<<g, kThreads, 0, s>>>(keys, n, lv.flags);
    CDS_TRY(w.inclusive_sum(lv.flags, lv.seg, n));
    CDS_CUDA(w.ctx, cudaMemsetAsync(lv.count, 0, (size_t) n_parents * sizeof(int32_t), s));
    bestsel_groups_kernel<<<g, kThreads, 0, s>>>(keys, vals, lv.flags, lv.seg, n, K, lv.g_parent, lv.g_id, lv.g_first, lv.g_start, lv.g_best, lv.count);
    CDS_TRY(w.exclusive_sum(lv.count, lv.off, n_parents));
    const int32_t *n_groups = lv.seg + n - 1;
    bestsel_rank_key1_kernel<<<g, kThreads, 0, s>>>(n_groups, n, lv.g_parent, lv.g_id, lv.g_first, lv.count, hash, lv.k1, lv.v1);
    CDS_TRY(w.sort_pairs(lv.k1, lv.k1s, lv.v1, lv.v1s, n));
    bestsel_rank_key2_kernel<<<g, kThreads, 0, s>>>(n_groups, n, lv.v1s, lv.g_parent, lv.g_best, lv.k2);
    CDS_TRY(w.sort_pairs(lv.k2, lv.k2s, lv.v1s, lv.order, n));
    bestsel_slots_kernel<<<g, kThreads, 0, s>>>(n_groups, n, lv.order, lv.g_parent, lv.off, limit, lv.slot);
    CDS_CUDA(w.ctx, cudaGetLastError());
    return CDS_OK;
}

}  // namespace

namespace cds {

void DevGroups::release(DevState &ds)
{
    for (int32_t **p : {&line, &sample, &line_hash, &sample_hash}) {
        if (*p) ds.pool.free(*p);
        *p = nullptr;
    }
}

std::string check_target_groups(const cds_target_groups *g, int64_t n_targets)
{
    if (!g) return "groups is NULL";
    if (g->n_lines < 0 || g->n_samples < 0) return "n_lines and n_samples must not be negative";
    if (n_targets > 0 && (!g->line || !g->sample)) return "groups->line / groups->sample is NULL";
    if ((g->n_lines > 0 && !g->line_hash) || (g->n_samples > 0 && !g->sample_hash)) return "groups->line_hash / groups->sample_hash is NULL";
    for (int64_t i = 0; i < n_targets; i++) {
        if (g->line[i] < 0 || g->line[i] >= g->n_lines)
            return "line id " + std::to_string(g->line[i]) + " of target " + std::to_string(i) + " is outside [0, n_lines)";
        if (g->sample[i] < 0 || g->sample[i] >= g->n_samples)
            return "sample id " + std::to_string(g->sample[i]) + " of target " + std::to_string(i) + " is outside [0, n_samples)";
    }
    return "";
}

cds_status upload_target_groups(cds_ctx *ctx, DevState &ds, const cds_target_groups *g, int64_t n_targets, DevGroups &out)
{
    CDS_CUDA(ctx, cudaSetDevice(ds.dev));
    const struct { int32_t **dst; const int32_t *src; int64_t n; } parts[] = {
        {&out.line, g->line, n_targets}, {&out.sample, g->sample, n_targets},
        {&out.line_hash, g->line_hash, g->n_lines}, {&out.sample_hash, g->sample_hash, g->n_samples}};
    for (const auto &pt : parts) {
        CDS_CUDA(ctx, ds.pool.alloc((void **) pt.dst, (size_t) std::max<int64_t>(pt.n, 1) * sizeof(int32_t)));
        if (pt.n > 0) CDS_CUDA(ctx, cudaMemcpyAsync(*pt.dst, pt.src, (size_t) pt.n * sizeof(int32_t), cudaMemcpyHostToDevice, ds.stream));
        ctx->stats.h2d_bytes += pt.n * (int64_t) sizeof(int32_t);
    }
    return CDS_OK;
}

void launch_bestsel_globalize(uint64_t *keys, int64_t n, int dev, int n_dev, cudaStream_t s)
{
    if (n > 0) bestsel_globalize_kernel<<<grid_for(n), kThreads, 0, s>>>(keys, n, dev, n_dev);
}

cds_status bestsel_compact(cds_ctx *ctx, DevState &ds, uint64_t *keys, int32_t *masks, int64_t &n, unsigned long long *counter,
                           const DevGroups &groups, int32_t top_matches, int dev, int n_dev)
{
    if (n <= 0 || top_matches <= 0) return CDS_OK;
    CDS_CUDA(ctx, cudaSetDevice(ds.dev));
    CDS_TRY(check_room(ctx, ds, n, kCompactBytesPerPair, "compaction"));
    cudaStream_t s = ds.stream;
    Work w(ctx, ds);
    uint64_t *Ks, *ml, *mls, *kout;
    int32_t *Ms, *iota, *perm1, *perm2, *flags, *seg, *start, *mout;
    uint32_t *sk, *sks;
    unsigned long long *d_kept;
    for (uint64_t **p : {&Ks, &ml, &mls, &kout}) CDS_TRY(w.get(*p, n));
    for (int32_t **p : {&Ms, &iota, &perm1, &perm2, &flags, &seg, &start, &mout}) CDS_TRY(w.get(*p, n));
    CDS_TRY(w.get(sk, n));
    CDS_TRY(w.get(sks, n));
    CDS_TRY(w.get(d_kept, 1));
    const unsigned g = grid_for(n);
    // (mask, line, sample, key) order by three stable passes
    CDS_TRY(w.sort_pairs(keys, Ks, masks, Ms, n));
    bestsel_cmp_sample_kernel<<<g, kThreads, 0, s>>>(Ks, n, groups.sample, dev, n_dev, sk, iota);
    CDS_TRY(w.sort_pairs(sk, sks, iota, perm1, n));
    bestsel_cmp_mask_line_kernel<<<g, kThreads, 0, s>>>(perm1, Ks, Ms, n, groups.line, dev, n_dev, ml);
    CDS_TRY(w.sort_pairs(ml, mls, perm1, perm2, n));
    bestsel_cmp_heads_kernel<<<g, kThreads, 0, s>>>(perm2, mls, Ks, n, groups.sample, dev, n_dev, flags);
    CDS_TRY(w.inclusive_sum(flags, seg, n));
    bestsel_cmp_start_kernel<<<g, kThreads, 0, s>>>(flags, seg, n, start);
    CDS_CUDA(ctx, cudaMemsetAsync(d_kept, 0, sizeof(unsigned long long), s));
    bestsel_cmp_keep_kernel<<<g, kThreads, 0, s>>>(perm2, seg, start, n, top_matches, Ks, Ms, kout, mout, d_kept);
    CDS_CUDA(ctx, cudaGetLastError());
    unsigned long long kept = 0;
    CDS_CUDA(ctx, cudaMemcpyAsync(&kept, d_kept, sizeof kept, cudaMemcpyDeviceToHost, s));
    CDS_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.d2h_bytes += (int64_t) sizeof kept;
    CDS_CUDA(ctx, cudaMemcpyAsync(keys, kout, (size_t) kept * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
    CDS_CUDA(ctx, cudaMemcpyAsync(masks, mout, (size_t) kept * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    CDS_CUDA(ctx, cudaMemcpyAsync(counter, d_kept, sizeof(unsigned long long), cudaMemcpyDeviceToDevice, s));
    n = (int64_t) kept;
    return CDS_OK;
}

cds_status bestsel_select(cds_ctx *ctx, DevState &ds, const uint64_t *keys, const int32_t *masks, int64_t n, int32_t n_masks, bool presorted,
                          const DevGroups &groups, int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                          const BestSelOut &out)
{
    if (n >= INT_MAX) {
        char buf[200];
        snprintf(buf, sizeof buf, "best matches: %lld passing pairs on one device, the selection handles at most %d", (long long) n, INT_MAX - 1);
        return ctx->fail(CDS_ERR_CAPACITY, buf);
    }
    CDS_CUDA(ctx, cudaSetDevice(ds.dev));
    if (n > 0) CDS_TRY(check_room(ctx, ds, n, kSelectBytesPerPair, "selection"));
    cudaStream_t s = ds.stream;
    Work w(ctx, ds);
    unsigned long long *d_nsel;
    CDS_TRY(w.get(d_nsel, 1));
    CDS_CUDA(ctx, cudaMemsetAsync(d_nsel, 0, sizeof(unsigned long long), s));
    const uint64_t *K = keys;
    const int32_t *Mk = masks;
    uint64_t *fks = nullptr;
    if (n > 0) {
        const unsigned g = grid_for(n);
        uint64_t *ka, *kb;
        int32_t *va, *vb;
        CDS_TRY(w.get(ka, n)); CDS_TRY(w.get(kb, n)); CDS_TRY(w.get(va, n)); CDS_TRY(w.get(vb, n));
        if (!presorted) {
            // (mask, key) order: by key (into ka / va), then stably by mask
            uint64_t *K2;
            int32_t *Ms;
            CDS_TRY(w.get(K2, n)); CDS_TRY(w.get(Ms, n));
            CDS_TRY(w.sort_pairs(keys, ka, masks, va, n));
            CDS_TRY(w.sort_pairs((const int32_t *) va, Ms, (const uint64_t *) ka, K2, n));
            K = K2;
            Mk = Ms;
        }
        // one set of level arrays serves both levels: level 2 reads level 1's result only while it builds its input
        Level lv;
        CDS_TRY(lv.alloc(w, n, std::max<int64_t>(n_masks, n)));
        // level 1: the lines of every mask
        bestsel_line_keys_kernel<<<g, kThreads, 0, s>>>(K, Mk, n, groups.line, ka, va);
        CDS_TRY(w.sort_pairs(ka, kb, va, vb, n));
        CDS_TRY(rank_level(w, lv, kb, vb, n, n_masks, K, groups.line_hash, top_lines));
        // level 2: the samples of every kept line (a line's slot identifies (mask, line))
        bestsel_sample_keys_kernel<<<g, kThreads, 0, s>>>(vb, lv.seg, n, lv.slot, K, groups.sample, ka, va);
        CDS_TRY(w.sort_pairs(ka, kb, va, vb, n));
        CDS_TRY(rank_level(w, lv, kb, vb, n, n, K, groups.sample_hash, top_samples_per_line));
        // matches: the first top_matches of every kept sample, then the output order (sample slot, position)
        bestsel_final_keys_kernel<<<g, kThreads, 0, s>>>(kb, vb, lv.seg, n, lv.slot, lv.g_start, top_matches_per_sample, ka, d_nsel);
        CDS_TRY(w.sort_keys(ka, kb, n));
        CDS_CUDA(ctx, cudaGetLastError());
        fks = kb;
    }
    unsigned long long n_sel = 0;
    CDS_CUDA(ctx, cudaMemcpyAsync(&n_sel, d_nsel, sizeof n_sel, cudaMemcpyDeviceToHost, s));
    CDS_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.d2h_bytes += (int64_t) sizeof n_sel;
    *out.count = (int64_t) n_sel;
    if (n_sel > (unsigned long long) out.capacity) {
        char buf[200];
        snprintf(buf, sizeof buf, "best matches: %llu pairs selected, capacity is %lld", n_sel, (long long) out.capacity);
        return ctx->fail(CDS_ERR_CAPACITY, buf);
    }
    if (n_sel == 0) return CDS_OK;
    const int64_t m = (int64_t) n_sel;
    int32_t *o_mask = nullptr, *o_score = nullptr;
    int64_t *o_target = nullptr, *o_pos = nullptr;
    uint8_t *o_mir = nullptr;
    if (out.selected) {
        CDS_TRY(w.get(o_pos, m));
    } else {
        CDS_TRY(w.get(o_mask, m)); CDS_TRY(w.get(o_target, m)); CDS_TRY(w.get(o_score, m)); CDS_TRY(w.get(o_mir, m));
    }
    bestsel_output_kernel<<<grid_for(m), kThreads, 0, s>>>(fks, d_nsel, K, Mk, o_mask, o_target, o_score, o_mir, o_pos);
    CDS_CUDA(ctx, cudaGetLastError());
    auto down = [&](void *dst, const void *src, size_t bytes) -> cds_status {
        CDS_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s));
        ctx->stats.d2h_bytes += (int64_t) bytes;
        return CDS_OK;
    };
    if (out.selected) {
        CDS_TRY(down(out.selected, o_pos, (size_t) m * sizeof(int64_t)));
    } else {
        CDS_TRY(down(out.mask, o_mask, (size_t) m * sizeof(int32_t)));
        CDS_TRY(down(out.target, o_target, (size_t) m * sizeof(int64_t)));
        CDS_TRY(down(out.score, o_score, (size_t) m * sizeof(int32_t)));
        if (out.mirrored) CDS_TRY(down(out.mirrored, o_mir, (size_t) m));
    }
    CDS_CUDA(ctx, cudaStreamSynchronize(s));
    return CDS_OK;
}

}  // namespace cds

// Test hook: the selection alone over a caller-given list sorted by (mask, score desc, target asc), on the context's first device.
extern "C" cds_status cds_debug_select_best_matches_device(cds_ctx *ctx, const int32_t *mask, const int64_t *target, const int32_t *score,
                                                           const uint8_t *mirrored, int64_t n, const cds_target_groups *groups,
                                                           int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                                           int64_t *selected, int64_t *n_selected)
{
    return cds::abi_guard("cds_debug_select_best_matches_device", [&]() -> cds_status {
        const std::string name = "cds_debug_select_best_matches_device: ";
        auto bad = [&](const std::string &msg) -> cds_status {
            if (!ctx) { set_tls_error(name + msg); return CDS_ERR_BAD_ARG; }
            std::lock_guard<std::recursive_mutex> lk(ctx->mu);
            return ctx->fail(CDS_ERR_BAD_ARG, name + msg);
        };
        if (n < 0 || !n_selected || (n > 0 && (!mask || !target || !score || !selected))) return bad("bad arguments");
        int64_t n_targets = 0;
        int32_t n_masks = 0;
        for (int64_t i = 0; i < n; i++) {
            if (mask[i] < 0 || target[i] < 0 || target[i] >= ((int64_t) 1 << 33) || score[i] < 0 || score[i] > 0x3FFFFFFF)
                return bad("entry " + std::to_string(i) + " out of range");
            if (i > 0 && (mask[i] < mask[i - 1] || (mask[i] == mask[i - 1] && (score[i] > score[i - 1] || (score[i] == score[i - 1] && target[i] <= target[i - 1])))))
                return bad("the list is not sorted by (mask, score desc, target asc) at entry " + std::to_string(i));
            n_targets = std::max(n_targets, target[i] + 1);
            n_masks = std::max(n_masks, mask[i] + 1);
        }
        const std::string err = check_target_groups(groups, n_targets);
        if (!err.empty()) return bad(err);
        if (!ctx) return bad("NULL ctx");
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        ctx->stats = cds_search_stats{};
        *n_selected = 0;
        DevState &ds = ctx->devs[0];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        std::vector<uint64_t> keys((size_t) n);
        for (int64_t i = 0; i < n; i++) keys[i] = topk_make_key(score[i], target[i], mirrored ? mirrored[i] : 0);
        DevGroups dg;
        uint64_t *d_keys = nullptr;
        int32_t *d_masks = nullptr;
        struct Cleanup {
            DevState &ds; DevGroups &dg; uint64_t *&k; int32_t *&m;
            ~Cleanup() { cudaStreamSynchronize(ds.stream); dg.release(ds); if (k) ds.pool.free(k); if (m) ds.pool.free(m); }
        } cleanup{ds, dg, d_keys, d_masks};
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_keys, (size_t) std::max<int64_t>(n, 1) * sizeof(uint64_t)));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_masks, (size_t) std::max<int64_t>(n, 1) * sizeof(int32_t)));
        if (n > 0) {
            CDS_CUDA(ctx, cudaMemcpyAsync(d_keys, keys.data(), (size_t) n * sizeof(uint64_t), cudaMemcpyHostToDevice, ds.stream));
            CDS_CUDA(ctx, cudaMemcpyAsync(d_masks, mask, (size_t) n * sizeof(int32_t), cudaMemcpyHostToDevice, ds.stream));
        }
        CDS_TRY(upload_target_groups(ctx, ds, groups, n_targets, dg));
        BestSelOut out;
        out.capacity = n;
        out.selected = selected;
        out.count = n_selected;
        return bestsel_select(ctx, ds, d_keys, d_masks, n, n_masks, true, dg, top_lines, top_samples_per_line, top_matches_per_sample, out);
    });
}
