// The (query, probe) grouping of the IVF scans (ivfflat.cu, binary.cu, ivfpq.cu): the nq * nprobe pairs sorted by list, work
// items (list, block of <= qb of its queries, chunk of its rows) taken by persistent CTAs from a device counter, and the
// merge levels of the partial lists.
//
//   ivf_probe_keys / radix sort  the pairs sorted by list id (stable: the queries of a list stay in ascending pair
//                                order);
//   ivf_list_items / scan        per list: its first sorted pair and its number of work items
//                                ceil(queries / qb) * chunks; exclusive scan -> item offsets;
//   decode_item                  work item -> (list, query block, row chunk);
//   merge_levels                 the nprobe * S partial lists of each query joined with ise_topk_merge, in levels of at
//                                most 256 lists.
// A list of len rows is cut into min(S, ceil(len / cb)) chunks of a granule of cb rows.  S is capped at 256 / nprobe
// (one merge level while nprobe <= 256) and by the caller's partial-list or segment budget.
#pragma once

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "common.cuh"

namespace {
namespace ivf {

constexpr int kThreads = 128;       // threads of every IVF scan kernel
constexpr int kMergeFanIn = 256;    // ise_topk_merge: at most 256 lists per row
constexpr int64_t kPartialBudget = int64_t(1) << 24;   // search: partial-list entries
constexpr int64_t kSegmentBudget = int64_t(1) << 22;   // range search: (pair, chunk) segments

static inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

static inline uint8_t* take(uint8_t*& w, size_t bytes) {
    uint8_t* r = w;
    w += bytes;
    return r;
}

__host__ __device__ __forceinline__ int64_t list_chunks(int64_t len, int S, int64_t cb) {
    return len == 0 ? 1 : (int64_t)min((int64_t)S, (len + cb - 1) / cb);
}

// a pair without a list (probe -1) sorts after every list and gets no work item: its partial slots are marked empty
__global__ void ivf_probe_keys_kernel(const int64_t* __restrict__ probes, int64_t nq, int nprobe, int64_t nlist, int S,
                                      int topk, int32_t* __restrict__ keys, int32_t* __restrict__ vals,
                                      int64_t* __restrict__ part_idx) {
    const int64_t npairs = nq * nprobe;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npairs; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t l = probes[i];
        const bool ok = l >= 0 && l < nlist;
        keys[i] = ok ? (int32_t)l : (int32_t)nlist;
        vals[i] = (int32_t)i;
        if (!ok && part_idx)
            for (int c = 0; c < S; ++c) part_idx[(((i % nprobe) * S + c) * nq + i / nprobe) * topk] = -1;
    }
}

__device__ __forceinline__ int64_t lower_bound_i32(const int32_t* __restrict__ a, int64_t n, int32_t key) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// qoff[l] = first sorted pair of list l (qoff[nlist] = number of valid pairs); items[l] = work items of list l
__global__ void ivf_list_items_kernel(const int32_t* __restrict__ keys_sorted, int64_t npairs,
                                      const int64_t* __restrict__ list_off, int64_t nlist, int S, int64_t cb, int qb,
                                      int32_t* __restrict__ qoff, int64_t* __restrict__ items) {
    for (int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; l <= nlist; l += (int64_t)gridDim.x * blockDim.x) {
        const int64_t lo = lower_bound_i32(keys_sorted, npairs, (int32_t)l);
        qoff[l] = (int32_t)lo;
        if (l == nlist) {
            items[l] = 0;
        } else {
            const int64_t nql = lower_bound_i32(keys_sorted, npairs, (int32_t)(l + 1)) - lo;
            items[l] = nql ? (nql + qb - 1) / qb * list_chunks(list_off[l + 1] - list_off[l], S, cb) : 0;
        }
    }
}

struct Item {
    int64_t lbase, nch, c;              // first row of the list, its chunks, this item's chunk
    int64_t v_begin, v_end;             // the chunk's rows, in list positions
};

// work item w of the persistent loop: its list (item_off[l] <= w < item_off[l + 1]), query block and row chunk; the
// block's qb pairs go to s_pair (-1 past the block).  The caller synchronises before reading s_pair.
__device__ __forceinline__ Item decode_item(int64_t w, const int64_t* __restrict__ list_off, int64_t nlist,
                                            const int32_t* __restrict__ pairs_sorted, const int32_t* __restrict__ qoff,
                                            const int64_t* __restrict__ item_off, int S, int64_t cb, int qb, int tid,
                                            int* s_pair) {
    int64_t lo = 0, hi = nlist;
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (item_off[mid] <= w) lo = mid;
        else hi = mid;
    }
    const int64_t l = lo;
    Item it;
    it.lbase = list_off[l];
    const int64_t len = list_off[l + 1] - it.lbase;
    const int64_t nch = list_chunks(len, S, cb);
    const int64_t local = w - item_off[l];
    const int64_t qblk = local / nch;
    it.nch = nch;
    it.c = local % nch;
    const int64_t p0 = qoff[l] + qblk * qb;
    const int nqb = (int)min((int64_t)qb, (int64_t)qoff[l + 1] - p0);
    if (tid < qb) s_pair[tid] = tid < nqb ? pairs_sorted[p0 + tid] : -1;
    const int64_t cl = (len + nch - 1) / nch;
    it.v_begin = min(len, it.c * cl);
    it.v_end = min(len, it.v_begin + cl);
    return it;
}

struct Plan {
    int S;                 // chunks per list (partial-list / segment slots per probe)
    int64_t cb, npairs, g; // chunk granule (rows); nq * nprobe; slots per query = nprobe * S
    int qb;                // pairs per work item
    int end_bit;           // radix-sort key bits (list ids 0 .. nlist)
    size_t sort_tmp, scan_tmp, pairs, lists, grouping;
    size_t parts, level;   // search: partial lists and merge levels
    int64_t segs;          // range: nq * nprobe * S (pair, chunk) segments
    size_t seg, lims_tmp;  // range: one int64 per segment + 1 (counts, offsets); ise_range_lims scratch
};

// the grouping both searches share; S covers the longest list, stays <= 256 / nprobe and <= room
static Plan make_plan(int64_t nq, int nprobe, int64_t nlist, int64_t max_list_len, int64_t room, int64_t cb, int qb) {
    Plan p{};
    p.cb = cb;
    p.qb = qb;
    const int64_t need = std::max<int64_t>(1, ceil_div64(max_list_len, cb));
    // a query's nprobe * S partial lists fit one merge while nprobe <= 256: beyond 256 / nprobe chunks per list the
    // (list, query block) items already fill the machine and more chunks only add merge levels
    const int64_t one_merge = std::max<int64_t>(1, kMergeFanIn / nprobe);
    p.S = (int)std::min({need, std::max<int64_t>(1, room), one_merge});
    p.npairs = nq * nprobe;
    p.g = (int64_t)nprobe * p.S;
    p.end_bit = 1;
    while (p.end_bit < 31 && ((int64_t)1 << p.end_bit) <= nlist) ++p.end_bit;
    cub::DeviceRadixSort::SortPairs(nullptr, p.sort_tmp, (const int32_t*)nullptr, (int32_t*)nullptr,
                                    (const int32_t*)nullptr, (int32_t*)nullptr, (int)p.npairs, 0, p.end_bit);
    cub::DeviceScan::ExclusiveSum(nullptr, p.scan_tmp, (const int64_t*)nullptr, (int64_t*)nullptr, (int)(nlist + 1));
    p.pairs = align256((size_t)p.npairs * sizeof(int32_t));
    p.lists = align256((size_t)(nlist + 1) * sizeof(int64_t));
    p.grouping = 4 * p.pairs + align256(p.sort_tmp) + 3 * p.lists + align256(p.scan_tmp) + 256;
    return p;
}

static inline size_t level_entries(const Plan& p, int64_t nq, int topk) {
    return p.g > kMergeFanIn ? (size_t)ceil_div64(p.g, kMergeFanIn) * nq * topk : 0;
}

// search: nq * nprobe * S * topk partial-list entries (float value, int64 id) and the merge levels' 1/256 of that
static Plan search_plan(int64_t nq, int nprobe, int64_t nlist, int64_t max_list_len, int topk, int64_t cb, int qb) {
    Plan p = make_plan(nq, nprobe, nlist, max_list_len, kPartialBudget / std::max<int64_t>(1, nq * nprobe * (int64_t)topk),
                       cb, qb);
    const size_t entries = (size_t)p.g * nq * topk;
    p.parts = align256(entries * sizeof(float)) + align256(entries * sizeof(int64_t));
    const size_t lv = level_entries(p, nq, topk);
    p.level = align256(lv * sizeof(float)) + align256(lv * sizeof(int64_t));
    return p;
}

// range search: a count and an offset per (pair, chunk) segment, and the offsets scan's scratch
static Plan range_plan(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist, int64_t max_list_len, int64_t cb, int qb) {
    Plan p = make_plan(nq, nprobe, nlist, max_list_len, kSegmentBudget / std::max<int64_t>(1, nq * nprobe), cb, qb);
    p.segs = p.g * nq;
    p.seg = align256((size_t)(p.segs + 1) * sizeof(int64_t));
    p.lims_tmp = align256(ise_range_lims_workspace_bytes(ctx, p.segs));
    return p;
}

static bool plan_args_ok(int64_t nq, int nprobe, int64_t nlist, int64_t max_list_len, int topk) {
    return nq > 0 && nprobe >= 1 && nlist >= 1 && nlist < ((int64_t)1 << 30) && max_list_len >= 0 && topk >= 1 &&
           topk <= 128 && nq * nprobe < ((int64_t)1 << 31);
}

struct Grouping {
    int32_t *keys, *keys_sorted, *vals, *pairs_sorted, *qoff;
    int64_t *items, *item_off;
    void *sort_tmp, *scan_tmp;
    unsigned long long* counter;   // next work item of the persistent kernels
};

// the first p.grouping bytes of a workspace
static Grouping carve_grouping(uint8_t*& w, const Plan& p) {
    Grouping g;
    g.keys = reinterpret_cast<int32_t*>(take(w, p.pairs));
    g.keys_sorted = reinterpret_cast<int32_t*>(take(w, p.pairs));
    g.vals = reinterpret_cast<int32_t*>(take(w, p.pairs));
    g.pairs_sorted = reinterpret_cast<int32_t*>(take(w, p.pairs));
    g.sort_tmp = take(w, align256(p.sort_tmp));
    g.qoff = reinterpret_cast<int32_t*>(take(w, p.lists));
    g.items = reinterpret_cast<int64_t*>(take(w, p.lists));
    g.item_off = reinterpret_cast<int64_t*>(take(w, p.lists));
    g.scan_tmp = take(w, align256(p.scan_tmp));
    g.counter = reinterpret_cast<unsigned long long*>(take(w, 256));
    return g;
}

// groups the (query, probe slot) pairs by list and numbers the work items; zeroes the item counter.  part_idx (search
// only, else null): the partial lists of pairs without a list are marked empty.
static int group_pairs(ise_ctx* ctx, const Plan& p, const Grouping& g, const int64_t* probes, int64_t nq, int nprobe,
                       int64_t nlist, const int64_t* list_off, int topk, int64_t* part_idx, cudaStream_t st) {
    ISE_CUDA(cudaMemsetAsync(g.counter, 0, sizeof(unsigned long long), st));
    const int grid_pairs = (int)std::min<int64_t>(ceil_div64(p.npairs, 256), (int64_t)ctx->sm_count * 8);
    ivf_probe_keys_kernel<<<grid_pairs, 256, 0, st>>>(probes, nq, nprobe, nlist, p.S, topk, g.keys, g.vals, part_idx);
    ISE_LAUNCH_CHECK();
    size_t sort_bytes = p.sort_tmp;
    ISE_CUDA(cub::DeviceRadixSort::SortPairs(g.sort_tmp, sort_bytes, g.keys, g.keys_sorted, g.vals, g.pairs_sorted,
                                             (int)p.npairs, 0, p.end_bit, st));
    const int grid_lists = (int)std::min<int64_t>(ceil_div64(nlist + 1, 256), (int64_t)ctx->sm_count * 8);
    ivf_list_items_kernel<<<grid_lists, 256, 0, st>>>(g.keys_sorted, p.npairs, list_off, nlist, p.S, p.cb, p.qb, g.qoff,
                                                      g.items);
    ISE_LAUNCH_CHECK();
    size_t scan_bytes = p.scan_tmp;
    ISE_CUDA(cub::DeviceScan::ExclusiveSum(g.scan_tmp, scan_bytes, g.items, g.item_off, (int)(nlist + 1), st));
    return 0;
}

// persistent CTAs (as many as fit with shm bytes of dynamic shared memory each) that take work items from the counter:
// the item count stays on the device
template <typename Kernel, typename... Args>
static int launch_persistent_shm(ise_ctx* ctx, cudaStream_t st, size_t shm, Kernel kernel, Args... args) {
    int per_sm = 0;
    ISE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, shm));
    kernel<<<ctx->sm_count * std::max(per_sm, 1), kThreads, shm, st>>>(args...);
    ISE_LAUNCH_CHECK();
    return 0;
}

template <typename Kernel, typename... Args>
static int launch_persistent(ise_ctx* ctx, cudaStream_t st, Kernel kernel, Args... args) {
    return launch_persistent_shm(ctx, st, 0, kernel, args...);
}

// merges the nprobe * S partial lists of every query (part_*, list-major [g][nq][topk]) into out_*, at most kMergeFanIn
// at a time; lvl_* hold level_entries(p) entries.  part_* are overwritten.
static int merge_levels(ise_ctx* ctx, const Plan& p, int64_t nq, int topk, int metric, float* part_val,
                        int64_t* part_idx, float* lvl_val, int64_t* lvl_idx, float* out_val, int64_t* out_idx,
                        void* stream) {
    float* src_val = part_val;
    int64_t* src_idx = part_idx;
    float* dst_val = lvl_val;
    int64_t* dst_idx = lvl_idx;
    int64_t g = p.g;
    const size_t list_stride = (size_t)nq * topk;
    while (g > kMergeFanIn) {
        const int64_t g2 = ceil_div64(g, kMergeFanIn);
        for (int64_t j = 0; j < g2; ++j) {
            const int n = (int)std::min<int64_t>(kMergeFanIn, g - j * kMergeFanIn);
            const size_t in = (size_t)j * kMergeFanIn * list_stride, out = (size_t)j * list_stride;
            const int rc = ise_topk_merge(ctx, src_val + in, src_idx + in, n, nq, topk, metric, dst_val + out,
                                          dst_idx + out, stream);
            if (rc) return rc;
        }
        std::swap(src_val, dst_val);
        std::swap(src_idx, dst_idx);
        g = g2;
    }
    return ise_topk_merge(ctx, src_val, src_idx, (int)g, nq, topk, metric, out_val, out_idx, stream);
}

struct RangeWork {
    Plan p;
    Grouping gr;
    int64_t *cnt, *offs;   // per (pair, chunk) segment: hits, output offset (offs[segs] = total)
    void* lims_tmp;
};

// the range workspace of plan p: grouping, counts, offsets, offsets-scan scratch
static RangeWork carve_range(void* workspace, const Plan& p) {
    RangeWork rw;
    rw.p = p;
    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    rw.gr = carve_grouping(w, p);
    rw.cnt = reinterpret_cast<int64_t*>(take(w, p.seg));
    rw.offs = reinterpret_cast<int64_t*>(take(w, p.seg));
    rw.lims_tmp = take(w, p.lims_tmp);
    return rw;
}

static inline size_t range_workspace(const Plan& p) { return p.grouping + 2 * p.seg + p.lims_tmp; }

}  // namespace ivf
}  // namespace

int ise_internal_range_offsets(const int64_t* cnt, int64_t rows, int64_t per_row, int64_t base,
                               int64_t* offs, int64_t* lims, void* tmp, size_t tmp_bytes, void* stream);   // range.cu
