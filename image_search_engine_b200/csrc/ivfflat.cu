// IndexIVFFlat search: exact FP32 scan of the probed inverted lists (faiss/IndexIVFFlat.cpp IVFFlatScanner,
// faiss/utils/distances.cpp fvec_inner_product / fvec_L2sqr) without an [nq, ntotal] score matrix.
//
//   ivf_probe_keys / radix sort  the nq * nprobe (query, probe slot) pairs sorted by list id (stable: the queries
//                                of a list stay in ascending pair order);
//   ivf_list_items / scan        per list: its first sorted pair and its number of work items
//                                ceil(queries / kQB) * chunks; exclusive scan -> item offsets;
//   ivfflat_scan_kernel          one work item = (list, block of <= kQB of its queries, chunk of its vectors).  The
//                                block's queries and kCB vectors at a time go through shared memory kDK dimensions at
//                                a time; each thread accumulates a 4 x 4 piece of the kQB x kCB score tile with the
//                                direct formulas (sum x*y, sum (x-y)^2), and four threads per query keep top-k lists
//                                over the chunk, offered in ascending list position (= ascending id);
//   ise_topk_merge               the nprobe * S partial lists of each query (S = chunks per list), in levels of at
//                                most 256 lists.
// Chunking the vectors keeps a long list from serialising onto one CTA and lets a single query (nq = 1) fill more
// than nprobe CTAs.  S is capped at 256 / nprobe (one merge level while nprobe <= 256) and so that the partial lists
// hold at most max(2^24, nq * nprobe * topk) entries.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "common.cuh"
#include "topk_list.cuh"

namespace {

constexpr int kQB = 32;             // queries per work item
constexpr int kCB = 64;             // vectors per score tile
constexpr int kDK = 32;             // dimensions per shared-memory slice
constexpr int kThreads = 128;       // 16 x 8 threads, 4 x 4 scores each
constexpr int kMergeFanIn = 256;    // ise_topk_merge: at most 256 lists per row
constexpr int64_t kPartialBudget = int64_t(1) << 24;

static inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

__host__ __device__ __forceinline__ int64_t list_chunks(int64_t len, int S) {
    return len == 0 ? 1 : (int64_t)min((int64_t)S, (len + kCB - 1) / kCB);
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
        if (!ok)
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
                                      const int64_t* __restrict__ list_off, int64_t nlist, int S,
                                      int32_t* __restrict__ qoff, int64_t* __restrict__ items) {
    for (int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; l <= nlist; l += (int64_t)gridDim.x * blockDim.x) {
        const int64_t lo = lower_bound_i32(keys_sorted, npairs, (int32_t)l);
        qoff[l] = (int32_t)lo;
        if (l == nlist) {
            items[l] = 0;
        } else {
            const int64_t nql = lower_bound_i32(keys_sorted, npairs, (int32_t)(l + 1)) - lo;
            items[l] = nql ? (nql + kQB - 1) / kQB * list_chunks(list_off[l + 1] - list_off[l], S) : 0;
        }
    }
}

// four consecutive columns c .. c+3 of a row (zeros past d or for a missing row); vec: d % 4 == 0, 16-byte rows
__device__ __forceinline__ float4 load4(const float* __restrict__ row, int c, int d, bool vec) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row == nullptr || c >= d) return v;
    if (vec) return __ldg(reinterpret_cast<const float4*>(row + c));
    v.x = __ldg(row + c);
    if (c + 1 < d) v.y = __ldg(row + c + 1);
    if (c + 2 < d) v.z = __ldg(row + c + 2);
    if (c + 3 < d) v.w = __ldg(row + c + 3);
    return v;
}

template <bool L2, int KMAX>
__global__ void __launch_bounds__(kThreads) ivfflat_scan_kernel(
        const float* __restrict__ q, int64_t nq, int d, bool vec, const float* __restrict__ xs,
        const int64_t* __restrict__ ids, const int64_t* __restrict__ list_off, int64_t nlist,
        const int32_t* __restrict__ pairs_sorted, const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off,
        int nprobe, int S, int topk, unsigned long long* __restrict__ counter,
        float* __restrict__ part_val, int64_t* __restrict__ part_idx) {
    __shared__ __align__(16) float s_q[kDK][kQB];
    __shared__ __align__(16) float s_x[kDK][kCB];
    __shared__ float s_s[kQB][kCB + 1];
    __shared__ int s_pair[kQB];
    __shared__ long long s_item;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int sq = tid >> 2, sub = tid & 3;          // selection: four threads per query row of the tile
    const int64_t total = item_off[nlist];
    const float pad = L2 ? 3.402823466e+38f : -3.402823466e+38f;
    for (;;) {
        if (tid == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= total) break;
        int64_t lo = 0, hi = nlist;                  // item_off[lo] <= w < item_off[hi]
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (item_off[mid] <= w) lo = mid;
            else hi = mid;
        }
        const int64_t l = lo;
        const int64_t lbase = list_off[l], len = list_off[l + 1] - lbase;
        const int64_t nch = list_chunks(len, S);
        const int64_t local = w - item_off[l];
        const int64_t qb = local / nch, c = local % nch;
        const int64_t p0 = qoff[l] + qb * kQB;
        const int nqb = (int)min((int64_t)kQB, (int64_t)qoff[l + 1] - p0);
        if (tid < kQB) s_pair[tid] = tid < nqb ? pairs_sorted[p0 + tid] : -1;
        const int64_t cl = (len + nch - 1) / nch;
        const int64_t v_begin = min(len, c * cl), v_end = min(len, v_begin + cl);
        const float* xl = xs + lbase * (int64_t)d;
        __syncthreads();

        TopKList<KMAX> list;
        list.init(topk);
        for (int64_t t0 = v_begin; t0 < v_end; t0 += kCB) {
            const int nv = (int)min((int64_t)kCB, v_end - t0);
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
            for (int d0 = 0; d0 < d; d0 += kDK) {
                for (int e = tid; e < kQB * (kDK / 4); e += kThreads) {
                    const int r = e / (kDK / 4), c4 = (e % (kDK / 4)) * 4;
                    const int pr = s_pair[r];
                    const float4 v = load4(pr >= 0 ? q + (int64_t)(pr / nprobe) * d : nullptr, d0 + c4, d, vec);
                    s_q[c4][r] = v.x; s_q[c4 + 1][r] = v.y; s_q[c4 + 2][r] = v.z; s_q[c4 + 3][r] = v.w;
                }
                for (int e = tid; e < kCB * (kDK / 4); e += kThreads) {
                    const int r = e / (kDK / 4), c4 = (e % (kDK / 4)) * 4;
                    const float4 v = load4(r < nv ? xl + (t0 + r) * d : nullptr, d0 + c4, d, vec);
                    s_x[c4][r] = v.x; s_x[c4 + 1][r] = v.y; s_x[c4 + 2][r] = v.z; s_x[c4 + 3][r] = v.w;
                }
                __syncthreads();
#pragma unroll
                for (int kk = 0; kk < kDK; ++kk) {
                    const float4 a4 = *reinterpret_cast<const float4*>(&s_q[kk][ty * 4]);
                    const float4 b4 = *reinterpret_cast<const float4*>(&s_x[kk][tx * 4]);
                    const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            if (L2) {
                                const float t = a[i] - b[j];
                                acc[i][j] = fmaf(t, t, acc[i][j]);
                            } else {
                                acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
                            }
                        }
                }
                __syncthreads();
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) s_s[ty * 4 + i][tx * 4 + j] = acc[i][j];
            __syncthreads();
            if (s_pair[sq] >= 0) {
                // ascending column per thread: the strict insert keeps the lower position (= lower id) on ties
                for (int j = sub; j < nv; j += 4) {
                    const float s = L2 ? -s_s[sq][j] : s_s[sq][j];
                    if (s > list.thr) list.insert(s, (int)(t0 + j));
                }
            }
            __syncthreads();
        }

        // merge the four lists of a query row (lanes 4 sq .. 4 sq + 3) and write the partial list of (pair, chunk)
        const int pair = s_pair[sq];
        const int64_t qi = pair >= 0 ? pair / nprobe : 0, slot = pair >= 0 ? pair % nprobe : 0;
        const int64_t obase = ((slot * S + c) * nq + qi) * topk;
        int head = 0;
        for (int j = 0; j < topk; ++j) {
            const bool live = head < topk && list.id[head] >= 0;
            float v = live ? list.v[head] : -CUDART_INF_F;
            int id = live ? list.id[head] : 0x7fffffff;
            int src = sub;
#pragma unroll
            for (int o = 1; o < 4; o <<= 1) {
                const float v2 = __shfl_xor_sync(0xffffffffu, v, o);
                const int id2 = __shfl_xor_sync(0xffffffffu, id, o);
                const int src2 = __shfl_xor_sync(0xffffffffu, src, o);
                if (v2 > v || (v2 == v && id2 < id)) { v = v2; id = id2; src = src2; }
            }
            if (src == sub && id != 0x7fffffff) ++head;
            if (sub == 0 && pair >= 0) {
                part_val[obase + j] = id != 0x7fffffff ? (L2 ? -v : v) : pad;
                part_idx[obase + j] = id != 0x7fffffff ? ids[lbase + id] : -1;
            }
        }
        // chunk slots this list does not use: an id -1 at the head makes ise_topk_merge skip the list
        if (sub == 0 && pair >= 0 && c == nch - 1)
            for (int64_t c2 = nch; c2 < S; ++c2) part_idx[((slot * S + c2) * nq + qi) * topk] = -1;
        __syncthreads();
    }
}

struct Plan {
    int S;                 // chunks per list (partial-list slots per probe)
    int64_t npairs, g;     // nq * nprobe; partial lists per query = nprobe * S
    int end_bit;           // radix-sort key bits (list ids 0 .. nlist)
    size_t sort_tmp, scan_tmp, pairs, lists, parts, level;
};

static Plan make_plan(int64_t nq, int nprobe, int64_t nlist, int64_t max_list_len, int topk) {
    Plan p{};
    const int64_t need = std::max<int64_t>(1, ceil_div64(max_list_len, kCB));
    const int64_t room = std::max<int64_t>(1, kPartialBudget / std::max<int64_t>(1, nq * nprobe * (int64_t)topk));
    // a query's nprobe * S partial lists fit one merge while nprobe <= 256: beyond 256 / nprobe chunks per list the
    // (list, query block) items already fill the machine and more chunks only add merge levels
    const int64_t one_merge = std::max<int64_t>(1, kMergeFanIn / nprobe);
    p.S = (int)std::min({need, room, one_merge});
    p.npairs = nq * nprobe;
    p.g = (int64_t)nprobe * p.S;
    p.end_bit = 1;
    while (p.end_bit < 31 && ((int64_t)1 << p.end_bit) <= nlist) ++p.end_bit;
    cub::DeviceRadixSort::SortPairs(nullptr, p.sort_tmp, (const int32_t*)nullptr, (int32_t*)nullptr,
                                    (const int32_t*)nullptr, (int32_t*)nullptr, (int)p.npairs, 0, p.end_bit);
    cub::DeviceScan::ExclusiveSum(nullptr, p.scan_tmp, (const int64_t*)nullptr, (int64_t*)nullptr, (int)(nlist + 1));
    p.pairs = align256((size_t)p.npairs * sizeof(int32_t));
    p.lists = align256((size_t)(nlist + 1) * sizeof(int64_t));
    const size_t entries = (size_t)p.g * nq * topk;
    p.parts = align256(entries * sizeof(float)) + align256(entries * sizeof(int64_t));
    const size_t lv = p.g > kMergeFanIn ? (size_t)ceil_div64(p.g, kMergeFanIn) * nq * topk : 0;
    p.level = align256(lv * sizeof(float)) + align256(lv * sizeof(int64_t));
    return p;
}

static bool plan_args_ok(int64_t nq, int nprobe, int64_t nlist, int64_t max_list_len, int topk) {
    return nq > 0 && nprobe >= 1 && nlist >= 1 && nlist < ((int64_t)1 << 30) && max_list_len >= 0 && topk >= 1 &&
           topk <= 128 && nq * nprobe < ((int64_t)1 << 31);
}

}  // namespace

ISE_EXPORT size_t ise_ivfflat_search_workspace_bytes(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist,
                                                     int64_t max_list_len, int topk) {
    if (!ctx || !plan_args_ok(nq, nprobe, nlist, max_list_len, topk)) return 0;
    const Plan p = make_plan(nq, nprobe, nlist, max_list_len, topk);
    return 4 * p.pairs + align256(p.sort_tmp) + 3 * p.lists + align256(p.scan_tmp) + 256 + p.parts + p.level;
}

ISE_EXPORT int ise_ivfflat_search(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* xs_sorted,
                                  const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist,
                                  int64_t max_list_len, const int64_t* probes, int nprobe, int metric, int topk,
                                  float* out_val, int64_t* out_idx, void* workspace, size_t workspace_bytes,
                                  void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(nq >= 0 && d > 0 && topk >= 1 && topk <= 128);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(plan_args_ok(nq, nprobe, nlist, max_list_len, topk));
    ISE_CHECK_ARG(q && list_off && probes && out_val && out_idx && workspace);
    ISE_CHECK_ARG(max_list_len == 0 || (xs_sorted && ids_sorted));
    const size_t need = ise_ivfflat_search_workspace_bytes(ctx, nq, nprobe, nlist, max_list_len, topk);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const Plan p = make_plan(nq, nprobe, nlist, max_list_len, topk);

    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    auto take = [&w](size_t bytes) { uint8_t* r = w; w += bytes; return r; };
    int32_t* keys = reinterpret_cast<int32_t*>(take(p.pairs));
    int32_t* keys_sorted = reinterpret_cast<int32_t*>(take(p.pairs));
    int32_t* vals = reinterpret_cast<int32_t*>(take(p.pairs));
    int32_t* pairs_sorted = reinterpret_cast<int32_t*>(take(p.pairs));
    void* sort_tmp = take(align256(p.sort_tmp));
    int32_t* qoff = reinterpret_cast<int32_t*>(take(p.lists));
    int64_t* items = reinterpret_cast<int64_t*>(take(p.lists));
    int64_t* item_off = reinterpret_cast<int64_t*>(take(p.lists));
    void* scan_tmp = take(align256(p.scan_tmp));
    unsigned long long* counter = reinterpret_cast<unsigned long long*>(take(256));
    const size_t entries = (size_t)p.g * nq * topk;
    float* part_val = reinterpret_cast<float*>(take(align256(entries * sizeof(float))));
    int64_t* part_idx = reinterpret_cast<int64_t*>(take(align256(entries * sizeof(int64_t))));
    const size_t lv = p.g > kMergeFanIn ? (size_t)ceil_div64(p.g, kMergeFanIn) * nq * topk : 0;
    float* lvl_val = reinterpret_cast<float*>(take(align256(lv * sizeof(float))));
    int64_t* lvl_idx = reinterpret_cast<int64_t*>(take(align256(lv * sizeof(int64_t))));

    // 1. group the (query, probe slot) pairs by list
    ISE_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), st));
    const int grid_pairs = (int)std::min<int64_t>(ceil_div64(p.npairs, 256), (int64_t)ctx->sm_count * 8);
    ivf_probe_keys_kernel<<<grid_pairs, 256, 0, st>>>(probes, nq, nprobe, nlist, p.S, topk, keys, vals, part_idx);
    ISE_LAUNCH_CHECK();
    size_t sort_bytes = p.sort_tmp;
    ISE_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, keys, keys_sorted, vals, pairs_sorted,
                                             (int)p.npairs, 0, p.end_bit, st));
    const int grid_lists = (int)std::min<int64_t>(ceil_div64(nlist + 1, 256), (int64_t)ctx->sm_count * 8);
    ivf_list_items_kernel<<<grid_lists, 256, 0, st>>>(keys_sorted, p.npairs, list_off, nlist, p.S, qoff, items);
    ISE_LAUNCH_CHECK();
    size_t scan_bytes = p.scan_tmp;
    ISE_CUDA(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, items, item_off, (int)(nlist + 1), st));

    // 2. scan: persistent CTAs take work items from a counter (the item count stays on the device)
    const bool vec = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(xs_sorted)) & 15) == 0;
    const bool l2 = metric == ISE_METRIC_L2;
    auto launch = [&](auto kernel) -> int {
        int per_sm = 0;
        ISE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, 0));
        kernel<<<ctx->sm_count * std::max(per_sm, 1), kThreads, 0, st>>>(
            q, nq, d, vec, xs_sorted, ids_sorted, list_off, nlist, pairs_sorted, qoff, item_off, nprobe, p.S, topk,
            counter, part_val, part_idx);
        ISE_LAUNCH_CHECK();
        return 0;
    };
    int rc;
    if (topk <= 32) rc = l2 ? launch(ivfflat_scan_kernel<true, 32>) : launch(ivfflat_scan_kernel<false, 32>);
    else rc = l2 ? launch(ivfflat_scan_kernel<true, 128>) : launch(ivfflat_scan_kernel<false, 128>);
    if (rc) return rc;

    // 3. merge the nprobe * S partial lists of every query, at most kMergeFanIn at a time
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
            rc = ise_topk_merge(ctx, src_val + in, src_idx + in, n, nq, topk, metric, dst_val + out, dst_idx + out, stream);
            if (rc) return rc;
        }
        std::swap(src_val, dst_val);
        std::swap(src_idx, dst_idx);
        g = g2;
    }
    return ise_topk_merge(ctx, src_val, src_idx, (int)g, nq, topk, metric, out_val, out_idx, stream);
}
