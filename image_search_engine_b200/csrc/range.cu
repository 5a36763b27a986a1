// Range search over the flat index: every database column whose exact FP32 score beats a radius
// (faiss/IndexFlat.cpp IndexFlat::range_search -> faiss/utils/distances.cpp range_search_inner_product /
// range_search_L2sqr).  IP keeps dis > radius, L2 keeps dis < radius on squared distances, both strict and in FP32.
//
// Tensor-core path (nq >= 20, Faiss's BLAS regime):
//   ise_range_seed   per-row coarse threshold = radius loosened by the rigorous coarse bound (CoarseBound), so that
//                    ise_gemm_collect over the hi planes appends EVERY column whose exact score can qualify;
//   ise_range_count  exact FP32 re-score of the appended candidates (rescore.cu's formulas), strict radius test,
//                    per-row kept counts; rows whose collect buffer overflowed are left to the caller;
//   ise_range_lims   exclusive scan of the kept counts -> lims (int64: totals can exceed 2^31);
//   ise_range_fill   compaction of the kept (dis, id) pairs into the result arrays (unordered within a row);
//   ise_range_sort   segmented sort of each row's results by id (Faiss scans the database in order).
// Exact path (nq < 20): ise_scores_range over the [nq, nb] matrix of ise_pair_scores, counted and written in column
// order (no sort needed).
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kScoreTile = 4 * kThreads;     // ise_scores_range: columns per block, four per thread

static inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

// IP:  seed = radius - slack,  L2: seed = radius + 2 slack  (collect keeps coarse score > / < seed).
// slack = CoarseBound eps (coarse hi-plane product vs the real inner product)
//       + the rounding of the FP32 re-score (per-lane sequential FMAs over <= d/32 + 4 terms, a 5-level warp tree:
//         <= (d/32 + 9) 2^-24 |a||b|, taken with a 2x margin)
//       + a few ulps of every magnitude the two comparisons round at (the collect epilogue's fma and threshold, the
//         re-score's norm expansion), so that the strict test of the collect can never drop a column whose exact
//         FP32 score qualifies.
template <bool L2>
__global__ void range_seed_kernel(const float* __restrict__ a_meta, const float* __restrict__ a_norms,
                                  const float* __restrict__ a_row_inv, const float* __restrict__ b_meta, int64_t m,
                                  int d, float radius, float* __restrict__ row_seed) {
    CoarseBound bound;
    bound.init(a_meta, b_meta, d);
    const float nb2 = b_meta[META_MAX_NORM_SQ];
    const float nbmax = sqrtf(nb2);
    const float fp32_rel = (float)(2 * (d / 32 + 9)) * 5.9604645e-8f;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < m; row += (int64_t)gridDim.x * blockDim.x) {
        if (a_row_inv) bound.set_a_inv_scale(a_row_inv[row]);
        const float an = a_norms[row];
        const float na = sqrtf(an);
        const float slack = bound.eps(an) + fp32_rel * na * nbmax;
        const float ulps = 9.5367432e-7f;        // 2^-20: 16 ulps
        row_seed[row] = L2 ? radius + 2.f * slack + ulps * (fabsf(radius) + an + nb2)
                           : radius - slack - ulps * (fabsf(radius) + na * nbmax);
    }
}

// One block per row: re-score min(row_count, cap) collected candidates exactly, keep the strict passes (exact score
// written over the coarse one), drop the rest (id -> -1).  kept[row] = number kept; 0 for overflowing rows
// (row_count > cap), which the caller re-runs with a larger buffer.
template <typename TA, bool L2>
__global__ void range_count_kernel(const TA* __restrict__ a, int64_t lda, const float* __restrict__ b, int64_t ldb,
                                   int64_t m, int d, float radius, int64_t id_base, const float* __restrict__ a_norms,
                                   const float* __restrict__ b_norms, int cap, const int32_t* __restrict__ row_count,
                                   float* __restrict__ cand_val, int64_t* __restrict__ cand_idx,
                                   int64_t* __restrict__ kept) {
    extern __shared__ float s_a[];
    __shared__ int s_kept;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) kept[m] = 0;     // lims scan runs over m + 1 entries
    for (int64_t row = blockIdx.x; row < m; row += gridDim.x) {
        const int rc = row_count[row];
        if (rc > cap) {
            if (threadIdx.x == 0) kept[row] = 0;
            continue;
        }
        const TA* arow = a + row * lda;
        for (int c = threadIdx.x; c < d; c += kThreads) s_a[c] = (float)arow[c];
        if (threadIdx.x == 0) s_kept = 0;
        __syncthreads();
        const float an = L2 ? a_norms[row] : 0.f;
        int mine = 0;
        for (int j = warp; j < rc; j += kWarps) {
            const int64_t slot = row * (int64_t)cap + j;
            const long long id = cand_idx[slot];
            if (id < 0) continue;                                   // warp-uniform
            const float* brow = b + (id - id_base) * ldb;
            float acc = 0.f;
            if ((d & 3) == 0 && (ldb & 3) == 0) {
                const float4* b4 = reinterpret_cast<const float4*>(brow);
                const float4* a4 = reinterpret_cast<const float4*>(s_a);
                for (int c = lane; c < d / 4; c += 32) {
                    const float4 y = __ldg(b4 + c);
                    const float4 x = a4[c];
                    acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc);
                    acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
                }
            } else {
                for (int c = lane; c < d; c += 32) acc = fmaf(s_a[c], __ldg(brow + c), acc);
            }
            acc = warp_sum(acc);
            float s = acc;
            if (L2) {
                const float dis = an + b_norms[id - id_base] - 2.f * acc;   // x_norms[i] + y_norms[j] - 2 * ip
                s = dis < 0.f ? 0.f : dis;
            }
            const bool keep = L2 ? (s < radius) : (s > radius);
            if (lane == 0) {
                if (keep) {
                    cand_val[slot] = s;
                    ++mine;
                } else {
                    cand_idx[slot] = -1;
                }
            }
        }
        if (lane == 0 && mine) atomicAdd(&s_kept, mine);
        __syncthreads();
        if (threadIdx.x == 0) kept[row] = s_kept;
        __syncthreads();
    }
}

// One block per candidate row: the kept entries (id >= 0 among the first row_count slots) go, in slot order, to
// out[lims[out_row] ...].  Overflowing rows are skipped.
__global__ void range_fill_kernel(int64_t m, int cap, const int32_t* __restrict__ row_count,
                                  const float* __restrict__ cand_val, const int64_t* __restrict__ cand_idx,
                                  const int64_t* __restrict__ row_map, const int64_t* __restrict__ lims,
                                  float* __restrict__ out_dis, int64_t* __restrict__ out_ids) {
    using Scan = cub::BlockScan<int, kThreads>;
    __shared__ typename Scan::TempStorage tmp;
    for (int64_t row = blockIdx.x; row < m; row += gridDim.x) {
        const int rc = row_count[row];
        if (rc > cap) continue;
        int64_t base = lims[row_map ? row_map[row] : row];
        for (int j0 = 0; j0 < rc; j0 += kThreads) {
            const int j = j0 + threadIdx.x;
            const int64_t slot = row * (int64_t)cap + j;
            const long long id = j < rc ? cand_idx[slot] : -1;
            const int flag = id >= 0 ? 1 : 0;
            int pos, total;
            Scan(tmp).ExclusiveSum(flag, pos, total);
            if (flag) {
                out_ids[base + pos] = id;
                out_dis[base + pos] = cand_val[slot];
            }
            base += total;
            __syncthreads();
        }
    }
}

// ise_scores_range: number of qualifying columns of each (row, tile of kScoreTile columns); cnt[nq * ntiles] = 0
template <bool L2>
__global__ void scores_range_count_kernel(const float* __restrict__ scores, int64_t nq, int64_t nb, int64_t ntiles,
                                          float radius, int64_t* __restrict__ cnt) {
    using Reduce = cub::BlockReduce<int, kThreads>;
    __shared__ typename Reduce::TempStorage tmp;
    const int64_t row = blockIdx.y;
    if (row == 0 && blockIdx.x == 0 && threadIdx.x == 0) cnt[nq * ntiles] = 0;
    const float* srow = scores + row * nb;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t c0 = t * kScoreTile + 4 * threadIdx.x;
        int n = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (c0 + i < nb) {
                const float s = srow[c0 + i];
                n += (L2 ? (s < radius) : (s > radius)) ? 1 : 0;
            }
        }
        const int total = Reduce(tmp).Sum(n);
        if (threadIdx.x == 0) cnt[row * ntiles + t] = total;
        __syncthreads();
    }
}

// lims[r] = offs[r * ntiles] (offs = base + exclusive scan of the tile counts), r = 0 .. nq
__global__ void scores_range_lims_kernel(const int64_t* __restrict__ offs, int64_t nq, int64_t ntiles,
                                         int64_t* __restrict__ lims) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r <= nq) lims[r] = offs[r * ntiles];
}

template <bool L2>
__global__ void scores_range_fill_kernel(const float* __restrict__ scores, int64_t nq, int64_t nb, int64_t ntiles,
                                         float radius, int64_t id_base, const int64_t* __restrict__ offs, int64_t base,
                                         float* __restrict__ out_dis, int64_t* __restrict__ out_ids) {
    using Scan = cub::BlockScan<int, kThreads>;
    __shared__ typename Scan::TempStorage tmp;
    const int64_t row = blockIdx.y;
    const float* srow = scores + row * nb;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t c0 = t * kScoreTile + 4 * threadIdx.x;
        float s[4];
        int n = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            s[i] = c0 + i < nb ? srow[c0 + i] : 0.f;
            n += (c0 + i < nb && (L2 ? (s[i] < radius) : (s[i] > radius))) ? 1 : 0;
        }
        int pos;
        Scan(tmp).ExclusiveSum(n, pos);
        int64_t o = offs[row * ntiles + t] - base + pos;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (c0 + i < nb && (L2 ? (s[i] < radius) : (s[i] > radius))) {
                out_dis[o] = s[i];
                out_ids[o] = id_base + c0 + i;
                ++o;
            }
        }
        __syncthreads();
    }
}

static size_t scan_temp_bytes(int64_t items) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveScan(nullptr, bytes, (const int64_t*)nullptr, (int64_t*)nullptr, cub::Sum(), (int64_t)0,
                                   items);
    return bytes;
}

static size_t sort_temp_bytes(int64_t m, int64_t total) {
    size_t bytes = 0;
    cub::DoubleBuffer<int64_t> keys(nullptr, nullptr);
    cub::DoubleBuffer<float> vals(nullptr, nullptr);
    cub::DeviceSegmentedSort::SortPairs(nullptr, bytes, keys, vals, (int)total, (int)m, (const int64_t*)nullptr,
                                        (const int64_t*)nullptr);
    return bytes;
}

}  // namespace

ISE_EXPORT int ise_range_seed(ise_ctx* ctx, const float* a_meta, const float* a_norms, const float* a_row_inv,
                              const float* b_meta, int64_t m, int d, int metric, float radius, float* row_seed,
                              void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(m >= 0 && d > 0);
    if (m == 0) return 0;
    ISE_CHECK_ARG(a_meta && a_norms && b_meta && row_seed);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (int)std::min<int64_t>(ceil_div64(m, kThreads), (int64_t)ctx->sm_count * 4);
    if (metric == ISE_METRIC_L2)
        range_seed_kernel<true><<<grid, kThreads, 0, st>>>(a_meta, a_norms, a_row_inv, b_meta, m, d, radius, row_seed);
    else
        range_seed_kernel<false><<<grid, kThreads, 0, st>>>(a_meta, a_norms, a_row_inv, b_meta, m, d, radius, row_seed);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_range_count(ise_ctx* ctx, const void* a, int a_dtype, int64_t lda, const float* b, int64_t ldb,
                               int64_t m, int64_t n, int d, int metric, float radius, int64_t id_base,
                               const float* a_norms, const float* b_norms, int cap, const int32_t* row_count,
                               float* cand_val, int64_t* cand_idx, int64_t* kept, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(a_dtype == ISE_DTYPE_F32 || a_dtype == ISE_DTYPE_U8);
    ISE_CHECK_ARG(m >= 0 && n > 0 && d > 0 && cap >= 1 && lda >= d && ldb >= d);
    ISE_CHECK_ARG((size_t)d * sizeof(float) <= 48 * 1024);
    ISE_CHECK_ARG(kept != nullptr);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m == 0) {
        ISE_CUDA(cudaMemsetAsync(kept, 0, sizeof(int64_t), st));
        return 0;
    }
    ISE_CHECK_ARG(a && b && row_count && cand_val && cand_idx);
    if (metric == ISE_METRIC_L2) ISE_CHECK_ARG(a_norms && b_norms);
    ISE_CHECK_ARG((reinterpret_cast<uintptr_t>(b) & 15) == 0);
    const int grid = (int)std::min<int64_t>(m, (int64_t)ctx->sm_count * 8);
    const size_t shm = (size_t)((d + 3) / 4 * 4) * sizeof(float);
#define ISE_RANGE_ARGS lda, b, ldb, m, d, radius, id_base, a_norms, b_norms, cap, row_count, cand_val, cand_idx, kept
    const bool l2 = metric == ISE_METRIC_L2;
    if (a_dtype == ISE_DTYPE_F32) {
        if (l2) range_count_kernel<float, true><<<grid, kThreads, shm, st>>>((const float*)a, ISE_RANGE_ARGS);
        else range_count_kernel<float, false><<<grid, kThreads, shm, st>>>((const float*)a, ISE_RANGE_ARGS);
    } else {
        if (l2) range_count_kernel<uint8_t, true><<<grid, kThreads, shm, st>>>((const uint8_t*)a, ISE_RANGE_ARGS);
        else range_count_kernel<uint8_t, false><<<grid, kThreads, shm, st>>>((const uint8_t*)a, ISE_RANGE_ARGS);
    }
#undef ISE_RANGE_ARGS
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT size_t ise_range_lims_workspace_bytes(ise_ctx* ctx, int64_t m) {
    if (!ctx || m < 0) return 0;
    return scan_temp_bytes(m + 1) + 256;
}

ISE_EXPORT int ise_range_lims(ise_ctx* ctx, const int64_t* kept, int64_t m, int64_t base, int64_t* lims,
                              void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && m >= 0 && kept && lims && workspace);
    if (workspace_bytes < ise_range_lims_workspace_bytes(ctx, m)) ISE_FAIL("workspace too small");
    DeviceGuard guard(ctx->device);
    size_t bytes = workspace_bytes;
    ISE_CUDA(cub::DeviceScan::ExclusiveScan(workspace, bytes, kept, lims, cub::Sum(), base, m + 1,
                                            (cudaStream_t)stream));
    return 0;
}

ISE_EXPORT int ise_range_fill(ise_ctx* ctx, int64_t m, int cap, const int32_t* row_count, const float* cand_val,
                              const int64_t* cand_idx, const int64_t* row_map, const int64_t* lims, float* out_dis,
                              int64_t* out_ids, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && m >= 0 && cap >= 1);
    if (m == 0) return 0;
    ISE_CHECK_ARG(row_count && cand_val && cand_idx && lims && out_dis && out_ids);
    DeviceGuard guard(ctx->device);
    const int grid = (int)std::min<int64_t>(m, (int64_t)ctx->sm_count * 8);
    range_fill_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(m, cap, row_count, cand_val, cand_idx, row_map, lims,
                                                                    out_dis, out_ids);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT size_t ise_range_sort_workspace_bytes(ise_ctx* ctx, int64_t m, int64_t total) {
    if (!ctx || m <= 0 || total <= 0 || total >= ((int64_t)1 << 31) || m >= ((int64_t)1 << 31)) return 0;
    return align256((size_t)total * sizeof(int64_t)) + align256((size_t)total * sizeof(float)) +
           sort_temp_bytes(m, total) + 256;
}

ISE_EXPORT int ise_range_sort(ise_ctx* ctx, int64_t m, const int64_t* lims, int64_t total, float* dis, int64_t* ids,
                              void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && m >= 0 && total >= 0);
    if (m == 0 || total == 0) return 0;
    ISE_CHECK_ARG(total < ((int64_t)1 << 31) && m < ((int64_t)1 << 31));
    ISE_CHECK_ARG(lims && dis && ids && workspace);
    if (workspace_bytes < ise_range_sort_workspace_bytes(ctx, m, total)) ISE_FAIL("workspace too small");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    int64_t* alt_ids = reinterpret_cast<int64_t*>(w);
    w += align256((size_t)total * sizeof(int64_t));
    float* alt_dis = reinterpret_cast<float*>(w);
    w += align256((size_t)total * sizeof(float));
    size_t bytes = sort_temp_bytes(m, total);
    cub::DoubleBuffer<int64_t> keys(ids, alt_ids);
    cub::DoubleBuffer<float> vals(dis, alt_dis);
    ISE_CUDA(cub::DeviceSegmentedSort::SortPairs(w, bytes, keys, vals, (int)total, (int)m, lims, lims + 1, st));
    if (keys.Current() != ids)
        ISE_CUDA(cudaMemcpyAsync(ids, keys.Current(), (size_t)total * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    if (vals.Current() != dis)
        ISE_CUDA(cudaMemcpyAsync(dis, vals.Current(), (size_t)total * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

ISE_EXPORT size_t ise_scores_range_workspace_bytes(ise_ctx* ctx, int64_t nq, int64_t nb) {
    if (!ctx || nq <= 0 || nb <= 0) return 0;
    const int64_t items = nq * ceil_div64(nb, kScoreTile) + 1;
    return 2 * align256((size_t)items * sizeof(int64_t)) + scan_temp_bytes(items) + 256;
}

ISE_EXPORT int ise_scores_range(ise_ctx* ctx, const float* scores, int64_t nq, int64_t nb, int metric, float radius,
                                int64_t id_base, int64_t base, int64_t* lims, float* out_dis, int64_t* out_ids,
                                void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(nq >= 0 && nb > 0 && nq <= 65535);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(scores && lims && workspace && (out_dis == nullptr) == (out_ids == nullptr));
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (workspace_bytes < ise_scores_range_workspace_bytes(ctx, nq, nb)) ISE_FAIL("workspace too small");
    const int64_t ntiles = ceil_div64(nb, kScoreTile), items = nq * ntiles + 1;
    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    int64_t* cnt = reinterpret_cast<int64_t*>(w);
    int64_t* offs = reinterpret_cast<int64_t*>(w + align256((size_t)items * sizeof(int64_t)));
    void* tmp = w + 2 * align256((size_t)items * sizeof(int64_t));
    size_t tmp_bytes = scan_temp_bytes(items);
    const dim3 grid((unsigned)std::min<int64_t>(ntiles, (int64_t)ctx->sm_count * 8), (unsigned)nq);
    const bool l2 = metric == ISE_METRIC_L2;
    if (l2) scores_range_count_kernel<true><<<grid, kThreads, 0, st>>>(scores, nq, nb, ntiles, radius, cnt);
    else scores_range_count_kernel<false><<<grid, kThreads, 0, st>>>(scores, nq, nb, ntiles, radius, cnt);
    ISE_LAUNCH_CHECK();
    ISE_CUDA(cub::DeviceScan::ExclusiveScan(tmp, tmp_bytes, cnt, offs, cub::Sum(), base, items, st));
    scores_range_lims_kernel<<<(unsigned)ceil_div64(nq + 1, kThreads), kThreads, 0, st>>>(offs, nq, ntiles, lims);
    ISE_LAUNCH_CHECK();
    if (out_dis) {
        if (l2) scores_range_fill_kernel<true><<<grid, kThreads, 0, st>>>(scores, nq, nb, ntiles, radius, id_base, offs, base, out_dis, out_ids);
        else scores_range_fill_kernel<false><<<grid, kThreads, 0, st>>>(scores, nq, nb, ntiles, radius, id_base, offs, base, out_dis, out_ids);
        ISE_LAUNCH_CHECK();
    }
    return 0;
}
