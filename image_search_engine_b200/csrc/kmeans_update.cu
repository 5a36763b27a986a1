// k-means centroid update: the device half of faiss Clustering.cpp compute_centroids /
// split_clusters / post_process_centroids (reached from kmeans_faiss.py:41).
//
// HBM-bound scatter-add: one warp per descriptor row, 128-bit row loads, 128-bit vector
// reductions (red.global.add.v4.f32) into the FP32 [k, d] sum matrix that lives in L2.
// Sums are accumulated in FP32 like Faiss; the order differs (atomics vs Faiss's data order),
// which stays inside the 1e-4 relative centroid tolerance of the parity contract.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

__device__ __forceinline__ void red_add_v4(float* addr, float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

// cent != nullptr: the objective term of each row is recomputed here in exact FP32 from the row that is
// already in registers and its centroid (L2-resident): <x, c> (spherical / IP) or sum (x - c)^2 (L2),
// instead of trusting a distance that came out of the tensor-core accumulator.
template <typename T>
__global__ void accumulate_kernel(const T* __restrict__ x, int64_t n, int d, int64_t ldx,
                                  const int64_t* __restrict__ assign, const float* __restrict__ dis,
                                  const float* __restrict__ cent, int metric,
                                  float* __restrict__ sums, float* __restrict__ counts, double* __restrict__ obj) {
    __shared__ double s_obj[kWarps];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int64_t warp = (int64_t)blockIdx.x * kWarps + wib;
    const int64_t nwarps = (int64_t)gridDim.x * kWarps;
    const bool vec4 = sizeof(T) == 4 && (d % 4 == 0) && (ldx % 4 == 0) &&
                      ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && ((reinterpret_cast<uintptr_t>(sums) & 15) == 0);
    double my_obj = 0.0;
    for (int64_t r = warp; r < n; r += nwarps) {
        const int64_t a = __ldg(assign + r);
        if (a < 0) continue;
        float* dst = sums + a * (int64_t)d;
        const T* row = x + r * ldx;
        const float* crow = cent ? cent + a * (int64_t)d : nullptr;
        float acc = 0.f;
        if (vec4) {
            const float4* row4 = reinterpret_cast<const float4*>(row);
            for (int c = lane; c < d / 4; c += 32) {
                const float4 v = __ldg(row4 + c);
                red_add_v4(dst + 4 * c, v);
                if (crow) {
                    const float4 y = __ldg(reinterpret_cast<const float4*>(crow) + c);
                    if (metric == ISE_METRIC_IP) {
                        acc = fmaf(v.x, y.x, acc); acc = fmaf(v.y, y.y, acc);
                        acc = fmaf(v.z, y.z, acc); acc = fmaf(v.w, y.w, acc);
                    } else {
                        const float e0 = v.x - y.x, e1 = v.y - y.y, e2 = v.z - y.z, e3 = v.w - y.w;
                        acc = fmaf(e0, e0, acc); acc = fmaf(e1, e1, acc);
                        acc = fmaf(e2, e2, acc); acc = fmaf(e3, e3, acc);
                    }
                }
            }
        } else {
            for (int c = lane; c < d; c += 32) {
                const float v = (float)row[c];
                atomicAdd(dst + c, v);
                if (crow) {
                    const float y = __ldg(crow + c);
                    if (metric == ISE_METRIC_IP) acc = fmaf(v, y, acc);
                    else { const float e = v - y; acc = fmaf(e, e, acc); }
                }
            }
        }
        if (crow) acc = warp_sum(acc);
        if (lane == 0) {
            atomicAdd(counts + a, 1.0f);
            if (crow) my_obj += (double)acc;
            else if (dis) my_obj += (double)__ldg(dis + r);
        }
    }
    if (lane == 0) s_obj[wib] = my_obj;
    __syncthreads();
    if (threadIdx.x == 0 && obj) {
        double t = 0.0;
        for (int i = 0; i < kWarps; ++i) t += s_obj[i];
        if (t != 0.0) atomicAdd(obj, t);
    }
}

// =====================================================================================================================
// Sorted-gather update (the default): no atomics per row at all.
//   (A) count_kernel      histogram of the assignment ids (shared-memory privatised when k fits)        8 B / row
//   (B) scan_kernel       exclusive scan -> segment starts; counts[c] += (float)cnt[c]                   O(k)
//   (C) scatter_kernel    counting sort: (key, row) pairs grouped by centroid                            8 + 8 B / row
//   (D) gather_reduce     the sorted list is cut into fixed chunks of kSegRows rows, one worker (a group of d / 4 lanes,
//                         a whole warp at d >= 128) per chunk: rows are gathered with 128-bit loads, kGatherRows in
//                         flight, and summed in REGISTERS while the centroid id does not change; a run that ends is
//                         flushed with one red.global.add.v4.f32 per lane.  4 d + 8 B / row, perfectly balanced
//                         whatever the cluster sizes, ~1.3 flushes per 64 rows at C2 instead of 64.
// The objective terms (<x, c> or |x - c|^2 in exact FP32) ride along in (D): the centroid row is loaded once per run.
// =====================================================================================================================
constexpr int kSegRows = 64;
constexpr int kGatherRows = 8;
constexpr int kCountSmemBins = 12 * 1024;

__global__ void count_kernel(const int64_t* __restrict__ assign, int64_t n, int k, int32_t* __restrict__ cnt, int use_smem) {
    extern __shared__ int s_bins[];
    const bool smem = use_smem != 0;
    if (smem) {
        for (int j = threadIdx.x; j < k; j += blockDim.x) s_bins[j] = 0;
        __syncthreads();
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // two ids per 128-bit load
    const bool al = (reinterpret_cast<uintptr_t>(assign) & 15) == 0;
    const int64_t n2 = al ? n / 2 : 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride) {
        const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(assign) + i);
        if (a.x >= 0 && a.x < k) { if (smem) atomicAdd(&s_bins[a.x], 1); else atomicAdd(cnt + a.x, 1); }
        if (a.y >= 0 && a.y < k) { if (smem) atomicAdd(&s_bins[a.y], 1); else atomicAdd(cnt + a.y, 1); }
    }
    for (int64_t i = 2 * n2 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t a = __ldg(assign + i);
        if (a >= 0 && a < k) { if (smem) atomicAdd(&s_bins[a], 1); else atomicAdd(cnt + a, 1); }
    }
    if (smem) {
        __syncthreads();
        for (int j = threadIdx.x; j < k; j += blockDim.x) {
            const int v = s_bins[j];
            if (v) atomicAdd(cnt + j, v);
        }
    }
}

// single CTA: offs[0..k] = exclusive scan of cnt; cursor = copy of the starts; counts += cnt (float, like hassign).
// Every thread owns a contiguous run of ceil(k / 1024) bins (serial), the 1024 run totals are scanned with two levels of
// warp shuffles: three barriers in all, whatever k.
__global__ void __launch_bounds__(1024)
scan_counts_kernel(const int32_t* __restrict__ cnt, int k, int32_t* __restrict__ offs, int32_t* __restrict__ cursor,
                   float* __restrict__ counts) {
    __shared__ int s_warp[32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int per = (k + 1023) / 1024;
    const int lo = min(k, (int)threadIdx.x * per), hi = min(k, lo + per);
    int total = 0;
    for (int i = lo; i < hi; ++i) total += cnt[i];
    int incl = total;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[wib] = incl;
    __syncthreads();
    if (wib == 0) {
        int w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        s_warp[lane] = w;                       // inclusive scan of the warp totals
    }
    __syncthreads();
    int run = (wib ? s_warp[wib - 1] : 0) + incl - total;       // exclusive prefix of this thread's run
    for (int i = lo; i < hi; ++i) {
        const int v = cnt[i];
        offs[i] = run;
        cursor[i] = run;
        if (v) counts[i] += (float)v;
        run += v;
    }
    if (threadIdx.x == 1023) offs[k] = s_warp[31];
}

// row_inv given (rows will be gathered from an FP16 plane): the row's scale travels with its pair, so the gather reads it
// as a stream instead of one more random 4-byte access per row
__global__ void scatter_kernel(const int64_t* __restrict__ assign, int64_t n, int k, int32_t* __restrict__ cursor,
                               int2* __restrict__ sorted, const float* __restrict__ row_inv,
                               float* __restrict__ sorted_inv) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t a = __ldg(assign + i);
        if (a < 0 || a >= k) continue;
        const int pos = atomicAdd(cursor + a, 1);
        sorted[pos] = make_int2((int)a, (int)i);
        if (row_inv) sorted_inv[pos] = __ldg(row_inv + i);
    }
}

// element types a row can be gathered as: FP32 rows, uint8 rows, or -- when the operand is EXACT in one FP16 plane
// (integer-valued SIFT, ORB: ise_prepare_rows wrote no lo plane) -- the FP16 hi plane itself, half the bytes of the
// FP32 rows: value = half * row_inv[row], both exact, so the sums are the same numbers.
template <typename T> struct RowVec;
template <> struct RowVec<float> {
    static constexpr bool kScaled = false;
    typedef float4 raw;
    static __device__ __forceinline__ raw ld(const float* row, int c4) { return __ldg(reinterpret_cast<const float4*>(row) + c4); }
    static __device__ __forceinline__ float4 cvt(raw r, float) { return r; }
};
template <> struct RowVec<uint8_t> {
    static constexpr bool kScaled = false;
    typedef uchar4 raw;
    static __device__ __forceinline__ raw ld(const uint8_t* row, int c4) { return __ldg(reinterpret_cast<const uchar4*>(row) + c4); }
    static __device__ __forceinline__ float4 cvt(raw u, float) { return make_float4((float)u.x, (float)u.y, (float)u.z, (float)u.w); }
};
template <> struct RowVec<__half> {
    static constexpr bool kScaled = true;      // FP16 hi plane: per-row power-of-two scale
    typedef uint2 raw;
    static __device__ __forceinline__ raw ld(const __half* row, int c4) { return __ldg(reinterpret_cast<const uint2*>(row) + c4); }
    static __device__ __forceinline__ float4 cvt(raw r, float inv) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
        return make_float4(a.x * inv, a.y * inv, b.x * inv, b.y * inv);
    }
};

// G = lanes per worker (4, 8, 16 or 32; 32 / G workers per warp), U = rows in flight per worker (<= G, sized so that a
// warp keeps ~4 KB of row loads in flight: measured effective latency under load is ~3 us, i.e. ~100 KB per SM are
// needed to fill HBM).  A worker owns one 64-row chunk at a time: its lanes load the chunk's (centroid, row) pairs
// ONCE, coalesced, 64 / G per lane, and every row's pair is then broadcast from its holder with a shuffle -- no
// per-row key registers, no per-row index loads.  A lane owns columns [4 (cb + lg), +4) of the rows for the
// column block cb (d > 4 G: the chunk is walked once per column block; the rows come back from L1 / L2).
__device__ __forceinline__ float run_dot(float4 a, float4 c) {
    return fmaf(a.w, c.w, fmaf(a.z, c.z, fmaf(a.y, c.y, a.x * c.x)));
}

template <typename T, int G, int U>
__global__ void __launch_bounds__(256)
gather_reduce_kernel(const T* __restrict__ x, int d, int64_t ldx, const int2* __restrict__ sorted,
                     const float* __restrict__ sorted_inv, const int32_t* __restrict__ n_sorted_ptr,
                     const float* __restrict__ cent, int metric, float* __restrict__ sums, double* __restrict__ obj) {
    static_assert(U <= G && kSegRows % G == 0, "rows in flight per worker");
    constexpr int PER = kSegRows / G;                    // (centroid, row) pairs held per lane
    constexpr bool SC = RowVec<T>::kScaled;
    __shared__ double s_obj[8];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int lg = lane & (G - 1);                       // lane within the worker
    const int64_t worker = ((int64_t)blockIdx.x * 8 + wib) * (32 / G) + lane / G;
    const int64_t n_workers = (int64_t)gridDim.x * 8 * (32 / G);
    const int64_t n_sorted = *n_sorted_ptr;             // rows with a valid id (all of them after an assign pass)
    const int64_t n_chunks = (n_sorted + kSegRows - 1) / kSegRows;
    const int d4 = d >> 2;
    double objd = 0.0;
    // inner-product objective: sum_rows <x, c> = <sum_rows x, c>, so it costs four FMAs per RUN (at the flush), not per
    // row; the L2 objective sum |x - c|^2 stays per row
    const bool ip_obj = cent != nullptr && metric == ISE_METRIC_IP, l2_obj = cent != nullptr && metric != ISE_METRIC_IP;
    // all workers of a warp run the same number of iterations (shuffles are warp-wide): idle workers carry empty chunks
    const int64_t iters = (n_chunks + n_workers - 1) / n_workers;
    for (int64_t itn = 0; itn < iters; ++itn) {
        const int64_t chunk = worker + itn * n_workers;
        const int64_t i0 = chunk * kSegRows;
        int key[PER], ridx[PER];
        float sinv[SC ? PER : 1];
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int64_t i = i0 + p * G + lg;
            const bool ok = chunk < n_chunks && i < n_sorted;
            const int2 kr = ok ? __ldg(sorted + i) : make_int2(-1, 0);
            key[p] = kr.x;
            ridx[p] = kr.y;
            if (SC) sinv[p] = ok ? __ldg(sorted_inv + i) : 1.f;
        }
        float objp = 0.f;
        for (int cb = 0; cb < d4; cb += G) {
            const int c4 = cb + lg;
            const bool col_ok = c4 < d4;
            int cur = -1;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), cc = acc;
#pragma unroll
            for (int p = 0; p < PER; ++p) {
#pragma unroll
                for (int jb = 0; jb < G; jb += U) {
                    typename RowVec<T>::raw v[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int kq = __shfl_sync(0xffffffffu, key[p], jb + u, G);
                        const int r = __shfl_sync(0xffffffffu, ridx[p], jb + u, G);
                        if (kq >= 0 && col_ok) v[u] = RowVec<T>::ld(x + (int64_t)r * ldx, c4);
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int kq = __shfl_sync(0xffffffffu, key[p], jb + u, G);
                        const float iv = SC ? __shfl_sync(0xffffffffu, sinv[SC ? p : 0], jb + u, G) : 1.f;
                        if (kq < 0) continue;
                        if (kq != cur) {
                            if (cur >= 0 && col_ok) {
                                red_add_v4(sums + (int64_t)cur * d + 4 * c4, acc);
                                if (ip_obj) objp += run_dot(acc, cc);
                            }
                            cur = kq;
                            acc = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (cent && col_ok) cc = __ldg(reinterpret_cast<const float4*>(cent + (int64_t)cur * d) + c4);
                        }
                        if (!col_ok) continue;
                        const float4 t = RowVec<T>::cvt(v[u], iv);
                        acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
                        if (l2_obj) {
                            const float e0 = t.x - cc.x, e1 = t.y - cc.y, e2 = t.z - cc.z, e3 = t.w - cc.w;
                            objp = fmaf(e0, e0, objp); objp = fmaf(e1, e1, objp);
                            objp = fmaf(e2, e2, objp); objp = fmaf(e3, e3, objp);
                        }
                    }
                }
            }
            if (cur >= 0 && col_ok) {
                red_add_v4(sums + (int64_t)cur * d + 4 * c4, acc);
                if (ip_obj) objp += run_dot(acc, cc);
            }
        }
        objd += (double)objp;            // FP32 partial of one chunk's 64 rows x 4 columns, FP64 from there on
    }
    if (obj && cent) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) objd += __shfl_xor_sync(0xffffffffu, objd, o);
        if (lane == 0) s_obj[wib] = objd;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int i = 0; i < 8; ++i) t += s_obj[i];
            if (t != 0.0) atomicAdd(obj, t);
        }
    }
}

__global__ void mean_kernel(const float* __restrict__ sums, const float* __restrict__ counts, int64_t k, int d,
                            float* __restrict__ centroids, int32_t* __restrict__ n_empty) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarps;
    int empties = 0;
    for (int64_t c = warp; c < k; c += nwarps) {
        const float h = counts[c];
        if (h == 0.f) {
            for (int j = lane; j < d; j += 32) centroids[c * d + j] = 0.f;
            empties++;
        } else {
            const float norm = 1.f / h;  // float norm = 1 / hassign[ci]; c[j] *= norm
            for (int j = lane; j < d; j += 32) centroids[c * d + j] = sums[c * d + j] * norm;
        }
    }
    if (lane == 0 && empties) atomicAdd(n_empty, empties);
}

// split_clusters: the (ci, cj) plan is ordered and later steps may read rows written by earlier ones,
// so one block walks the plan sequentially and parallelises over the dimension.
__global__ void apply_splits_kernel(float* __restrict__ centroids, int d, const int32_t* __restrict__ pairs,
                                    int nsplit) {
    const float up = 1.f + 1.f / 1024.f, dn = 1.f - 1.f / 1024.f;  // EPS = 1/1024
    for (int s = 0; s < nsplit; ++s) {
        float* ci = centroids + (int64_t)pairs[2 * s] * d;
        float* cj = centroids + (int64_t)pairs[2 * s + 1] * d;
        for (int j = threadIdx.x; j < d; j += blockDim.x) {
            const float v = cj[j];
            if ((j & 1) == 0) { ci[j] = v * up; cj[j] = v * dn; }
            else { ci[j] = v * dn; cj[j] = v * up; }
        }
        __syncthreads();
    }
}

}  // namespace

ISE_EXPORT int ise_kmeans_accumulate(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx,
                                     const int64_t* assign, const float* dis, const float* centroids, int64_t /*k*/,
                                     int metric, float* sums, float* counts, double* obj, void* stream) {
    ISE_CHECK_ARG(ctx && n >= 0 && d > 0 && ldx >= d);
    ISE_CHECK_ARG(dtype == ISE_DTYPE_F32 || dtype == ISE_DTYPE_U8);
    if (n == 0) return 0;
    ISE_CHECK_ARG(x && assign && sums && counts);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    if (centroids) ISE_CHECK_ARG((reinterpret_cast<uintptr_t>(centroids) & 15) == 0);
    DeviceGuard guard(ctx->device);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(n, kWarps), (int64_t)ctx->sm_count * 8));
    if (dtype == ISE_DTYPE_F32)
        accumulate_kernel<float><<<grid, kThreads, 0, (cudaStream_t)stream>>>((const float*)x, n, d, ldx, assign, dis,
                                                                             centroids, metric, sums, counts, obj);
    else
        accumulate_kernel<uint8_t><<<grid, kThreads, 0, (cudaStream_t)stream>>>((const uint8_t*)x, n, d, ldx, assign,
                                                                               dis, centroids, metric, sums, counts, obj);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT size_t ise_kmeans_accumulate_workspace_bytes(ise_ctx* ctx, int64_t n, int64_t k) {
    if (!ctx || n <= 0 || k <= 0) return 0;
    // cnt[k] | offs[k + 1] | cursor[k] (int32) | sorted[n] (int2) | sorted_inv[n] (float), 16-byte aligned sections
    return (size_t)(((3 * k + 1) * 4 + 15) & ~(int64_t)15) + (size_t)n * (sizeof(int2) + sizeof(float)) + 256;
}

template <typename T, int UMAX>
static void launch_gather(const T* x, int d, int64_t ldx, const int2* sorted, const float* sorted_inv, int64_t n,
                          const int32_t* n_sorted, const float* cent, int metric, float* sums, double* obj, int sm_count,
                          cudaStream_t st) {
    const int d4 = d / 4;
    int g = 4;
    while (g < d4 && g < 32) g <<= 1;
    const int64_t chunks = ceil_div64(n, kSegRows);
    const int64_t workers_per_cta = 8 * (32 / g);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(chunks, workers_per_cta), (int64_t)sm_count * 8));
#define ISE_GATHER(G) gather_reduce_kernel<T, G, (UMAX < G ? UMAX : G)><<<grid, 256, 0, st>>>(x, d, ldx, sorted, sorted_inv, n_sorted, cent, metric, sums, obj)
    switch (g) {
        case 4: ISE_GATHER(4); break;
        case 8: ISE_GATHER(8); break;
        case 16: ISE_GATHER(16); break;
        default: ISE_GATHER(32); break;
    }
#undef ISE_GATHER
}

ISE_EXPORT int ise_kmeans_accumulate_sorted(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx,
                                            const float* row_inv, const int64_t* assign, const float* centroids,
                                            int64_t k, int metric, float* sums, float* counts, double* obj,
                                            void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx && n >= 0 && d > 0 && ldx >= d && k > 0 && k < ((int64_t)1 << 31) && n < ((int64_t)1 << 31));
    ISE_CHECK_ARG(dtype == ISE_DTYPE_F32 || dtype == ISE_DTYPE_U8 || dtype == ISE_DTYPE_F16);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(dtype != ISE_DTYPE_F16 || row_inv != nullptr);      // FP16 hi planes carry per-row scales
    if (n == 0) return 0;
    ISE_CHECK_ARG(x && assign && sums && counts && workspace);
    // rows are gathered as 4-column vectors: 16-byte (float32) / 8-byte (FP16 plane) / 4-byte (uint8) aligned rows
    const uintptr_t amask = dtype == ISE_DTYPE_F32 ? 15 : (dtype == ISE_DTYPE_F16 ? 7 : 3);
    const bool vec_ok = d % 4 == 0 && ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(sums) & 15) == 0 &&
                        (reinterpret_cast<uintptr_t>(x) & amask) == 0 &&
                        (!centroids || (reinterpret_cast<uintptr_t>(centroids) & 15) == 0);
    if (!vec_ok) {
        if (dtype == ISE_DTYPE_F16) ISE_FAIL("FP16 plane rows must be 8-byte aligned with d % 4 == 0");
        return ise_kmeans_accumulate(ctx, x, dtype, n, d, ldx, assign, nullptr, centroids, 0, metric, sums, counts, obj, stream);
    }
    if (workspace_bytes < ise_kmeans_accumulate_workspace_bytes(ctx, n, k)) ISE_FAIL("workspace too small");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    int32_t* cnt = reinterpret_cast<int32_t*>((reinterpret_cast<uintptr_t>(workspace) + 15) & ~uintptr_t(15));
    int32_t* offs = cnt + k;
    int32_t* cursor = offs + k + 1;
    int2* sorted = reinterpret_cast<int2*>(reinterpret_cast<uint8_t*>(cnt) + (((3 * k + 1) * 4 + 15) & ~(int64_t)15));
    float* sorted_inv = reinterpret_cast<float*>(sorted + n);
    ISE_CUDA(cudaMemsetAsync(cnt, 0, (size_t)k * sizeof(int32_t), st));
    const int grid_n = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(n, 256 * 4), (int64_t)ctx->sm_count * 8));
    // shared-memory bins pay only when a CTA sees many more ids than there are bins
    const bool smem_bins = k <= kCountSmemBins && n / ctx->sm_count >= 8 * k;
    count_kernel<<<smem_bins ? std::min(grid_n, ctx->sm_count) : grid_n, 256, smem_bins ? (size_t)k * sizeof(int) : 0, st>>>(
        assign, n, (int)k, cnt, smem_bins ? 1 : 0);
    ISE_LAUNCH_CHECK();
    scan_counts_kernel<<<1, 1024, 0, st>>>(cnt, (int)k, offs, cursor, counts);
    ISE_LAUNCH_CHECK();
    scatter_kernel<<<grid_n, 256, 0, st>>>(assign, n, (int)k, cursor, sorted, dtype == ISE_DTYPE_F16 ? row_inv : nullptr, sorted_inv);
    ISE_LAUNCH_CHECK();
    // rows with ids outside [0, k) are left out, like the atomic kernels skip negative ids: the sorted list holds
    // offs[k] entries, which the gather kernel reads on the device (== n after an assign pass)
    if (dtype == ISE_DTYPE_F32)
        launch_gather<float, 8>((const float*)x, d, ldx, sorted, nullptr, n, offs + k, centroids, metric, sums, obj, ctx->sm_count, st);
    else if (dtype == ISE_DTYPE_F16)
        launch_gather<__half, 16>((const __half*)x, d, ldx, sorted, sorted_inv, n, offs + k, centroids, metric, sums, obj, ctx->sm_count, st);
    else
        launch_gather<uint8_t, 16>((const uint8_t*)x, d, ldx, sorted, nullptr, n, offs + k, centroids, metric, sums, obj, ctx->sm_count, st);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_kmeans_mean(ise_ctx* ctx, const float* sums, const float* counts, int64_t k, int d,
                               float* centroids, int32_t* n_empty, void* stream) {
    ISE_CHECK_ARG(ctx && sums && counts && centroids && n_empty && k > 0 && d > 0);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    ISE_CUDA(cudaMemsetAsync(n_empty, 0, sizeof(int32_t), st));
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(k, kWarps), (int64_t)ctx->sm_count * 8));
    mean_kernel<<<grid, kThreads, 0, st>>>(sums, counts, k, d, centroids, n_empty);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_kmeans_apply_splits(ise_ctx* ctx, float* centroids, int64_t k, int d, const int32_t* pairs,
                                       int32_t nsplit, void* stream) {
    ISE_CHECK_ARG(ctx && centroids && k > 0 && d > 0 && nsplit >= 0);
    if (nsplit == 0) return 0;
    ISE_CHECK_ARG(pairs != nullptr);
    DeviceGuard guard(ctx->device);
    apply_splits_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(centroids, d, pairs, nsplit);
    ISE_LAUNCH_CHECK();
    return 0;
}
