// Exact FP32 re-scoring + re-ranking of the candidates chosen by the tensor-core selection pass.
//
// The tcgen05 accumulator adds with truncation, so a K-long contraction carries a (mostly common-mode)
// relative error of up to ~K/16 * 2^-23 -- harmless for choosing candidates, visible in returned
// distances (e.g. a self-match at 2e-5 instead of 0).  This pass recomputes the k selected scores per
// row with plain FP32 FMAs on the original rows, applies Faiss's own formulas (IndexFlat search,
// distances.cpp: inner product, or |x|^2 + |y|^2 - 2<x,y> clamped at 0) and re-sorts the row by
// (score, id).  HBM-bound and tiny: m*k rows of B gathered once.
#include "common.cuh"

namespace {

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxK = 1024;   // candidates per row (collect mode hands in up to 1024 unsorted ones)

// kc candidates in (ids + coarse scores), topk exact results out.  With `flag_count` non-null the row is
// verified against the coarse pass's error bound and appended to `flag_rows` when the candidate list
// cannot be PROVEN to contain the true top-k (the caller re-runs those rows at full precision).
//
// Bound (CoarseBound in common.cuh): every coarse inner product is within eps = kappa |a| max_col|b| of
// the exact one; a column outside the candidate list has coarse score <= T (the worst kept one, or the
// seed), hence exact score <= T + eps: if the k-th exact candidate beats that, the list provably holds
// the true top-k.  (L2: scores are |a|^2 + |b|^2 - 2<a,b>, so the slack is 2 eps.)
template <typename TA, bool L2>
__global__ void rescore_kernel(const TA* __restrict__ a, int64_t lda, const float* __restrict__ b, int64_t ldb,
                               int64_t m, int64_t n, int d, int kc, int topk, int64_t id_base,
                               const float* __restrict__ a_norms, const float* __restrict__ b_norms,
                               const float* __restrict__ cand_val, const int64_t* __restrict__ cand_idx,
                               float* __restrict__ val, int64_t* __restrict__ idx,
                               const float* __restrict__ a_meta, const float* __restrict__ b_meta,
                               const float* __restrict__ a_row_inv, const float* __restrict__ row_seed, const int32_t* __restrict__ row_count,
                               int32_t* __restrict__ flag_rows, int32_t* __restrict__ flag_count) {
    extern __shared__ float s_a[];          // the row of A as float32
    __shared__ float s_v[kMaxK];
    __shared__ long long s_i[kMaxK];
    __shared__ float s_kth;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float worst = L2 ? 3.402823466e+38f : -3.402823466e+38f;
    CoarseBound bound;
    if (flag_count) bound.init(a_meta, b_meta, d);
    for (int64_t row = blockIdx.x; row < m; row += gridDim.x) {
        const TA* arow = a + row * lda;
        for (int c = threadIdx.x; c < d; c += kThreads) s_a[c] = (float)arow[c];
        if (threadIdx.x == 0) s_kth = worst;
        __syncthreads();
        const float an = (L2 || flag_count) ? a_norms[row] : 0.f;
        if (flag_count && a_row_inv) bound.set_a_inv_scale(a_row_inv[row]);    // row operand with per-row plane scales
        // collect mode appends candidates to slots [0, row_count): re-score and rank only those (the ranking below is
        // quadratic in the number of slots looked at -- 1024^2 per row at the full buffer against ~375^2 used)
        const int kv = row_count ? min(max(row_count[row], 0), kc) : kc;
        for (int j = warp; j < kv; j += kWarps) {
            const long long id = cand_idx[row * kc + j];
            float out = worst;
            if (id >= 0) {
                const int64_t col = id - id_base;
                out = exact_score<L2>(s_a, b + col * ldb, d, ldb, an, b_norms + col, lane);
            }
            if (lane == 0) { s_v[j] = out; s_i[j] = id; }
        }
        __syncthreads();
        // rank by counting: (score, id) is a strict total order over the real candidates
        for (int r = kv + threadIdx.x; r < topk; r += kThreads) {      // fewer candidates than k: pad the tail
            val[row * topk + r] = worst;
            idx[row * topk + r] = -1;
        }
        for (int me = threadIdx.x; me < kv; me += kThreads) {
            const float v = s_v[me];
            const long long id = s_i[me];
            int rank = 0;
            for (int t = 0; t < kv; ++t) {
                if (t == me) continue;
                const bool t_first = (id < 0 && s_i[t] < 0) ? (t < me)
                                                            : cand_better<!L2>(s_v[t], s_i[t], v, id);
                rank += t_first ? 1 : 0;
            }
            if (rank < topk) {
                val[row * topk + rank] = v;
                idx[row * topk + rank] = id;
            }
            if (rank == topk - 1 && id >= 0) s_kth = v;
        }
        __syncthreads();
        if (flag_count && threadIdx.x == 0) {
            // T bounds the coarse score of every column that is NOT in the list: the worst kept
            // candidate when the list is full, and/or the seed every kept candidate had to beat
            // collect mode (row_count given): the buffer holds EVERY column beating the seed unless it
            // overflowed; list mode: the list is sorted by coarse score and full when its last slot is used
            const bool overflow = row_count != nullptr && row_count[row] > kc;
            const bool full = row_count == nullptr && cand_idx[row * kc + kc - 1] >= 0;
            float T = worst;
            bool bounded = false;
            if (full) { T = cand_val[row * kc + kc - 1]; bounded = true; }
            if (row_seed) {
                const float sd = row_seed[row];
                T = bounded ? (L2 ? fminf(T, sd) : fmaxf(T, sd)) : sd;
                bounded = true;
            }
            if (bounded) {                          // otherwise every column is a candidate
                const float eps = bound.eps(an);
                const bool proven = !overflow && (L2 ? (s_kth < T - 2.f * eps) : (s_kth > T + eps));
                if (!proven) flag_rows[atomicAdd(flag_count, 1)] = (int32_t)row;
            }
        }
        __syncthreads();
    }
}

// topk == 1 fast path (k-means assign / quantisation distances): one warp per row, no sorting; ROWS rows (and their
// gathered winners) in flight per warp so the loads cover HBM latency
// It reads A from global memory but does exact_score's arithmetic (common.cuh) whenever both step by the same width:
// float4 steps here also need float32 A rows with lda % 4 == 0 and 16-byte alignment (uint8 rows step by one).
template <typename TA, bool L2, int ROWS>
__global__ void rescore_top1_kernel(const TA* __restrict__ a, int64_t lda, const float* __restrict__ b, int64_t ldb,
                                    int64_t m, int d, int64_t id_base, const float* __restrict__ a_norms,
                                    const float* __restrict__ b_norms, float* __restrict__ val,
                                    const int64_t* __restrict__ idx) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const bool vec = sizeof(TA) == 4 && (d & 3) == 0 && (lda & 3) == 0 && (ldb & 3) == 0 &&
                     ((reinterpret_cast<uintptr_t>(a) & 15) == 0);
    for (int64_t r0 = warp * ROWS; r0 < m; r0 += nwarps * ROWS) {
        int64_t col[ROWS];
        float acc[ROWS];
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
            const long long id = r0 + i < m ? idx[r0 + i] : -1;
            col[i] = id < 0 ? -1 : id - id_base;
            acc[i] = 0.f;
        }
        if (vec) {
            for (int c = lane; c < d / 4; c += 32) {
                float4 x[ROWS], y[ROWS];
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    if (col[i] < 0) continue;
                    x[i] = __ldg(reinterpret_cast<const float4*>(a + (r0 + i) * lda) + c);
                    y[i] = __ldg(reinterpret_cast<const float4*>(b + col[i] * ldb) + c);
                }
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    if (col[i] < 0) continue;
                    acc[i] = fmaf(x[i].x, y[i].x, acc[i]); acc[i] = fmaf(x[i].y, y[i].y, acc[i]);
                    acc[i] = fmaf(x[i].z, y[i].z, acc[i]); acc[i] = fmaf(x[i].w, y[i].w, acc[i]);
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < ROWS; ++i)
                if (col[i] >= 0)
                    for (int c = lane; c < d; c += 32)
                        acc[i] = fmaf((float)a[(r0 + i) * lda + c], __ldg(b + col[i] * ldb + c), acc[i]);
        }
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
            if (col[i] < 0) continue;      // warp-uniform
            const float t = warp_sum(acc[i]);
            if (lane == 0) {
                if (L2) {
                    const float dis = a_norms[r0 + i] + b_norms[col[i]] - 2.f * t;
                    val[r0 + i] = dis < 0.f ? 0.f : dis;
                } else {
                    val[r0 + i] = t;
                }
            }
        }
    }
}

}  // namespace

static int launch_rescore(ise_ctx* ctx, const void* a, int a_dtype, int64_t lda, const float* b, int64_t ldb,
                          int64_t m, int64_t n, int d, int metric, int kc, int topk, int64_t id_base,
                          const float* a_norms, const float* b_norms, const float* cand_val, const int64_t* cand_idx,
                          float* val, int64_t* idx, const float* a_meta, const float* b_meta, const float* a_row_inv,
                          const float* row_seed,
                          const int32_t* row_count, int32_t* flag_rows, int32_t* flag_count, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(a_dtype == ISE_DTYPE_F32 || a_dtype == ISE_DTYPE_U8);
    ISE_CHECK_ARG(m >= 0 && n > 0 && d > 0 && topk >= 1 && kc >= topk && kc <= kMaxK && lda >= d && ldb >= d);
    ISE_CHECK_ARG((size_t)d * sizeof(float) <= 48 * 1024);
    if (m == 0) return 0;
    ISE_CHECK_ARG(a && b && val && idx && cand_idx);
    if (metric == ISE_METRIC_L2) ISE_CHECK_ARG(a_norms && b_norms);
    if (flag_count) ISE_CHECK_ARG(flag_rows && cand_val && a_meta && b_meta && a_norms);
    if (row_count) ISE_CHECK_ARG(row_seed != nullptr);
    ISE_CHECK_ARG((reinterpret_cast<uintptr_t>(b) & 15) == 0);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (flag_count) ISE_CUDA(cudaMemsetAsync(flag_count, 0, sizeof(int32_t), st));
    const bool l2 = metric == ISE_METRIC_L2;
    if (kc == 1 && topk == 1 && !flag_count && cand_idx == idx) {
        const int g1 = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(m, 8 * 4), (int64_t)ctx->sm_count * 8));
        if (a_dtype == ISE_DTYPE_F32) {
            if (l2) rescore_top1_kernel<float, true, 4><<<g1, 256, 0, st>>>((const float*)a, lda, b, ldb, m, d, id_base, a_norms, b_norms, val, idx);
            else rescore_top1_kernel<float, false, 4><<<g1, 256, 0, st>>>((const float*)a, lda, b, ldb, m, d, id_base, a_norms, b_norms, val, idx);
        } else {
            if (l2) rescore_top1_kernel<uint8_t, true, 4><<<g1, 256, 0, st>>>((const uint8_t*)a, lda, b, ldb, m, d, id_base, a_norms, b_norms, val, idx);
            else rescore_top1_kernel<uint8_t, false, 4><<<g1, 256, 0, st>>>((const uint8_t*)a, lda, b, ldb, m, d, id_base, a_norms, b_norms, val, idx);
        }
        ISE_LAUNCH_CHECK();
        return 0;
    }
    const int grid = (int)std::min<int64_t>(m, (int64_t)ctx->sm_count * 16);
    const size_t shm = (size_t)((d + 3) / 4 * 4) * sizeof(float);
#define ISE_RESCORE_ARGS lda, b, ldb, m, n, d, kc, topk, id_base, a_norms, b_norms, cand_val, cand_idx, val, idx, \
                         a_meta, b_meta, a_row_inv, row_seed, row_count, flag_rows, flag_count
    if (a_dtype == ISE_DTYPE_F32) {
        if (l2) rescore_kernel<float, true><<<grid, kThreads, shm, st>>>((const float*)a, ISE_RESCORE_ARGS);
        else rescore_kernel<float, false><<<grid, kThreads, shm, st>>>((const float*)a, ISE_RESCORE_ARGS);
    } else {
        if (l2) rescore_kernel<uint8_t, true><<<grid, kThreads, shm, st>>>((const uint8_t*)a, ISE_RESCORE_ARGS);
        else rescore_kernel<uint8_t, false><<<grid, kThreads, shm, st>>>((const uint8_t*)a, ISE_RESCORE_ARGS);
    }
#undef ISE_RESCORE_ARGS
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_rescore_topk(ise_ctx* ctx, const void* a, int a_dtype, int64_t lda, const float* b, int64_t ldb,
                                int64_t m, int64_t n, int d, int metric, int topk, int64_t id_base,
                                const float* a_norms, const float* b_norms, float* val, int64_t* idx,
                                void* stream) {
    return launch_rescore(ctx, a, a_dtype, lda, b, ldb, m, n, d, metric, topk, topk, id_base, a_norms, b_norms,
                          nullptr, idx, val, idx, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, stream);
}

ISE_EXPORT int ise_rescore_select(ise_ctx* ctx, const void* a, int a_dtype, int64_t lda, const float* a_meta,
                                  const float* a_norms, const float* a_row_inv, const float* b, int64_t ldb, const float* b_meta,
                                  const float* b_norms, int64_t m, int64_t n, int d, int metric, int kc, int topk,
                                  int64_t id_base, const float* row_seed, const int32_t* row_count,
                                  const float* cand_val, const int64_t* cand_idx, float* out_val, int64_t* out_idx,
                                  int32_t* flag_rows, int32_t* flag_count, void* stream) {
    ISE_CHECK_ARG(flag_rows && flag_count);
    return launch_rescore(ctx, a, a_dtype, lda, b, ldb, m, n, d, metric, kc, topk, id_base, a_norms, b_norms, cand_val,
                          cand_idx, out_val, out_idx, a_meta, b_meta, a_row_inv, row_seed, row_count, flag_rows,
                          flag_count, stream);
}
