// IVFPQ ("cell-probe" index type, utils.py:311-325: IndexIVFPQ(IndexFlatL2(d), d, 8, 16, 8), nprobe = 5).
// Off every default path of the reference; built from the pieces of the hot path: the coarse quantizer and the
// 16 sub-quantizers are trained by the k-means kernels, vectors are encoded by the fused top-1 assign, and only the
// steps below are specific: residuals, and the asymmetric-distance scan of the probed inverted lists.
//
// Two scans share one arithmetic (faiss/IndexIVFPQ.cpp IVFPQScanner, by_residual, no precomputed tables):
//   ivfpq_scan_kernel            one CTA per (query, probe) writes an [nq, ntotal] distance matrix (the k > 128 path
//                                and the bit-level reference of the grouped scan);
//   grouped search / range       the (query, probe) pairs grouped by list (ivf_grouping.cuh) as in ivfflat.cu:
//     ivfpq_lut_kernel             one look-up table tab[m][code] = |(q - c_list)_m - pq[m][code]|^2 per pair and call,
//                                  [pairs, M, ksub] float32 in the workspace;
//     ivfpq_grouped_scan_kernel    one work item = (list, block of <= kQB of its queries, chunk of its codes): the
//                                  block's tables are staged in shared memory and one warp per query walks the chunk,
//                                  32 codes at a time, keeping per-lane top-k lists merged across the warp;
//     ivfpq_range_count / _fill    the same items counting, then writing, the codes with dis < radius per (pair, chunk)
//                                  segment, in Faiss's order (probe rank, then list position);
//     ise_topk_merge               the nprobe * S partial lists of each query (search).
// Every table entry is one fmaf chain over j = 0 .. dsub-1 of t = (q - c_list)[m dsub + j] - pq[m][code][j], and every
// distance is dis = 0; dis += tab[m][code_m] for m = 0 .. M-1, so all of them return the same bits.
#include "common.cuh"
#include "ivf_grouping.cuh"
#include "topk_list.cuh"

namespace {

constexpr int kThreads = 256;

__global__ void residual_kernel(const float* __restrict__ x, int64_t ldx, int64_t n, int d,
                                const float* __restrict__ cent, const int64_t* __restrict__ assign,
                                float* __restrict__ out) {
    const int64_t total = n * d;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / d;
        const int c = (int)(i - r * d);
        const int64_t a = assign[r];
        out[i] = x[r * ldx + c] - (a >= 0 ? cent[a * d + c] : 0.f);     // compute_residual: x - reconstruct(key)
    }
}

// One CTA per (query, probe): look-up table tab[m][code] = |(q - c_list)_m - pq[m][code]|^2 in shared memory, then
// every code of the list costs M table reads: dis = sum_m tab[m][code_m], summed in m order like Faiss's scanner.
// dist is [nq, ntotal] in list-sorted order, pre-filled with +inf (entries of lists that are not probed).
__global__ void ivfpq_scan_kernel(const float* __restrict__ q, int d, const float* __restrict__ coarse,
                                  const int64_t* __restrict__ probes, int nprobe, const float* __restrict__ pq,
                                  int M, int ksub, const uint8_t* __restrict__ codes,
                                  const int64_t* __restrict__ list_off, int64_t ntotal, float* __restrict__ dist) {
    extern __shared__ float sm[];
    float* res = sm;                 // [d]
    float* tab = sm + d;             // [M * ksub]
    const int64_t qi = blockIdx.y;
    const int64_t key = probes[qi * nprobe + blockIdx.x];
    if (key < 0) return;
    const int64_t lo = list_off[key], hi = list_off[key + 1];
    if (lo == hi) return;
    const int dsub = d / M;
    for (int c = threadIdx.x; c < d; c += kThreads) res[c] = q[qi * d + c] - coarse[key * d + c];
    __syncthreads();
    for (int e = threadIdx.x; e < M * ksub; e += kThreads) {
        const int m = e / ksub;
        const float* cj = pq + (int64_t)e * dsub;
        const float* rj = res + m * dsub;
        float acc = 0.f;
        for (int j = 0; j < dsub; ++j) {
            const float t = rj[j] - cj[j];
            acc = fmaf(t, t, acc);
        }
        tab[e] = acc;
    }
    __syncthreads();
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
        const uint8_t* code = codes + i * M;
        float dis = 0.f;
        for (int m = 0; m < M; ++m) dis += tab[m * ksub + code[m]];
        dist[qi * ntotal + i] = dis;
    }
}

}  // namespace

ISE_EXPORT int ise_ivfpq_residual(ise_ctx* ctx, const float* x, int64_t ldx, int64_t n, int d, const float* centroids,
                                  const int64_t* assign, float* out, void* stream) {
    ISE_CHECK_ARG(ctx && n >= 0 && d > 0 && ldx >= d);
    if (n == 0) return 0;
    ISE_CHECK_ARG(x && centroids && assign && out);
    DeviceGuard guard(ctx->device);
    const int grid = (int)std::min<int64_t>(ceil_div64(n * d, kThreads), (int64_t)ctx->sm_count * 8);
    residual_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(x, ldx, n, d, centroids, assign, out);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_ivfpq_scan(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* coarse_centroids,
                              int64_t nlist, const int64_t* probes, int nprobe, const float* pq_centroids, int M,
                              int ksub, const uint8_t* codes, const int64_t* list_offsets, int64_t ntotal,
                              float* dist, void* stream) {
    ISE_CHECK_ARG(ctx && nq >= 0 && d > 0 && nlist > 0 && nprobe >= 1 && M >= 1 && d % M == 0 && ksub >= 1 && ksub <= 256);
    ISE_CHECK_ARG(nq <= 65535);
    if (nq == 0 || ntotal == 0) return 0;
    ISE_CHECK_ARG(q && coarse_centroids && probes && pq_centroids && codes && list_offsets && dist);
    const size_t shm = ((size_t)d + (size_t)M * ksub) * sizeof(float);
    ISE_CHECK_ARG(shm <= 200 * 1024);
    DeviceGuard guard(ctx->device);
    ISE_CUDA(cudaFuncSetAttribute(ivfpq_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
    dim3 grid((unsigned)nprobe, (unsigned)nq);
    ivfpq_scan_kernel<<<grid, kThreads, shm, (cudaStream_t)stream>>>(q, d, coarse_centroids, probes, nprobe, pq_centroids, M,
                                                                    ksub, codes, list_offsets, ntotal, dist);
    ISE_LAUNCH_CHECK();
    return 0;
}

namespace {

constexpr int kQB = 4;              // queries per work item: one warp each
constexpr int kCB = 1024;           // codes per chunk granule: a chunk amortises staging its tables
constexpr int kMaxTable = 8192;     // M * ksub: kQB tables of at most 32 KB in shared memory (M <= 32 at 8 bits)
constexpr int kMaxResidual = 200 * 1024;   // bytes: the residual of the table kernel in shared memory
constexpr float kFltMax = 3.402823466e+38f;

// tab[m][code] of pair p (= q * nprobe + slot) at lut + p * M * ksub: the table ivfpq_scan_kernel builds, entry by
// entry the same fmaf chain.  Pairs without a list (probe -1 or >= nlist) are skipped.
__global__ void __launch_bounds__(kThreads) ivfpq_lut_kernel(const float* __restrict__ q, int d,
                                                             const float* __restrict__ coarse, int64_t nlist,
                                                             const int64_t* __restrict__ probes, int nprobe,
                                                             const float* __restrict__ pq, int M, int ksub,
                                                             float* __restrict__ lut) {
    extern __shared__ float res[];   // [d]
    const int64_t pair = blockIdx.x;
    const int64_t qi = pair / nprobe;
    const int64_t key = probes[pair];
    if (key < 0 || key >= nlist) return;
    const int dsub = d / M;
    for (int c = threadIdx.x; c < d; c += kThreads) res[c] = q[qi * d + c] - coarse[key * d + c];
    __syncthreads();
    float* tab = lut + pair * (int64_t)(M * ksub);
    for (int e = threadIdx.x; e < M * ksub; e += kThreads) {
        const int m = e / ksub;
        const float* cj = pq + (int64_t)e * dsub;
        const float* rj = res + m * dsub;
        float acc = 0.f;
        for (int j = 0; j < dsub; ++j) {
            const float t = rj[j] - cj[j];
            acc = fmaf(t, t, acc);
        }
        tab[e] = acc;
    }
}

// copies the tables of the item's pairs (s_pair, -1 = none) to s_lut[r * tab]
__device__ __forceinline__ void stage_tables(int tid, const float* __restrict__ lut, int tab, const int* s_pair,
                                             float* s_lut) {
    for (int r = 0; r < kQB; ++r) {
        const int pair = s_pair[r];
        if (pair < 0) continue;
        const float* src = lut + (int64_t)pair * tab;
        float* dst = s_lut + r * tab;
        if ((tab & 3) == 0) {
            for (int e = tid * 4; e < tab; e += ivf::kThreads * 4)
                *reinterpret_cast<float4*>(dst + e) = __ldg(reinterpret_cast<const float4*>(src + e));
        } else {
            for (int e = tid; e < tab; e += ivf::kThreads) dst[e] = __ldg(src + e);
        }
    }
}

// dis = sum_m tab[m][code[m]], added in m order from 0 like ivfpq_scan_kernel.  words: M % 4 == 0 and 4-byte aligned
// code rows, read as 32-bit words.
__device__ __forceinline__ float code_distance(const float* tab, int M, int ksub, const uint8_t* __restrict__ code,
                                               bool words) {
    float dis = 0.f;
    if (words) {
        for (int m = 0; m < M; m += 4) {
            const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(code + m));
            dis += tab[m * ksub + (w & 255u)];
            dis += tab[(m + 1) * ksub + ((w >> 8) & 255u)];
            dis += tab[(m + 2) * ksub + ((w >> 16) & 255u)];
            dis += tab[(m + 3) * ksub + (w >> 24)];
        }
    } else {
        for (int m = 0; m < M; ++m) dis += tab[m * ksub + code[m]];
    }
    return dis;
}

// search: warp r takes pair s_pair[r]; lane l scans list positions v_begin + l, + 32, ... (ascending, so the strict
// insert keeps the lower position = lower id on ties); the 32 lane lists are merged by (distance, position) and written
// as the partial list of (pair, chunk)
template <int KMAX>
__global__ void __launch_bounds__(ivf::kThreads) ivfpq_grouped_scan_kernel(
        const float* __restrict__ lut, int64_t nq, int M, int ksub, bool words, const uint8_t* __restrict__ codes,
        const int64_t* __restrict__ ids, const int64_t* __restrict__ list_off, int64_t nlist,
        const int32_t* __restrict__ pairs_sorted, const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off,
        int nprobe, int S, int topk, unsigned long long* __restrict__ counter, float* __restrict__ part_val,
        int64_t* __restrict__ part_idx) {
    extern __shared__ __align__(16) float s_lut[];   // [kQB][M * ksub]
    __shared__ int s_pair[kQB];
    __shared__ long long s_item;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tab = M * ksub;
    for (;;) {
        if (tid == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= item_off[nlist]) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, kCB, kQB, tid, s_pair);
        __syncthreads();
        stage_tables(tid, lut, tab, s_pair, s_lut);
        __syncthreads();
        const int pair = s_pair[warp];
        if (pair >= 0) {                                     // warp-uniform
            const float* t = s_lut + warp * tab;
            const uint8_t* cl = codes + it.lbase * M;
            TopKList<KMAX> list;
            list.init(topk);
            for (int64_t i = it.v_begin + lane; i < it.v_end; i += 32) {
                const float s = -code_distance(t, M, ksub, cl + i * M, words);
                if (s > list.thr) list.insert(s, (int)i);
            }
            const int64_t qi = pair / nprobe, slot = pair % nprobe;
            const int64_t obase = ((slot * S + it.c) * nq + qi) * topk;
            int head = 0, j = 0;
            for (; j < topk; ++j) {
                const bool live = head < topk && list.id[head] >= 0;
                float v = live ? list.v[head] : -CUDART_INF_F;
                int id = live ? list.id[head] : 0x7fffffff;
                int src = lane;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float v2 = __shfl_xor_sync(0xffffffffu, v, o);
                    const int id2 = __shfl_xor_sync(0xffffffffu, id, o);
                    const int src2 = __shfl_xor_sync(0xffffffffu, src, o);
                    if (v2 > v || (v2 == v && id2 < id)) { v = v2; id = id2; src = src2; }
                }
                if (id == 0x7fffffff) break;                 // every lane list is drained (warp-uniform)
                if (src == lane) ++head;
                if (lane == 0) {
                    part_val[obase + j] = -v;
                    part_idx[obase + j] = ids[it.lbase + id];
                }
            }
            for (j += lane; j < topk; j += 32) {
                part_val[obase + j] = kFltMax;
                part_idx[obase + j] = -1;
            }
            // chunk slots this list does not use: an id -1 at the head makes ise_topk_merge skip the list
            if (lane == 0 && it.c == it.nch - 1)
                for (int64_t c2 = it.nch; c2 < S; ++c2) part_idx[((slot * S + c2) * nq + qi) * topk] = -1;
        }
        __syncthreads();
    }
}

// range pass 1: cnt[pair * S + c] = codes of chunk c of the pair's list with dis < radius.  Segments of probe -1 and
// chunk slots a list does not use keep the zero the caller wrote.
__global__ void __launch_bounds__(ivf::kThreads) ivfpq_range_count_kernel(
        const float* __restrict__ lut, int M, int ksub, bool words, const uint8_t* __restrict__ codes,
        const int64_t* __restrict__ list_off, int64_t nlist, const int32_t* __restrict__ pairs_sorted,
        const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off, int S, float radius,
        unsigned long long* __restrict__ counter, int64_t* __restrict__ cnt) {
    extern __shared__ __align__(16) float s_lut[];
    __shared__ int s_pair[kQB];
    __shared__ long long s_item;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tab = M * ksub;
    for (;;) {
        if (tid == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= item_off[nlist]) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, kCB, kQB, tid, s_pair);
        __syncthreads();
        stage_tables(tid, lut, tab, s_pair, s_lut);
        __syncthreads();
        const int pair = s_pair[warp];
        if (pair >= 0) {
            const float* t = s_lut + warp * tab;
            const uint8_t* cl = codes + it.lbase * M;
            int64_t hits = 0;
            for (int64_t h = it.v_begin; h < it.v_end; h += 32) {
                const int64_t i = h + lane;
                const bool hit = i < it.v_end && code_distance(t, M, ksub, cl + i * M, words) < radius;
                hits += __popc(__ballot_sync(0xffffffffu, hit));
            }
            if (lane == 0) cnt[(int64_t)pair * S + it.c] = hits;
        }
        __syncthreads();
    }
}

// range pass 2: the hits of segment (pair, c) go to out[offs[seg] .. offs[seg + 1]) in list position order; an item
// whose segments are all empty is skipped before its tables are staged, and a warp stops once its segment is full.
// Writes are bounded by the segment end.
__global__ void __launch_bounds__(ivf::kThreads) ivfpq_range_fill_kernel(
        const float* __restrict__ lut, int M, int ksub, bool words, const uint8_t* __restrict__ codes,
        const int64_t* __restrict__ ids, const int64_t* __restrict__ list_off, int64_t nlist,
        const int32_t* __restrict__ pairs_sorted, const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off,
        int S, float radius, unsigned long long* __restrict__ counter, const int64_t* __restrict__ offs,
        float* __restrict__ out_dis, int64_t* __restrict__ out_ids) {
    extern __shared__ __align__(16) float s_lut[];
    __shared__ int s_pair[kQB];
    __shared__ long long s_item;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned below = (1u << lane) - 1u;
    const int tab = M * ksub;
    for (;;) {
        if (tid == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= item_off[nlist]) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, kCB, kQB, tid, s_pair);
        __syncthreads();
        const int pair = s_pair[warp];
        const int64_t seg = (int64_t)pair * S + it.c;
        int64_t cur = pair >= 0 ? offs[seg] : 0;
        const int64_t e = pair >= 0 ? offs[seg + 1] : 0;
        if (!__syncthreads_or(cur < e)) continue;
        stage_tables(tid, lut, tab, s_pair, s_lut);
        __syncthreads();
        if (cur < e) {                                       // warp-uniform
            const float* t = s_lut + warp * tab;
            const uint8_t* cl = codes + it.lbase * M;
            const int64_t* il = ids + it.lbase;
            for (int64_t h = it.v_begin; h < it.v_end && cur < e; h += 32) {
                const int64_t i = h + lane;
                const float s = i < it.v_end ? code_distance(t, M, ksub, cl + i * M, words) : 0.f;
                const bool hit = i < it.v_end && s < radius;
                const unsigned m = __ballot_sync(0xffffffffu, hit);
                const int64_t pos = cur + __popc(m & below);
                if (hit && pos < e) {
                    out_dis[pos] = s;
                    out_ids[pos] = il[i];
                }
                cur += __popc(m);
            }
        }
        __syncthreads();
    }
}

static size_t lut_bytes(int64_t nq, int nprobe, int M, int ksub) {
    return ivf::align256((size_t)nq * nprobe * M * ksub * sizeof(float));
}

static size_t table_smem(int M, int ksub) { return (size_t)kQB * M * ksub * sizeof(float); }

static bool pq_args_ok(int d, int M, int ksub) {
    return d > 0 && M >= 1 && d % M == 0 && ksub >= 1 && ksub <= 256 && (int64_t)M * ksub <= kMaxTable &&
           (size_t)d * sizeof(float) <= (size_t)kMaxResidual;
}

static bool code_words(const uint8_t* codes, int M) {
    return M % 4 == 0 && (reinterpret_cast<uintptr_t>(codes) & 3) == 0;
}

// the tables of the nq * nprobe pairs of a call
static int build_tables(const float* q, int64_t nq, int d, const float* coarse, int64_t nlist, const int64_t* probes,
                        int nprobe, const float* pq, int M, int ksub, float* lut, cudaStream_t st) {
    const size_t shm = (size_t)d * sizeof(float);
    if (shm > 48 * 1024)
        ISE_CUDA(cudaFuncSetAttribute(ivfpq_lut_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
    ivfpq_lut_kernel<<<(unsigned)(nq * nprobe), kThreads, shm, st>>>(q, d, coarse, nlist, probes, nprobe, pq, M, ksub,
                                                                     lut);
    ISE_LAUNCH_CHECK();
    return 0;
}

// persistent launch of one of the table-staging kernels with kQB tables of dynamic shared memory
template <typename Kernel, typename... Args>
static int launch_staged(ise_ctx* ctx, cudaStream_t st, int M, int ksub, Kernel kernel, Args... args) {
    const size_t shm = table_smem(M, ksub);
    ISE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
    return ivf::launch_persistent_shm(ctx, st, shm, kernel, args...);
}

}  // namespace

ISE_EXPORT size_t ise_ivfpq_search_workspace_bytes(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist,
                                                   int64_t max_list_len, int M, int ksub, int topk) {
    if (!ctx || M < 1 || ksub < 1 || ksub > 256 || (int64_t)M * ksub > kMaxTable ||
        !ivf::plan_args_ok(nq, nprobe, nlist, max_list_len, topk))
        return 0;
    const ivf::Plan p = ivf::search_plan(nq, nprobe, nlist, max_list_len, topk, kCB, kQB);
    return p.grouping + p.parts + p.level + lut_bytes(nq, nprobe, M, ksub);
}

ISE_EXPORT int ise_ivfpq_search(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* coarse_centroids,
                                int64_t nlist, const float* pq_centroids, int M, int ksub, const uint8_t* codes,
                                const int64_t* ids_sorted, const int64_t* list_off, int64_t max_list_len,
                                const int64_t* probes, int nprobe, int topk, float* out_val, int64_t* out_idx,
                                void* workspace, size_t workspace_bytes, void* stream) {
    using namespace ivf;
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(nq >= 0 && topk >= 1 && topk <= 128);
    ISE_CHECK_ARG(pq_args_ok(d, M, ksub));
    if (nq == 0) return 0;
    ISE_CHECK_ARG(plan_args_ok(nq, nprobe, nlist, max_list_len, topk));
    ISE_CHECK_ARG(q && coarse_centroids && pq_centroids && list_off && probes && out_val && out_idx && workspace);
    ISE_CHECK_ARG(max_list_len == 0 || (codes && ids_sorted));
    const size_t need = ise_ivfpq_search_workspace_bytes(ctx, nq, nprobe, nlist, max_list_len, M, ksub, topk);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const Plan p = search_plan(nq, nprobe, nlist, max_list_len, topk, kCB, kQB);

    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    const Grouping gr = carve_grouping(w, p);
    const size_t entries = (size_t)p.g * nq * topk;
    float* part_val = reinterpret_cast<float*>(take(w, align256(entries * sizeof(float))));
    int64_t* part_idx = reinterpret_cast<int64_t*>(take(w, align256(entries * sizeof(int64_t))));
    const size_t lv = level_entries(p, nq, topk);
    float* lvl_val = reinterpret_cast<float*>(take(w, align256(lv * sizeof(float))));
    int64_t* lvl_idx = reinterpret_cast<int64_t*>(take(w, align256(lv * sizeof(int64_t))));
    float* lut = reinterpret_cast<float*>(take(w, lut_bytes(nq, nprobe, M, ksub)));

    // 1. group the (query, probe slot) pairs by list; one table per pair
    int rc = group_pairs(ctx, p, gr, probes, nq, nprobe, nlist, list_off, topk, part_idx, st);
    if (rc) return rc;
    rc = build_tables(q, nq, d, coarse_centroids, nlist, probes, nprobe, pq_centroids, M, ksub, lut, st);
    if (rc) return rc;

    // 2. scan: persistent CTAs take work items from a counter
    const bool words = code_words(codes, M);
#define ISE_SCAN_ARGS lut, nq, M, ksub, words, codes, ids_sorted, list_off, nlist, gr.pairs_sorted, gr.qoff, \
                      gr.item_off, nprobe, p.S, topk, gr.counter, part_val, part_idx
    rc = topk <= 32 ? launch_staged(ctx, st, M, ksub, ivfpq_grouped_scan_kernel<32>, ISE_SCAN_ARGS)
                    : launch_staged(ctx, st, M, ksub, ivfpq_grouped_scan_kernel<128>, ISE_SCAN_ARGS);
#undef ISE_SCAN_ARGS
    if (rc) return rc;

    // 3. merge the nprobe * S partial lists of every query, at most kMergeFanIn at a time
    return merge_levels(ctx, p, nq, topk, ISE_METRIC_L2, part_val, part_idx, lvl_val, lvl_idx, out_val, out_idx,
                        stream);
}

ISE_EXPORT size_t ise_ivfpq_range_workspace_bytes(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist,
                                                  int64_t max_list_len, int M, int ksub) {
    if (!ctx || M < 1 || ksub < 1 || ksub > 256 || (int64_t)M * ksub > kMaxTable ||
        !ivf::plan_args_ok(nq, nprobe, nlist, max_list_len, 1))
        return 0;
    return ivf::range_workspace(ivf::range_plan(ctx, nq, nprobe, nlist, max_list_len, kCB, kQB)) +
           lut_bytes(nq, nprobe, M, ksub);
}

namespace {

// the range workspace: grouping, segment counts / offsets, offsets-scan scratch, then the tables
static int pq_range_setup(ise_ctx* ctx, int64_t nq, int d, int64_t nlist, int M, int ksub, const uint8_t* codes,
                          const int64_t* ids_sorted, const int64_t* list_off, int64_t max_list_len, int nprobe,
                          void* workspace, size_t workspace_bytes, ivf::RangeWork* rw, float** lut) {
    ISE_CHECK_ARG(ivf::plan_args_ok(nq, nprobe, nlist, max_list_len, 1));
    ISE_CHECK_ARG(pq_args_ok(d, M, ksub));
    ISE_CHECK_ARG(list_off && workspace);
    ISE_CHECK_ARG(max_list_len == 0 || (codes && ids_sorted));
    const size_t need = ise_ivfpq_range_workspace_bytes(ctx, nq, nprobe, nlist, max_list_len, M, ksub);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    const ivf::Plan p = ivf::range_plan(ctx, nq, nprobe, nlist, max_list_len, kCB, kQB);
    *rw = ivf::carve_range(workspace, p);
    *lut = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + ivf::range_workspace(p));
    return 0;
}

}  // namespace

ISE_EXPORT int ise_ivfpq_range_count(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* coarse_centroids,
                                     int64_t nlist, const float* pq_centroids, int M, int ksub, const uint8_t* codes,
                                     const int64_t* ids_sorted, const int64_t* list_off, int64_t max_list_len,
                                     const int64_t* probes, int nprobe, float radius, int64_t* lims, void* workspace,
                                     size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0 && lims != nullptr);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (nq == 0) {
        ISE_CUDA(cudaMemsetAsync(lims, 0, sizeof(int64_t), st));
        return 0;
    }
    ISE_CHECK_ARG(q && coarse_centroids && pq_centroids && probes);
    ivf::RangeWork rw;
    float* lut = nullptr;
    int rc = pq_range_setup(ctx, nq, d, nlist, M, ksub, codes, ids_sorted, list_off, max_list_len, nprobe, workspace,
                            workspace_bytes, &rw, &lut);
    if (rc) return rc;
    const ivf::Plan& p = rw.p;
    // segments no item writes (probe -1, chunk slots a list does not use) count 0; cnt[segs] = 0 ends the scan
    ISE_CUDA(cudaMemsetAsync(rw.cnt, 0, (size_t)(p.segs + 1) * sizeof(int64_t), st));
    rc = ivf::group_pairs(ctx, p, rw.gr, probes, nq, nprobe, nlist, list_off, 0, nullptr, st);
    if (rc) return rc;
    rc = build_tables(q, nq, d, coarse_centroids, nlist, probes, nprobe, pq_centroids, M, ksub, lut, st);
    if (rc) return rc;
    rc = launch_staged(ctx, st, M, ksub, ivfpq_range_count_kernel, (const float*)lut, M, ksub, code_words(codes, M),
                       codes, list_off, nlist, (const int32_t*)rw.gr.pairs_sorted, (const int32_t*)rw.gr.qoff,
                       (const int64_t*)rw.gr.item_off, p.S, radius, rw.gr.counter, rw.cnt);
    if (rc) return rc;
    return ise_internal_range_offsets(rw.cnt, nq, p.g, 0, rw.offs, lims, rw.lims_tmp, p.lims_tmp, stream);
}

ISE_EXPORT int ise_ivfpq_range_fill(ise_ctx* ctx, int64_t nq, int d, int64_t nlist, int M, int ksub,
                                    const uint8_t* codes, const int64_t* ids_sorted, const int64_t* list_off,
                                    int64_t max_list_len, int nprobe, float radius, float* out_dis, int64_t* out_ids,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(out_dis && out_ids);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    ivf::RangeWork rw;
    float* lut = nullptr;
    int rc = pq_range_setup(ctx, nq, d, nlist, M, ksub, codes, ids_sorted, list_off, max_list_len, nprobe, workspace,
                            workspace_bytes, &rw, &lut);
    if (rc) return rc;
    ISE_CUDA(cudaMemsetAsync(rw.gr.counter, 0, sizeof(unsigned long long), st));
    return launch_staged(ctx, st, M, ksub, ivfpq_range_fill_kernel, (const float*)lut, M, ksub, code_words(codes, M),
                         codes, ids_sorted, list_off, nlist, (const int32_t*)rw.gr.pairs_sorted,
                         (const int32_t*)rw.gr.qoff, (const int64_t*)rw.gr.item_off, rw.p.S, radius, rw.gr.counter,
                         (const int64_t*)rw.offs, out_dis, out_ids);
}
