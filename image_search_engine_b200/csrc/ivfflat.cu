// IndexIVFFlat search: exact FP32 scan of the probed inverted lists (faiss/IndexIVFFlat.cpp IVFFlatScanner,
// faiss/utils/distances.cpp fvec_inner_product / fvec_L2sqr) without an [nq, ntotal] score matrix.
//
//   grouping (ivf_grouping.cuh)  the nq * nprobe (query, probe slot) pairs sorted by list id, and per list
//                                ceil(queries / kQB) * chunks work items of chunks of kCB-row granules;
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
//
// Range search (faiss/IndexIVF.cpp range_search_preassigned, IVFFlatScanner::scan_codes_range) reuses the grouping and
// the work items, and replaces the top-k with two passes over the same score tiles:
//   ivfflat_range_count_kernel   hits of every (pair, chunk) segment, cnt[(q * nprobe + slot) * S + c] (query-major,
//                                so the flat range search's offsets scan, ise_internal_range_offsets in range.cu,
//                                gives every segment its output offset in
//                                Faiss's order: probe rank, then list position); lims[q] = offset of segment (q, 0, 0);
//   ivfflat_range_fill_kernel    re-runs the items with hits and writes each segment's hits in list order.
// Every kernel scores through score_tile, so search and range search return bit-identical distances.  S is capped at
// 256 / nprobe and so that the segment table holds at most max(2^22, nq * nprobe) entries.
#include "common.cuh"
#include "ivf_grouping.cuh"
#include "topk_list.cuh"

namespace {

using ivf::kThreads;                // 16 x 8 threads, 4 x 4 scores each
constexpr int kQB = 32;             // queries per work item
constexpr int kCB = 64;             // vectors per score tile (the chunk granule)
constexpr int kDK = 32;             // dimensions per shared-memory slice
constexpr int kWarps = kThreads / 32;

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

// s_s[r][j] = score of pair s_pair[r] against list vector t0 + j (r < kQB, j < nv) with the direct formulas: one
// sequential fmaf chain over the dimensions per (query, vector), sum x*y or sum (x-y)^2, zeros past d.  The queries
// and kCB vectors go through shared memory kDK dimensions at a time; each thread accumulates a 4 x 4 piece of the
// tile.  Search and both range passes score through this function only, so they see the same bits.
template <bool L2>
__device__ __forceinline__ void score_tile(int tid, const float* __restrict__ q, int d, bool vec, int nprobe,
                                           const int* s_pair, const float* __restrict__ xl, int64_t t0, int nv,
                                           float (*s_q)[kQB], float (*s_x)[kCB], float (*s_s)[kCB + 1]) {
    const int tx = tid & 15, ty = tid >> 4;
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
}

template <bool L2>
__device__ __forceinline__ bool in_range(float s, float radius) { return L2 ? s < radius : s > radius; }

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
    const int tid = threadIdx.x;
    const int sq = tid >> 2, sub = tid & 3;          // selection: four threads per query row of the tile
    const int64_t total = item_off[nlist];
    const float pad = L2 ? 3.402823466e+38f : -3.402823466e+38f;
    for (;;) {
        if (tid == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= total) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, kCB, kQB, tid, s_pair);
        const int64_t lbase = it.lbase, c = it.c;
        const float* xl = xs + lbase * (int64_t)d;
        __syncthreads();

        TopKList<KMAX> list;
        list.init(topk);
        for (int64_t t0 = it.v_begin; t0 < it.v_end; t0 += kCB) {
            const int nv = (int)min((int64_t)kCB, it.v_end - t0);
            score_tile<L2>(tid, q, d, vec, nprobe, s_pair, xl, t0, nv, s_q, s_x, s_s);
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
        if (sub == 0 && pair >= 0 && c == it.nch - 1)
            for (int64_t c2 = it.nch; c2 < S; ++c2) part_idx[((slot * S + c2) * nq + qi) * topk] = -1;
        __syncthreads();
    }
}

// range pass 1: cnt[pair * S + c] = hits (strict radius test) of pair against chunk c of its list.  Segments of probe
// -1 and chunk slots a list does not use keep the zero the caller wrote.  A warp takes rows warp, warp + kWarps, ...
// of the tile and counts 32 columns per ballot.
template <bool L2>
__global__ void __launch_bounds__(kThreads) ivfflat_range_count_kernel(
        const float* __restrict__ q, int d, bool vec, const float* __restrict__ xs,
        const int64_t* __restrict__ list_off, int64_t nlist, const int32_t* __restrict__ pairs_sorted,
        const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off, int nprobe, int S, float radius,
        unsigned long long* __restrict__ counter, int64_t* __restrict__ cnt) {
    __shared__ __align__(16) float s_q[kDK][kQB];
    __shared__ __align__(16) float s_x[kDK][kCB];
    __shared__ float s_s[kQB][kCB + 1];
    __shared__ int s_pair[kQB];
    __shared__ long long s_item;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t total = item_off[nlist];
    for (;;) {
        if (tid == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= total) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, kCB, kQB, tid, s_pair);
        const float* xl = xs + it.lbase * (int64_t)d;
        __syncthreads();
        int hits[kQB / kWarps];
#pragma unroll
        for (int i = 0; i < kQB / kWarps; ++i) hits[i] = 0;
        for (int64_t t0 = it.v_begin; t0 < it.v_end; t0 += kCB) {
            const int nv = (int)min((int64_t)kCB, it.v_end - t0);
            score_tile<L2>(tid, q, d, vec, nprobe, s_pair, xl, t0, nv, s_q, s_x, s_s);
#pragma unroll
            for (int i = 0; i < kQB / kWarps; ++i) {
                const int r = warp + i * kWarps;
#pragma unroll
                for (int h = 0; h < kCB; h += 32) {
                    const int j = h + lane;
                    hits[i] += __popc(__ballot_sync(0xffffffffu, j < nv && in_range<L2>(s_s[r][j], radius)));
                }
            }
            __syncthreads();
        }
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < kQB / kWarps; ++i) {
                const int pair = s_pair[warp + i * kWarps];
                if (pair >= 0) cnt[(int64_t)pair * S + it.c] = hits[i];
            }
        }
        __syncthreads();
    }
}

// range pass 2: the hits of segment (pair, c) go to out[offs[seg] .. offs[seg + 1]) in list position order.  An item
// whose segments are all empty is skipped before any vector is loaded, and a chunk stops once every segment is full.
// Each row has a cursor (s_cur, owned by the warp of the row); a ballot over 32 columns and popc prefixes give the
// slots.  Writes are bounded by the segment end.
template <bool L2>
__global__ void __launch_bounds__(kThreads) ivfflat_range_fill_kernel(
        const float* __restrict__ q, int d, bool vec, const float* __restrict__ xs, const int64_t* __restrict__ ids,
        const int64_t* __restrict__ list_off, int64_t nlist, const int32_t* __restrict__ pairs_sorted,
        const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off, int nprobe, int S, float radius,
        unsigned long long* __restrict__ counter, const int64_t* __restrict__ offs, float* __restrict__ out_dis,
        int64_t* __restrict__ out_ids) {
    __shared__ __align__(16) float s_q[kDK][kQB];
    __shared__ __align__(16) float s_x[kDK][kCB];
    __shared__ float s_s[kQB][kCB + 1];
    __shared__ int s_pair[kQB];
    __shared__ long long s_item;
    __shared__ long long s_cur[kQB], s_end[kQB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned below = (1u << lane) - 1u;
    const int64_t total = item_off[nlist];
    for (;;) {
        if (tid == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= total) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, kCB, kQB, tid, s_pair);
        const float* xl = xs + it.lbase * (int64_t)d;
        const int64_t* il = ids + it.lbase;
        __syncthreads();
        bool left = false;
#pragma unroll
        for (int i = 0; i < kQB / kWarps; ++i) {
            const int r = warp + i * kWarps;
            const int pair = s_pair[r];
            const int64_t seg = (int64_t)pair * S + it.c;
            const int64_t b = pair >= 0 ? offs[seg] : 0, e = pair >= 0 ? offs[seg + 1] : 0;
            if (lane == 0) { s_cur[r] = b; s_end[r] = e; }
            left |= b < e;
        }
        if (!__syncthreads_or(left)) continue;
        for (int64_t t0 = it.v_begin; t0 < it.v_end; t0 += kCB) {
            const int nv = (int)min((int64_t)kCB, it.v_end - t0);
            score_tile<L2>(tid, q, d, vec, nprobe, s_pair, xl, t0, nv, s_q, s_x, s_s);
            left = false;
#pragma unroll
            for (int i = 0; i < kQB / kWarps; ++i) {
                const int r = warp + i * kWarps;
                int64_t cur = s_cur[r];
                const int64_t e = s_end[r];
                if (cur < e) {                                   // warp-uniform
#pragma unroll
                    for (int h = 0; h < kCB; h += 32) {
                        const int j = h + lane;
                        const float s = s_s[r][j];
                        const bool hit = j < nv && in_range<L2>(s, radius);
                        const unsigned m = __ballot_sync(0xffffffffu, hit);
                        const int64_t pos = cur + __popc(m & below);
                        if (hit && pos < e) {
                            out_dis[pos] = s;
                            out_ids[pos] = il[t0 + j];
                        }
                        cur += __popc(m);
                    }
                    if (lane == 0) s_cur[r] = cur;
                    left |= cur < e;
                }
            }
            if (!__syncthreads_or(left)) break;
        }
    }
}

static bool vec_rows(const float* q, const float* xs, int d) {
    return (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(xs)) & 15) == 0;
}

}  // namespace

ISE_EXPORT size_t ise_ivfflat_search_workspace_bytes(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist,
                                                     int64_t max_list_len, int topk) {
    if (!ctx || !ivf::plan_args_ok(nq, nprobe, nlist, max_list_len, topk)) return 0;
    const ivf::Plan p = ivf::search_plan(nq, nprobe, nlist, max_list_len, topk, kCB, kQB);
    return p.grouping + p.parts + p.level;
}

ISE_EXPORT int ise_ivfflat_search(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* xs_sorted,
                                  const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist,
                                  int64_t max_list_len, const int64_t* probes, int nprobe, int metric, int topk,
                                  float* out_val, int64_t* out_idx, void* workspace, size_t workspace_bytes,
                                  void* stream) {
    using namespace ivf;
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
    const Plan p = search_plan(nq, nprobe, nlist, max_list_len, topk, kCB, kQB);

    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    const Grouping gr = carve_grouping(w, p);
    const size_t entries = (size_t)p.g * nq * topk;
    float* part_val = reinterpret_cast<float*>(take(w, align256(entries * sizeof(float))));
    int64_t* part_idx = reinterpret_cast<int64_t*>(take(w, align256(entries * sizeof(int64_t))));
    const size_t lv = level_entries(p, nq, topk);
    float* lvl_val = reinterpret_cast<float*>(take(w, align256(lv * sizeof(float))));
    int64_t* lvl_idx = reinterpret_cast<int64_t*>(take(w, align256(lv * sizeof(int64_t))));

    // 1. group the (query, probe slot) pairs by list
    int rc = group_pairs(ctx, p, gr, probes, nq, nprobe, nlist, list_off, topk, part_idx, st);
    if (rc) return rc;

    // 2. scan: persistent CTAs take work items from a counter
    const bool vec = vec_rows(q, xs_sorted, d);
    const bool l2 = metric == ISE_METRIC_L2;
#define ISE_SCAN_ARGS q, nq, d, vec, xs_sorted, ids_sorted, list_off, nlist, gr.pairs_sorted, gr.qoff, gr.item_off, \
                      nprobe, p.S, topk, gr.counter, part_val, part_idx
    if (topk <= 32)
        rc = l2 ? launch_persistent(ctx, st, ivfflat_scan_kernel<true, 32>, ISE_SCAN_ARGS)
                : launch_persistent(ctx, st, ivfflat_scan_kernel<false, 32>, ISE_SCAN_ARGS);
    else
        rc = l2 ? launch_persistent(ctx, st, ivfflat_scan_kernel<true, 128>, ISE_SCAN_ARGS)
                : launch_persistent(ctx, st, ivfflat_scan_kernel<false, 128>, ISE_SCAN_ARGS);
#undef ISE_SCAN_ARGS
    if (rc) return rc;

    // 3. merge the nprobe * S partial lists of every query, at most kMergeFanIn at a time
    return merge_levels(ctx, p, nq, topk, metric, part_val, part_idx, lvl_val, lvl_idx, out_val, out_idx, stream);
}

ISE_EXPORT size_t ise_ivfflat_range_workspace_bytes(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist,
                                                    int64_t max_list_len) {
    if (!ctx || !ivf::plan_args_ok(nq, nprobe, nlist, max_list_len, 1)) return 0;
    return ivf::range_workspace(ivf::range_plan(ctx, nq, nprobe, nlist, max_list_len, kCB, kQB));
}

namespace {

static int range_setup(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* xs_sorted,
                       const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist, int64_t max_list_len,
                       int nprobe, int metric, void* workspace, size_t workspace_bytes, ivf::RangeWork* rw) {
    ISE_CHECK_ARG(ivf::plan_args_ok(nq, nprobe, nlist, max_list_len, 1));
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(d > 0 && q && list_off && workspace);
    ISE_CHECK_ARG(max_list_len == 0 || (xs_sorted && ids_sorted));
    const size_t need = ise_ivfflat_range_workspace_bytes(ctx, nq, nprobe, nlist, max_list_len);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    *rw = ivf::carve_range(workspace, ivf::range_plan(ctx, nq, nprobe, nlist, max_list_len, kCB, kQB));
    return 0;
}

}  // namespace

ISE_EXPORT int ise_ivfflat_range_count(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* xs_sorted,
                                       const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist,
                                       int64_t max_list_len, const int64_t* probes, int nprobe, int metric,
                                       float radius, int64_t* lims, void* workspace, size_t workspace_bytes,
                                       void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0 && lims != nullptr);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (nq == 0) {
        ISE_CUDA(cudaMemsetAsync(lims, 0, sizeof(int64_t), st));
        return 0;
    }
    ISE_CHECK_ARG(probes != nullptr);
    ivf::RangeWork rw;
    int rc = range_setup(ctx, q, nq, d, xs_sorted, ids_sorted, list_off, nlist, max_list_len, nprobe, metric,
                         workspace, workspace_bytes, &rw);
    if (rc) return rc;
    const ivf::Plan& p = rw.p;
    // segments no item writes (probe -1, chunk slots a list does not use) count 0; cnt[segs] = 0 ends the scan
    ISE_CUDA(cudaMemsetAsync(rw.cnt, 0, (size_t)(p.segs + 1) * sizeof(int64_t), st));
    rc = ivf::group_pairs(ctx, p, rw.gr, probes, nq, nprobe, nlist, list_off, 0, nullptr, st);
    if (rc) return rc;
    const bool vec = vec_rows(q, xs_sorted, d);
#define ISE_COUNT_ARGS q, d, vec, xs_sorted, list_off, nlist, rw.gr.pairs_sorted, rw.gr.qoff, rw.gr.item_off, nprobe, \
                       p.S, radius, rw.gr.counter, rw.cnt
    rc = metric == ISE_METRIC_L2 ? ivf::launch_persistent(ctx, st, ivfflat_range_count_kernel<true>, ISE_COUNT_ARGS)
                                 : ivf::launch_persistent(ctx, st, ivfflat_range_count_kernel<false>, ISE_COUNT_ARGS);
#undef ISE_COUNT_ARGS
    if (rc) return rc;
    return ise_internal_range_offsets(rw.cnt, nq, p.g, 0, rw.offs, lims, rw.lims_tmp, p.lims_tmp, stream);
}

ISE_EXPORT int ise_ivfflat_range_fill(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* xs_sorted,
                                      const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist,
                                      int64_t max_list_len, int nprobe, int metric, float radius, float* out_dis,
                                      int64_t* out_ids, void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(out_dis && out_ids);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    ivf::RangeWork rw;
    int rc = range_setup(ctx, q, nq, d, xs_sorted, ids_sorted, list_off, nlist, max_list_len, nprobe, metric,
                         workspace, workspace_bytes, &rw);
    if (rc) return rc;
    ISE_CUDA(cudaMemsetAsync(rw.gr.counter, 0, sizeof(unsigned long long), st));
    const bool vec = vec_rows(q, xs_sorted, d);
#define ISE_FILL_ARGS q, d, vec, xs_sorted, ids_sorted, list_off, nlist, rw.gr.pairs_sorted, rw.gr.qoff, \
                      rw.gr.item_off, nprobe, rw.p.S, radius, rw.gr.counter, rw.offs, out_dis, out_ids
    rc = metric == ISE_METRIC_L2 ? ivf::launch_persistent(ctx, st, ivfflat_range_fill_kernel<true>, ISE_FILL_ARGS)
                                 : ivf::launch_persistent(ctx, st, ivfflat_range_fill_kernel<false>, ISE_FILL_ARGS);
#undef ISE_FILL_ARGS
    return rc;
}
