// IndexBinaryFlat: exact Hamming kNN and range search over packed binary codes (faiss/IndexBinaryFlat.cpp,
// faiss/utils/hamming.cpp hammings_knn_hc / hamming_range_search), without an [nq, ntotal] distance matrix.
//
// Codes and queries are rows of `pitch` bytes (a multiple of 16, zero bytes past code_size), read as nw = ceil(code_size
// / 8) 64-bit words; the distance of a pair is sum_w popc(q_w ^ x_w), exact in int32 and in float (<= 2048).
//
// A CTA takes (block of QB queries, column chunk c of the database).  The chunk streams through shared memory in
// stages of kStageBytes, double-buffered with cp.async and stored word-major (s[w][row]), so that the lanes of a warp
// read one row (a broadcast) or consecutive rows (conflict-free).  TPQ = 128 / QB threads share a query: thread sub of
// a query scores rows sub, sub + TPQ, ... of every stage, in ascending id.  TPQ is 1 for large batches and 4 or 32 for
// small ones, so that one image's descriptors or a single query still give every thread work.
//   binary_knn_kernel          per thread a TopKList of -distance (insertion is strict, so among equal distances the
//                              lowest ids stay); the TPQ lists of a query merge by shuffles into the partial list of
//                              (chunk, query); ise_topk_merge joins the S chunk lists; binary_dis_kernel turns the
//                              float distances into int32 (2^31 - 1 with id -1 on padding);
//   binary_range_count_kernel  hits (distance < radius) of every (query, chunk) segment, cnt[q * S + c]; the offsets
//                              scan of range.cu (ise_internal_range_offsets) gives each segment its output offset, so
//                              a query's results come in ascending id;
//   binary_range_fill_kernel   re-scores the segments with hits and writes them in id order: a ballot over the TPQ
//                              lanes of a query and popc prefixes give the slots, no sort.
// S (chunks) is chosen so that the grid fills kCtasPerSm CTAs per SM, and capped at 256 (one merge), at ntotal / 256
// rows, and so that the partial lists hold at most max(2^24, nq * topk) entries (search) or the segment table at most
// max(2^22, nq) segments (range search).
#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "topk_list.cuh"

namespace {

constexpr int kThreads = 128;
constexpr int kStageBytes = 16 * 1024;      // shared memory per stage; two stages per CTA
constexpr int kCtasPerSm = 4;
constexpr int kMaxChunks = 256;             // ise_topk_merge: at most 256 lists per row
constexpr int kMinChunkRows = 256;
constexpr int kMaxWords = 32;               // 2048 bits
constexpr int64_t kPartialBudget = int64_t(1) << 24;
constexpr int64_t kSegmentBudget = int64_t(1) << 22;

static inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// The state every kernel shares: the CTA's queries and chunk, the thread's query words in registers, and the stage
// buffers.  NW = words per row rounded up to a power of two (the shared layout); only the first nw are read.
template <int NW>
struct Scan {
    static constexpr int kRows = kStageBytes / (8 * NW);    // rows per stage
    const uint8_t* codes;
    int64_t pitch, v0, v1;     // chunk rows [v0, v1)
    int nw, tpq, sub;
    int64_t qi;                // this thread's query (>= nq: none)
    bool valid;
    uint64_t q[NW];

    __device__ __forceinline__ void init(const uint8_t* qc, int64_t nq, const uint8_t* codes_, int64_t ntotal,
                                         int64_t pitch_, int nw_, int tpq_, int S) {
        codes = codes_;
        pitch = pitch_;
        nw = nw_;
        tpq = tpq_;
        sub = threadIdx.x % tpq_;
        qi = (int64_t)blockIdx.x * (kThreads / tpq_) + threadIdx.x / tpq_;
        valid = qi < nq;
        const int64_t cl = (ntotal + S - 1) / S;
        v0 = min(ntotal, (int64_t)blockIdx.y * cl);
        v1 = min(ntotal, v0 + cl);
        const uint64_t* qrow = reinterpret_cast<const uint64_t*>(qc + (valid ? qi : 0) * pitch);
#pragma unroll
        for (int w = 0; w < NW; ++w) q[w] = (valid && w < nw) ? __ldg(qrow + w) : 0ull;
    }
    __device__ __forceinline__ int stages() const { return (int)((v1 - v0 + kRows - 1) / kRows); }
    __device__ __forceinline__ int64_t stage_row(int s) const { return v0 + (int64_t)s * kRows; }
    __device__ __forceinline__ int stage_len(int s) const { return (int)min((int64_t)kRows, v1 - stage_row(s)); }

    // cp.async of stage s into buf (word-major), one commit group
    __device__ __forceinline__ void issue(uint64_t (*buf)[kRows], int s) const {
        const int64_t r0 = stage_row(s);
        const int n = stage_len(s);
        for (int e = threadIdx.x; e < n * NW; e += kThreads) {
            const int r = e / NW, w = e % NW;
            if (w < nw) cp_async8(&buf[w][r], codes + (r0 + r) * pitch + 8 * w);
        }
        cp_async_commit();
    }
    __device__ __forceinline__ int dist(uint64_t (*buf)[kRows], int r) const {
        int acc = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w)
            if (w < nw) acc += __popcll(q[w] ^ buf[w][r]);
        return acc;
    }

    // runs body(buf, stage row, stage length) over every stage, double-buffered; body may not write to buf
    template <typename Body>
    __device__ __forceinline__ void run(uint64_t (*bufs)[NW][kRows], Body&& body) const {
        const int ns = stages();
        if (ns > 0) issue(bufs[0], 0);
        for (int s = 0; s < ns; ++s) {
            if (s + 1 < ns) {
                issue(bufs[(s + 1) & 1], s + 1);
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();
            body(bufs[s & 1], stage_row(s), stage_len(s));
            __syncthreads();
        }
    }
};

template <int KMAX, int NW>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) binary_knn_kernel(
        const uint8_t* __restrict__ qc, int64_t nq, const uint8_t* __restrict__ codes, int64_t ntotal, int64_t pitch,
        int nw, int tpq, int S, int topk, float* __restrict__ part_val, int64_t* __restrict__ part_idx) {
    using Sc = Scan<NW>;
    __shared__ __align__(16) uint64_t bufs[2][NW][Sc::kRows];
    Sc sc;
    sc.init(qc, nq, codes, ntotal, pitch, nw, tpq, S);
    TopKList<KMAX> list;
    list.init(topk);
    sc.run(bufs, [&](uint64_t (*buf)[Sc::kRows], int64_t r0, int n) {
        for (int r = sc.sub; r < n; r += sc.tpq) {
            const float s = -(float)sc.dist(buf, r);
            if (s > list.thr) list.insert(s, (int)(r0 + r));
        }
    });
    // merge the lists of the TPQ lanes of a query (aligned lane groups) into the partial list of (chunk, query)
    const int64_t obase = ((int64_t)blockIdx.y * nq + sc.qi) * topk;
    int head = 0;
    for (int j = 0; j < topk; ++j) {
        const bool live = head < topk && list.id[head] >= 0;
        float v = live ? list.v[head] : -CUDART_INF_F;
        int id = live ? list.id[head] : 0x7fffffff;
        int src = sc.sub;
        for (int o = 1; o < tpq; o <<= 1) {
            const float v2 = __shfl_xor_sync(0xffffffffu, v, o);
            const int id2 = __shfl_xor_sync(0xffffffffu, id, o);
            const int src2 = __shfl_xor_sync(0xffffffffu, src, o);
            if (v2 > v || (v2 == v && id2 < id)) { v = v2; id = id2; src = src2; }
        }
        if (src == sc.sub && id != 0x7fffffff) ++head;
        if (sc.sub == 0 && sc.valid) {
            part_val[obase + j] = id != 0x7fffffff ? -v : 3.402823466e+38f;
            part_idx[obase + j] = id != 0x7fffffff ? (int64_t)id : -1;
        }
    }
}

__global__ void binary_dis_kernel(const float* __restrict__ val, const int64_t* __restrict__ idx, int64_t n,
                                  int32_t* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = idx[i] < 0 ? 0x7fffffff : (int32_t)val[i];
}

// sum of v over the TPQ lanes of a query (every lane of the group gets it)
__device__ __forceinline__ int group_sum(int v, int tpq) {
    for (int o = 1; o < tpq; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int NW>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) binary_range_count_kernel(
        const uint8_t* __restrict__ qc, int64_t nq, const uint8_t* __restrict__ codes, int64_t ntotal, int64_t pitch,
        int nw, int tpq, int S, int radius, int64_t* __restrict__ cnt) {
    using Sc = Scan<NW>;
    __shared__ __align__(16) uint64_t bufs[2][NW][Sc::kRows];
    Sc sc;
    sc.init(qc, nq, codes, ntotal, pitch, nw, tpq, S);
    int hits = 0;
    sc.run(bufs, [&](uint64_t (*buf)[Sc::kRows], int64_t, int n) {
        for (int r = sc.sub; r < n; r += sc.tpq) hits += sc.dist(buf, r) < radius ? 1 : 0;
    });
    hits = group_sum(hits, tpq);
    if (sc.sub == 0 && sc.valid) cnt[sc.qi * S + blockIdx.y] = hits;
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) cnt[nq * S] = 0;   // the offsets scan's last entry
}

// writes the hits of segment (query, chunk) to out[offs[seg] .. offs[seg + 1]) in id order.  Every lane of a query group
// runs the same number of steps (rows r0 + step * TPQ + sub), so the group's ballot gives each hit its slot; writes are
// bounded by the segment end.
template <int NW>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) binary_range_fill_kernel(
        const uint8_t* __restrict__ qc, int64_t nq, const uint8_t* __restrict__ codes, int64_t ntotal, int64_t pitch,
        int nw, int tpq, int S, int radius, const int64_t* __restrict__ offs, int32_t* __restrict__ out_dis,
        int64_t* __restrict__ out_ids) {
    using Sc = Scan<NW>;
    __shared__ __align__(16) uint64_t bufs[2][NW][Sc::kRows];
    Sc sc;
    sc.init(qc, nq, codes, ntotal, pitch, nw, tpq, S);
    const int64_t seg = sc.qi * S + blockIdx.y;
    int64_t cur = sc.valid ? offs[seg] : 0;
    const int64_t end = sc.valid ? offs[seg + 1] : 0;
    if (!__syncthreads_or(cur < end)) return;        // the whole CTA: no hits in this chunk
    const int lane = threadIdx.x & 31;
    const unsigned group = (tpq == 32 ? 0xffffffffu : ((1u << tpq) - 1u)) << (lane & ~(tpq - 1) & 31);
    const unsigned below = (1u << lane) - 1u;
    sc.run(bufs, [&](uint64_t (*buf)[Sc::kRows], int64_t r0, int n) {
        for (int base = 0; base < n; base += sc.tpq) {
            const int r = base + sc.sub;
            int dis = 0;
            bool hit = false;
            if (r < n) {
                dis = sc.dist(buf, r);
                hit = dis < radius;
            }
            const unsigned m = __ballot_sync(0xffffffffu, hit) & group;
            const int64_t pos = cur + __popc(m & below);
            if (hit && pos < end) {
                out_dis[pos] = dis;
                out_ids[pos] = r0 + r;
            }
            cur += __popc(m);
        }
    });
}

struct Plan {
    int nw, NW, tpq, S;
    int64_t qblocks;
    size_t parts_val, parts_idx, merged;   // search: partial lists, merged float distances
    int64_t segs;                          // range: nq * S (query, chunk) segments
    size_t seg, lims_tmp;                  // range: one int64 per segment + 1 (counts, offsets); offsets-scan scratch
};

static bool args_ok(int64_t nq, int64_t ntotal, int code_size, int64_t pitch) {
    return nq >= 0 && ntotal >= 0 && ntotal < ((int64_t)1 << 31) && code_size >= 1 && code_size <= 8 * kMaxWords &&
           pitch >= code_size && pitch % 16 == 0;
}

// budget: the largest S the caller's workspace formula allows
static Plan make_plan(const ise_ctx* ctx, int64_t nq, int64_t ntotal, int code_size, int64_t budget) {
    Plan p{};
    p.nw = (code_size + 7) / 8;
    p.NW = 1;
    while (p.NW < p.nw) p.NW *= 2;
    // threads per query: 1 fills a CTA with 128 queries; small batches share each query between 4 or 32 lanes
    p.tpq = nq >= 256 ? 1 : nq >= 32 ? 4 : 32;
    p.qblocks = std::max<int64_t>(1, ceil_div64(nq, kThreads / p.tpq));
    const int64_t fill = std::max<int64_t>(1, (int64_t)ctx->sm_count * kCtasPerSm / p.qblocks);
    p.S = (int)std::max<int64_t>(1, std::min({fill, (int64_t)kMaxChunks, ntotal / kMinChunkRows, budget}));
    return p;
}

static Plan knn_plan(const ise_ctx* ctx, int64_t nq, int64_t ntotal, int code_size, int topk) {
    Plan p = make_plan(ctx, nq, ntotal, code_size, kPartialBudget / std::max<int64_t>(1, nq * topk));
    const size_t entries = (size_t)p.S * nq * topk;
    p.parts_val = align256(entries * sizeof(float));
    p.parts_idx = align256(entries * sizeof(int64_t));
    p.merged = align256((size_t)nq * topk * sizeof(float));
    return p;
}

static Plan range_plan(ise_ctx* ctx, int64_t nq, int64_t ntotal, int code_size) {
    Plan p = make_plan(ctx, nq, ntotal, code_size, kSegmentBudget / std::max<int64_t>(1, nq));
    p.segs = (int64_t)p.S * nq;
    p.seg = align256((size_t)(p.segs + 1) * sizeof(int64_t));
    p.lims_tmp = align256(ise_range_lims_workspace_bytes(ctx, p.segs));
    return p;
}

static uint8_t* take(uint8_t*& w, size_t bytes) {
    uint8_t* r = w;
    w += bytes;
    return r;
}

// calls f(std::integral_constant<int, NW>) for the plan's word bucket
template <typename F>
static int by_words(int NW, F&& f) {
    switch (NW) {
        case 1: return f(std::integral_constant<int, 1>());
        case 2: return f(std::integral_constant<int, 2>());
        case 4: return f(std::integral_constant<int, 4>());
        case 8: return f(std::integral_constant<int, 8>());
        case 16: return f(std::integral_constant<int, 16>());
        default: return f(std::integral_constant<int, 32>());
    }
}

}  // namespace

ISE_EXPORT size_t ise_binary_knn_workspace_bytes(ise_ctx* ctx, int64_t nq, int64_t ntotal, int code_size, int topk) {
    if (!ctx || nq <= 0 || !args_ok(nq, ntotal, code_size, 16 * ((code_size + 15) / 16)) || topk < 1 || topk > 128)
        return 0;
    const Plan p = knn_plan(ctx, nq, ntotal, code_size, topk);
    return p.parts_val + p.parts_idx + p.merged;
}

ISE_EXPORT int ise_binary_knn(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes, int64_t ntotal,
                              int code_size, int64_t pitch, int topk, int32_t* out_dis, int64_t* out_idx,
                              void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(args_ok(nq, ntotal, code_size, pitch) && topk >= 1 && topk <= 128);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(q && out_dis && out_idx && workspace && (ntotal == 0 || codes));
    ISE_CHECK_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(codes)) & 15) == 0);
    const size_t need = ise_binary_knn_workspace_bytes(ctx, nq, ntotal, code_size, topk);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const Plan p = knn_plan(ctx, nq, ntotal, code_size, topk);
    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    float* part_val = reinterpret_cast<float*>(take(w, p.parts_val));
    int64_t* part_idx = reinterpret_cast<int64_t*>(take(w, p.parts_idx));
    float* merged = reinterpret_cast<float*>(take(w, p.merged));
    const dim3 grid((unsigned)p.qblocks, (unsigned)p.S);
    int rc = by_words(p.NW, [&](auto nwc) {
        constexpr int NW = decltype(nwc)::value;
        if (topk <= 32)
            binary_knn_kernel<32, NW><<<grid, kThreads, 0, st>>>(q, nq, codes, ntotal, pitch, p.nw, p.tpq, p.S, topk,
                                                                  part_val, part_idx);
        else
            binary_knn_kernel<128, NW><<<grid, kThreads, 0, st>>>(q, nq, codes, ntotal, pitch, p.nw, p.tpq, p.S, topk,
                                                                   part_val, part_idx);
        ISE_LAUNCH_CHECK();
        return 0;
    });
    if (rc) return rc;
    rc = ise_topk_merge(ctx, part_val, part_idx, p.S, nq, topk, ISE_METRIC_L2, merged, out_idx, stream);
    if (rc) return rc;
    const int64_t n = nq * topk;
    binary_dis_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(n, 256), (int64_t)ctx->sm_count * 8), 256, 0, st>>>(
            merged, out_idx, n, out_dis);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT size_t ise_binary_range_workspace_bytes(ise_ctx* ctx, int64_t nq, int64_t ntotal, int code_size) {
    if (!ctx || nq <= 0 || !args_ok(nq, ntotal, code_size, 16 * ((code_size + 15) / 16))) return 0;
    const Plan p = range_plan(ctx, nq, ntotal, code_size);
    return 2 * p.seg + p.lims_tmp;
}

int ise_internal_range_offsets(const int64_t* cnt, int64_t rows, int64_t per_row, int64_t base,
                               int64_t* offs, int64_t* lims, void* tmp, size_t tmp_bytes, void* stream);   // range.cu

namespace {

struct RangeWork {
    Plan p;
    int64_t *cnt, *offs;   // per (query, chunk) segment: hits, output offset (offs[segs] = total)
    void* lims_tmp;
};

static int range_setup(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes, int64_t ntotal,
                       int code_size, int64_t pitch, void* workspace, size_t workspace_bytes, RangeWork* rw) {
    ISE_CHECK_ARG(args_ok(nq, ntotal, code_size, pitch));
    ISE_CHECK_ARG(q && workspace && (ntotal == 0 || codes));
    ISE_CHECK_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(codes)) & 15) == 0);
    const size_t need = ise_binary_range_workspace_bytes(ctx, nq, ntotal, code_size);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    rw->p = range_plan(ctx, nq, ntotal, code_size);
    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    rw->cnt = reinterpret_cast<int64_t*>(take(w, rw->p.seg));
    rw->offs = reinterpret_cast<int64_t*>(take(w, rw->p.seg));
    rw->lims_tmp = take(w, rw->p.lims_tmp);
    return 0;
}

}  // namespace

ISE_EXPORT int ise_binary_range_count(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes, int64_t ntotal,
                                      int code_size, int64_t pitch, int radius, int64_t* lims, void* workspace,
                                      size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0 && lims != nullptr);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (nq == 0) {
        ISE_CUDA(cudaMemsetAsync(lims, 0, sizeof(int64_t), st));
        return 0;
    }
    RangeWork rw;
    int rc = range_setup(ctx, q, nq, codes, ntotal, code_size, pitch, workspace, workspace_bytes, &rw);
    if (rc) return rc;
    const Plan& p = rw.p;
    const dim3 grid((unsigned)p.qblocks, (unsigned)p.S);
    rc = by_words(p.NW, [&](auto nwc) {
        constexpr int NW = decltype(nwc)::value;
        binary_range_count_kernel<NW><<<grid, kThreads, 0, st>>>(q, nq, codes, ntotal, pitch, p.nw, p.tpq, p.S, radius,
                                                                  rw.cnt);
        ISE_LAUNCH_CHECK();
        return 0;
    });
    if (rc) return rc;
    return ise_internal_range_offsets(rw.cnt, nq, p.S, 0, rw.offs, lims, rw.lims_tmp, p.lims_tmp, stream);
}

ISE_EXPORT int ise_binary_range_fill(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes, int64_t ntotal,
                                     int code_size, int64_t pitch, int radius, int32_t* out_dis, int64_t* out_ids,
                                     void* workspace, size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(out_dis && out_ids);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    RangeWork rw;
    int rc = range_setup(ctx, q, nq, codes, ntotal, code_size, pitch, workspace, workspace_bytes, &rw);
    if (rc) return rc;
    const Plan& p = rw.p;
    const dim3 grid((unsigned)p.qblocks, (unsigned)p.S);
    return by_words(p.NW, [&](auto nwc) {
        constexpr int NW = decltype(nwc)::value;
        binary_range_fill_kernel<NW><<<grid, kThreads, 0, st>>>(q, nq, codes, ntotal, pitch, p.nw, p.tpq, p.S, radius,
                                                                 rw.offs, out_dis, out_ids);
        ISE_LAUNCH_CHECK();
        return 0;
    });
}
