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
#include "ivf_grouping.cuh"
#include "topk_list.cuh"

namespace {

constexpr int kThreads = ivf::kThreads;      // the IVF kernels run on the shared persistent launch
constexpr int kStageBytes = 16 * 1024;      // shared memory per stage; two stages per CTA
constexpr int kCtasPerSm = 4;
constexpr int kMaxChunks = 256;             // ise_topk_merge: at most 256 lists per row
constexpr int kMinChunkRows = 256;
constexpr int kMaxWords = 32;               // 2048 bits
constexpr int64_t kPartialBudget = int64_t(1) << 24;
constexpr int64_t kSegmentBudget = int64_t(1) << 22;

using ivf::align256;
using ivf::take;

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// The state every kernel shares, flat and IVF: the thread's query words in registers and the row range the stage
// buffers stream.  NW = words per row rounded up to a power of two (the shared layout); only the first nw are read.
template <int NW>
struct Scan {
    static constexpr int kRows = kStageBytes / (8 * NW);    // rows per stage
    const uint8_t* codes;
    int64_t pitch, v0, v1;     // chunk rows [v0, v1)
    int nw, tpq, sub;
    int64_t qi;                // flat search: this thread's query (>= nq: none)
    bool valid;
    uint64_t q[NW];

    // the query row qrow (null: none) in registers
    __device__ __forceinline__ void load_query(const uint8_t* qrow, int nw_, int tpq_) {
        nw = nw_;
        tpq = tpq_;
        sub = threadIdx.x % tpq_;
        const uint64_t* qw = reinterpret_cast<const uint64_t*>(qrow);
#pragma unroll
        for (int w = 0; w < NW; ++w) q[w] = (qrow != nullptr && w < nw) ? __ldg(qw + w) : 0ull;
    }
    // the rows [v0_, v1_) of codes_ (row r at codes_ + r * pitch_) are the ones run() stages
    __device__ __forceinline__ void set_rows(const uint8_t* codes_, int64_t pitch_, int64_t v0_, int64_t v1_) {
        codes = codes_;
        pitch = pitch_;
        v0 = v0_;
        v1 = v1_;
    }
    // flat search: the CTA's queries (blockIdx.x) against column chunk blockIdx.y of S
    __device__ __forceinline__ void init(const uint8_t* qc, int64_t nq, const uint8_t* codes_, int64_t ntotal,
                                         int64_t pitch_, int nw_, int tpq_, int S) {
        qi = (int64_t)blockIdx.x * (kThreads / tpq_) + threadIdx.x / tpq_;
        valid = qi < nq;
        load_query(valid ? qc + qi * pitch_ : nullptr, nw_, tpq_);
        const int64_t cl = (ntotal + S - 1) / S;
        const int64_t a = min(ntotal, (int64_t)blockIdx.y * cl);
        set_rows(codes_, pitch_, a, min(ntotal, a + cl));
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

// merges the TopKLists of the TPQ lanes of a query (aligned lane groups) best first: lane sub == 0 gets emit(j, value,
// position) for j < topk, position 0x7fffffff past the lanes' entries.  Every lane of the warp takes part.
template <int KMAX, typename Emit>
__device__ __forceinline__ void merge_lanes(const TopKList<KMAX>& list, int topk, int tpq, int sub, Emit&& emit) {
    int head = 0;
    for (int j = 0; j < topk; ++j) {
        const bool live = head < topk && list.id[head] >= 0;
        float v = live ? list.v[head] : -CUDART_INF_F;
        int id = live ? list.id[head] : 0x7fffffff;
        int src = sub;
        for (int o = 1; o < tpq; o <<= 1) {
            const float v2 = __shfl_xor_sync(0xffffffffu, v, o);
            const int id2 = __shfl_xor_sync(0xffffffffu, id, o);
            const int src2 = __shfl_xor_sync(0xffffffffu, src, o);
            if (v2 > v || (v2 == v && id2 < id)) { v = v2; id = id2; src = src2; }
        }
        if (src == sub && id != 0x7fffffff) ++head;
        if (sub == 0) emit(j, v, id);
    }
}

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
    // the partial list of (chunk, query)
    const int64_t obase = ((int64_t)blockIdx.y * nq + sc.qi) * topk;
    merge_lanes(list, topk, tpq, sc.sub, [&](int j, float v, int id) {
        if (!sc.valid) return;
        part_val[obase + j] = id != 0x7fffffff ? -v : 3.402823466e+38f;
        part_idx[obase + j] = id != 0x7fffffff ? (int64_t)id : -1;
    });
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

// ---- IndexBinaryIVF: the probed lists of a query, grouped by list (ivf_grouping.cuh) ----------------------------------
// A work item is (list, block of qb = 128 / TPQ of its queries, chunk of its rows); the chunk streams through the same
// stages as the flat kernels, from the list's first code.  Thread t serves pair s_pair[t / TPQ]; rows are list
// positions (ascending id inside a list), mapped to ids through ids_sorted on output.

// the thread's pair of the item, its query words and the item's rows; the caller has synchronised after decode_item
template <int NW>
__device__ __forceinline__ int ivf_item_scan(Scan<NW>& sc, const ivf::Item& it, const int* s_pair,
                                             const uint8_t* __restrict__ qc, const uint8_t* __restrict__ codes,
                                             int64_t pitch, int nw, int tpq, int nprobe) {
    const int pair = s_pair[threadIdx.x / tpq];
    sc.load_query(pair >= 0 ? qc + (int64_t)(pair / nprobe) * pitch : nullptr, nw, tpq);
    sc.set_rows(codes + it.lbase * pitch, pitch, it.v_begin, it.v_end);
    return pair;
}

// search: the partial list of every (pair, chunk), part[((slot * S + c) * nq + q) * topk], as binary_knn_kernel's
template <int KMAX, int NW>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) binary_ivf_scan_kernel(
        const uint8_t* __restrict__ qc, int64_t nq, const uint8_t* __restrict__ codes, const int64_t* __restrict__ ids,
        int64_t pitch, int nw, int tpq, const int64_t* __restrict__ list_off, int64_t nlist,
        const int32_t* __restrict__ pairs_sorted, const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off,
        int nprobe, int S, int64_t cb, int topk, unsigned long long* __restrict__ counter, float* __restrict__ part_val,
        int64_t* __restrict__ part_idx) {
    using Sc = Scan<NW>;
    __shared__ __align__(16) uint64_t bufs[2][NW][Sc::kRows];
    __shared__ int s_pair[kThreads];
    __shared__ long long s_item;
    const int64_t total = item_off[nlist];
    for (;;) {
        if (threadIdx.x == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= total) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, cb, kThreads / tpq,
                                              threadIdx.x, s_pair);
        __syncthreads();
        Sc sc;
        const int pair = ivf_item_scan(sc, it, s_pair, qc, codes, pitch, nw, tpq, nprobe);
        TopKList<KMAX> list;
        list.init(topk);
        sc.run(bufs, [&](uint64_t (*buf)[Sc::kRows], int64_t r0, int n) {
            for (int r = sc.sub; r < n; r += sc.tpq) {
                const float s = -(float)sc.dist(buf, r);
                if (s > list.thr) list.insert(s, (int)(r0 + r));
            }
        });
        const int64_t qi = pair >= 0 ? pair / nprobe : 0, slot = pair >= 0 ? pair % nprobe : 0;
        const int64_t obase = ((slot * S + it.c) * nq + qi) * topk;
        const int64_t* il = ids + it.lbase;
        merge_lanes(list, topk, tpq, sc.sub, [&](int j, float v, int id) {
            if (pair < 0) return;
            part_val[obase + j] = id != 0x7fffffff ? -v : 3.402823466e+38f;
            part_idx[obase + j] = id != 0x7fffffff ? il[id] : -1;
        });
        // chunk slots this list does not use: an id -1 at the head makes ise_topk_merge skip the list
        if (sc.sub == 0 && pair >= 0 && it.c == it.nch - 1)
            for (int64_t c2 = it.nch; c2 < S; ++c2) part_idx[((slot * S + c2) * nq + qi) * topk] = -1;
        __syncthreads();
    }
}

// range pass 1: cnt[pair * S + c] = hits (distance < radius) of pair against chunk c of its list (query-major, so the
// offsets scan orders a query's results by probe rank, then list position).  Segments no item writes keep the caller's 0.
template <int NW>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) binary_ivf_range_count_kernel(
        const uint8_t* __restrict__ qc, const uint8_t* __restrict__ codes, int64_t pitch, int nw, int tpq,
        const int64_t* __restrict__ list_off, int64_t nlist, const int32_t* __restrict__ pairs_sorted,
        const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off, int nprobe, int S, int64_t cb,
        int radius, unsigned long long* __restrict__ counter, int64_t* __restrict__ cnt) {
    using Sc = Scan<NW>;
    __shared__ __align__(16) uint64_t bufs[2][NW][Sc::kRows];
    __shared__ int s_pair[kThreads];
    __shared__ long long s_item;
    const int64_t total = item_off[nlist];
    for (;;) {
        if (threadIdx.x == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= total) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, cb, kThreads / tpq,
                                              threadIdx.x, s_pair);
        __syncthreads();
        Sc sc;
        const int pair = ivf_item_scan(sc, it, s_pair, qc, codes, pitch, nw, tpq, nprobe);
        int hits = 0;
        sc.run(bufs, [&](uint64_t (*buf)[Sc::kRows], int64_t, int n) {
            for (int r = sc.sub; r < n; r += sc.tpq) hits += sc.dist(buf, r) < radius ? 1 : 0;
        });
        hits = group_sum(hits, tpq);
        if (sc.sub == 0 && pair >= 0) cnt[(int64_t)pair * S + it.c] = hits;
        __syncthreads();
    }
}

// range pass 2: the hits of segment (pair, c) go to out[offs[seg] .. offs[seg + 1]) in list order, as
// binary_range_fill_kernel writes them; an item whose segments are all empty is skipped before any code is loaded.
template <int NW>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) binary_ivf_range_fill_kernel(
        const uint8_t* __restrict__ qc, const uint8_t* __restrict__ codes, const int64_t* __restrict__ ids,
        int64_t pitch, int nw, int tpq, const int64_t* __restrict__ list_off, int64_t nlist,
        const int32_t* __restrict__ pairs_sorted, const int32_t* __restrict__ qoff, const int64_t* __restrict__ item_off,
        int nprobe, int S, int64_t cb, int radius, unsigned long long* __restrict__ counter,
        const int64_t* __restrict__ offs, int32_t* __restrict__ out_dis, int64_t* __restrict__ out_ids) {
    using Sc = Scan<NW>;
    __shared__ __align__(16) uint64_t bufs[2][NW][Sc::kRows];
    __shared__ int s_pair[kThreads];
    __shared__ long long s_item;
    const int64_t total = item_off[nlist];
    const int lane = threadIdx.x & 31;
    const unsigned group = (tpq == 32 ? 0xffffffffu : ((1u << tpq) - 1u)) << (lane & ~(tpq - 1) & 31);
    const unsigned below = (1u << lane) - 1u;
    for (;;) {
        if (threadIdx.x == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const int64_t w = s_item;
        if (w >= total) break;
        const ivf::Item it = ivf::decode_item(w, list_off, nlist, pairs_sorted, qoff, item_off, S, cb, kThreads / tpq,
                                              threadIdx.x, s_pair);
        __syncthreads();
        Sc sc;
        const int pair = ivf_item_scan(sc, it, s_pair, qc, codes, pitch, nw, tpq, nprobe);
        const int64_t seg = (int64_t)pair * S + it.c;
        int64_t cur = pair >= 0 ? offs[seg] : 0;
        const int64_t end = pair >= 0 ? offs[seg + 1] : 0;
        if (!__syncthreads_or(cur < end)) continue;       // the whole item: no hits
        const int64_t* il = ids + it.lbase;
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
                    out_ids[pos] = il[r0 + r];
                }
                cur += __popc(m);
            }
        });
    }
}

// IndexBinaryIVF::train: bit j of byte i -> coordinate 8 i + j (LSB first), 1 -> +1, 0 -> -1
__global__ void binary_to_real_kernel(const uint8_t* __restrict__ codes, int64_t n, int code_size, int64_t pitch,
                                      float* __restrict__ out) {
    const int64_t d = 8 * (int64_t)code_size;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * d; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / d, j = i % d;
        out[i] = (codes[r * pitch + j / 8] >> (j % 8)) & 1 ? 1.f : -1.f;
    }
}

// and back: bit = 1 iff the coordinate is > 0 (an exact 0 gives 0); bytes past code_size up to pitch are zero
__global__ void real_to_binary_kernel(const float* __restrict__ x, int64_t n, int code_size, int64_t pitch,
                                      uint8_t* __restrict__ codes) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * pitch; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / pitch, b = i % pitch;
        unsigned v = 0;
        if (b < code_size) {
            const float* xr = x + r * 8 * (int64_t)code_size + 8 * b;
#pragma unroll
            for (int j = 0; j < 8; ++j) v |= (xr[j] > 0.f ? 1u : 0u) << j;
        }
        codes[i] = (uint8_t)v;
    }
}

// threads per query from the number of queries a CTA can share its rows with (flat: nq; IVF: the queries per probed
// list): 1 fills a CTA with 128 queries; fewer share each query between 4 or 32 lanes
static int threads_per_query(int64_t n) { return n >= 256 ? 1 : n >= 32 ? 4 : 32; }

// words per row and their power-of-two bucket (the template argument of the kernels)
static void word_bucket(int code_size, int* nw, int* NW) {
    *nw = (code_size + 7) / 8;
    *NW = 1;
    while (*NW < *nw) *NW *= 2;
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
    word_bucket(code_size, &p.nw, &p.NW);
    p.tpq = threads_per_query(nq);
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

// ---- IndexBinaryIVF entry points ----------------------------------------------------------------------------------

namespace {

// the IVF scans' shape: word bucket, lanes per query from the average number of queries per probed list
// (nq * nprobe / nlist), and the chunk granule of one stage buffer
struct IvfShape {
    int nw, NW, tpq;
    int64_t cb;
};

static IvfShape ivf_shape(int64_t nq, int nprobe, int64_t nlist, int code_size) {
    IvfShape s;
    word_bucket(code_size, &s.nw, &s.NW);
    s.tpq = threads_per_query(ceil_div64(nq * nprobe, nlist));
    s.cb = kStageBytes / (8 * s.NW);
    return s;
}

static bool ivf_args_ok(int64_t nq, int nprobe, int64_t nlist, int64_t max_list_len, int code_size, int topk) {
    return ivf::plan_args_ok(nq, nprobe, nlist, max_list_len, topk) && max_list_len < ((int64_t)1 << 31) &&
           code_size >= 1 && code_size <= 8 * kMaxWords;
}

static size_t ivf_merged_bytes(int64_t nq, int topk) { return align256((size_t)nq * topk * sizeof(float)); }

}  // namespace

ISE_EXPORT size_t ise_binary_ivf_search_workspace_bytes(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist,
                                                        int64_t max_list_len, int code_size, int topk) {
    if (!ctx || !ivf_args_ok(nq, nprobe, nlist, max_list_len, code_size, topk)) return 0;
    const IvfShape sh = ivf_shape(nq, nprobe, nlist, code_size);
    const ivf::Plan p = ivf::search_plan(nq, nprobe, nlist, max_list_len, topk, sh.cb, kThreads / sh.tpq);
    return p.grouping + p.parts + p.level + ivf_merged_bytes(nq, topk);
}

ISE_EXPORT int ise_binary_ivf_search(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes_sorted,
                                     const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist,
                                     int64_t max_list_len, int code_size, int64_t pitch, const int64_t* probes,
                                     int nprobe, int topk, int32_t* out_dis, int64_t* out_idx, void* workspace,
                                     size_t workspace_bytes, void* stream) {
    using ivf::Grouping;
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0 && topk >= 1 && topk <= 128);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(ivf_args_ok(nq, nprobe, nlist, max_list_len, code_size, topk));
    ISE_CHECK_ARG(pitch >= code_size && pitch % 16 == 0);
    ISE_CHECK_ARG(q && list_off && probes && out_dis && out_idx && workspace);
    ISE_CHECK_ARG(max_list_len == 0 || (codes_sorted && ids_sorted));
    ISE_CHECK_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(codes_sorted)) & 15) == 0);
    const size_t need = ise_binary_ivf_search_workspace_bytes(ctx, nq, nprobe, nlist, max_list_len, code_size, topk);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const IvfShape sh = ivf_shape(nq, nprobe, nlist, code_size);
    const ivf::Plan p = ivf::search_plan(nq, nprobe, nlist, max_list_len, topk, sh.cb, kThreads / sh.tpq);

    uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
    const Grouping gr = ivf::carve_grouping(w, p);
    const size_t entries = (size_t)p.g * nq * topk;
    float* part_val = reinterpret_cast<float*>(take(w, align256(entries * sizeof(float))));
    int64_t* part_idx = reinterpret_cast<int64_t*>(take(w, align256(entries * sizeof(int64_t))));
    const size_t lv = ivf::level_entries(p, nq, topk);
    float* lvl_val = reinterpret_cast<float*>(take(w, align256(lv * sizeof(float))));
    int64_t* lvl_idx = reinterpret_cast<int64_t*>(take(w, align256(lv * sizeof(int64_t))));
    float* merged = reinterpret_cast<float*>(take(w, ivf_merged_bytes(nq, topk)));

    int rc = ivf::group_pairs(ctx, p, gr, probes, nq, nprobe, nlist, list_off, topk, part_idx, st);
    if (rc) return rc;
    rc = by_words(sh.NW, [&](auto nwc) {
        constexpr int NW = decltype(nwc)::value;
#define ISE_BIVF_ARGS q, nq, codes_sorted, ids_sorted, pitch, sh.nw, sh.tpq, list_off, nlist, gr.pairs_sorted, gr.qoff, \
                      gr.item_off, nprobe, p.S, p.cb, topk, gr.counter, part_val, part_idx
        return topk <= 32 ? ivf::launch_persistent(ctx, st, binary_ivf_scan_kernel<32, NW>, ISE_BIVF_ARGS)
                          : ivf::launch_persistent(ctx, st, binary_ivf_scan_kernel<128, NW>, ISE_BIVF_ARGS);
#undef ISE_BIVF_ARGS
    });
    if (rc) return rc;
    rc = ivf::merge_levels(ctx, p, nq, topk, ISE_METRIC_L2, part_val, part_idx, lvl_val, lvl_idx, merged, out_idx, stream);
    if (rc) return rc;
    const int64_t n = nq * topk;
    binary_dis_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(n, 256), (int64_t)ctx->sm_count * 8), 256, 0, st>>>(
            merged, out_idx, n, out_dis);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT size_t ise_binary_ivf_range_workspace_bytes(ise_ctx* ctx, int64_t nq, int nprobe, int64_t nlist,
                                                       int64_t max_list_len, int code_size) {
    if (!ctx || !ivf_args_ok(nq, nprobe, nlist, max_list_len, code_size, 1)) return 0;
    const IvfShape sh = ivf_shape(nq, nprobe, nlist, code_size);
    return ivf::range_workspace(ivf::range_plan(ctx, nq, nprobe, nlist, max_list_len, sh.cb, kThreads / sh.tpq));
}

namespace {

static int ivf_range_setup(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes_sorted,
                           const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist, int64_t max_list_len,
                           int code_size, int64_t pitch, int nprobe, void* workspace, size_t workspace_bytes,
                           IvfShape* sh, ivf::RangeWork* rw) {
    ISE_CHECK_ARG(ivf_args_ok(nq, nprobe, nlist, max_list_len, code_size, 1));
    ISE_CHECK_ARG(pitch >= code_size && pitch % 16 == 0);
    ISE_CHECK_ARG(q && list_off && workspace);
    ISE_CHECK_ARG(max_list_len == 0 || (codes_sorted && ids_sorted));
    ISE_CHECK_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(codes_sorted)) & 15) == 0);
    const size_t need = ise_binary_ivf_range_workspace_bytes(ctx, nq, nprobe, nlist, max_list_len, code_size);
    if (workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
    *sh = ivf_shape(nq, nprobe, nlist, code_size);
    *rw = ivf::carve_range(workspace, ivf::range_plan(ctx, nq, nprobe, nlist, max_list_len, sh->cb, kThreads / sh->tpq));
    return 0;
}

}  // namespace

ISE_EXPORT int ise_binary_ivf_range_count(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes_sorted,
                                          const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist,
                                          int64_t max_list_len, int code_size, int64_t pitch, const int64_t* probes,
                                          int nprobe, int radius, int64_t* lims, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0 && lims != nullptr);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (nq == 0) {
        ISE_CUDA(cudaMemsetAsync(lims, 0, sizeof(int64_t), st));
        return 0;
    }
    ISE_CHECK_ARG(probes != nullptr);
    IvfShape sh;
    ivf::RangeWork rw;
    int rc = ivf_range_setup(ctx, q, nq, codes_sorted, ids_sorted, list_off, nlist, max_list_len, code_size, pitch,
                             nprobe, workspace, workspace_bytes, &sh, &rw);
    if (rc) return rc;
    const ivf::Plan& p = rw.p;
    // segments no item writes (probe -1, chunk slots a list does not use) count 0; cnt[segs] = 0 ends the scan
    ISE_CUDA(cudaMemsetAsync(rw.cnt, 0, (size_t)(p.segs + 1) * sizeof(int64_t), st));
    rc = ivf::group_pairs(ctx, p, rw.gr, probes, nq, nprobe, nlist, list_off, 0, nullptr, st);
    if (rc) return rc;
    rc = by_words(sh.NW, [&](auto nwc) {
        constexpr int NW = decltype(nwc)::value;
        return ivf::launch_persistent(ctx, st, binary_ivf_range_count_kernel<NW>, q, codes_sorted, pitch, sh.nw, sh.tpq,
                                      list_off, nlist, rw.gr.pairs_sorted, rw.gr.qoff, rw.gr.item_off, nprobe, p.S,
                                      p.cb, radius, rw.gr.counter, rw.cnt);
    });
    if (rc) return rc;
    return ise_internal_range_offsets(rw.cnt, nq, p.g, 0, rw.offs, lims, rw.lims_tmp, p.lims_tmp, stream);
}

ISE_EXPORT int ise_binary_ivf_range_fill(ise_ctx* ctx, const uint8_t* q, int64_t nq, const uint8_t* codes_sorted,
                                         const int64_t* ids_sorted, const int64_t* list_off, int64_t nlist,
                                         int64_t max_list_len, int code_size, int64_t pitch, int nprobe, int radius,
                                         int32_t* out_dis, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                                         void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && nq >= 0);
    if (nq == 0) return 0;
    ISE_CHECK_ARG(out_dis && out_ids);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    IvfShape sh;
    ivf::RangeWork rw;
    int rc = ivf_range_setup(ctx, q, nq, codes_sorted, ids_sorted, list_off, nlist, max_list_len, code_size, pitch,
                             nprobe, workspace, workspace_bytes, &sh, &rw);
    if (rc) return rc;
    ISE_CUDA(cudaMemsetAsync(rw.gr.counter, 0, sizeof(unsigned long long), st));
    return by_words(sh.NW, [&](auto nwc) {
        constexpr int NW = decltype(nwc)::value;
        return ivf::launch_persistent(ctx, st, binary_ivf_range_fill_kernel<NW>, q, codes_sorted, ids_sorted, pitch,
                                      sh.nw, sh.tpq, list_off, nlist, rw.gr.pairs_sorted, rw.gr.qoff, rw.gr.item_off,
                                      nprobe, rw.p.S, rw.p.cb, radius, rw.gr.counter, rw.offs, out_dis, out_ids);
    });
}

ISE_EXPORT int ise_binary_to_real(ise_ctx* ctx, const uint8_t* codes, int64_t n, int code_size, int64_t pitch,
                                  float* out, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && n >= 0 && code_size >= 1 && pitch >= code_size);
    if (n == 0) return 0;
    ISE_CHECK_ARG(codes && out);
    DeviceGuard guard(ctx->device);
    const int64_t m = n * 8 * (int64_t)code_size;
    binary_to_real_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(m, 256), (int64_t)ctx->sm_count * 8), 256, 0,
                            (cudaStream_t)stream>>>(codes, n, code_size, pitch, out);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_real_to_binary(ise_ctx* ctx, const float* x, int64_t n, int code_size, int64_t pitch,
                                  uint8_t* codes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr && n >= 0 && code_size >= 1 && pitch >= code_size);
    if (n == 0) return 0;
    ISE_CHECK_ARG(x && codes);
    DeviceGuard guard(ctx->device);
    const int64_t m = n * pitch;
    real_to_binary_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(m, 256), (int64_t)ctx->sm_count * 8), 256, 0,
                            (cudaStream_t)stream>>>(x, n, code_size, pitch, codes);
    ISE_LAUNCH_CHECK();
    return 0;
}
