// BoVW histogram (+ fused Okapi/BM25 tf weighting): CTAs walk images, shared-memory-privatised counts,
// ids read once into registers (next image prefetched), 128-bit row stores with the counters cleared in the same sweep.  HBM-bound: 8 B per descriptor id read plus one
// write of the [n_img, k] matrix.
// Replaces create_visual_word_histogram (bag_of_visual_words.py:98-106: np.histogram per image into a
// float64 matrix) and OkapiTransformer.transform (utils.py:153-202).
#include <stdlib.h>

#include <climits>

#include "common.cuh"

namespace {

constexpr int kThreads = 128;   // 8 CTAs per SM: the per-image critical path (barriers, FP64 edges) wants many images in flight
constexpr int kMaxSmemBins = 12 * 1024;  // 48 KiB of int32 counters

// np.histogram(a, bins=k) for integer input, restated with the same float64 operations
// (numpy/lib/_histograms_impl.py: _get_outer_edges, linspace edges, f_indices + edge corrections).
struct NumpyBins {
    double first, last, denom, step, kscale;
    int k;
    __device__ __forceinline__ void setup(int64_t mn, int64_t mx, int k_) {
        k = k_;
        if (mn == mx) { first = (double)mn - 0.5; last = (double)mx + 0.5; }
        else { first = (double)mn; last = (double)mx; }
        denom = __dsub_rn(last, first);       // _unsigned_subtract(last_edge, first_edge)
        step = __ddiv_rn(denom, (double)k);   // linspace: step = delta / div
        kscale = __ddiv_rn((double)k, denom); // per image, so that the per-id estimate below needs no division
    }
    __device__ __forceinline__ double edge(int i) const {  // linspace(first, last, k + 1)[i]
        if (i == k) return last;
        return __dadd_rn(__dmul_rn((double)i, step), first);
    }
    __device__ __forceinline__ int bin(int64_t a) const {
        const double x = (double)a;
        // numpy: f = ((x - first) / denom) * k, truncated, then corrected by at most one bin against the edges below.
        // The corrected result is the unique bin whose edges bracket x whenever the estimate is within one bin of
        // it, so (x - first) * (k / denom) -- a few ulps away from numpy's f -- yields the identical bin without a
        // division on every id's critical path.
        const double f = __dmul_rn(__dsub_rn(x, first), kscale);
        int idx = (int)f;  // astype(np.intp) truncation
        if (idx == k) idx -= 1;
        if (x < edge(idx)) idx -= 1;
        if (x >= edge(idx + 1) && idx != k - 1) idx += 1;
        return idx;
    }
};

// tf*k1 / (tf*k1 + k2*(1 - b + b*(dl/avgdl))) with numpy's float64 operation order (utils.py:199-200)
__device__ __forceinline__ double okapi_weight(double tf, double k1, double k2, double b, double ratio) {
    const double t = __dmul_rn(tf, k1);
    const double den = __dadd_rn(t, __dmul_rn(k2, __dadd_rn(__dsub_rn(1.0, b), __dmul_rn(b, ratio))));
    return __ddiv_rn(t, den);
}

// 4 (float) or 2 x 2 (double) values per 128-bit store
__device__ __forceinline__ void store4(float* p, double a, double b, double c, double d) {
    *reinterpret_cast<float4*>(p) = make_float4((float)a, (float)b, (float)c, (float)d);
}
__device__ __forceinline__ void store4(double* p, double a, double b, double c, double d) {
    reinterpret_cast<double2*>(p)[0] = make_double2(a, b);
    reinterpret_cast<double2*>(p)[1] = make_double2(c, d);
}

// Zero fill sized to run BESIDE the verified assign (one 512-thread CTA per SM, 95 registers, 205.8 KB of shared
// memory): 128 threads, no shared memory and at most 32 registers per thread (the 16 of __launch_bounds__ cap them),
// so its blocks fit in what the assign's CTA leaves of an SM.  ise_clear gives it the max-shared carveout: with the
// default, an SM that holds clear blocks is configured for little shared memory and cannot take the assign's CTA
// until they drain (measured on a B200: the two kernels then ran one after the other).  The assign also slows under
// a concurrent full-rate HBM stream, so ns_per_sweep > 0 paces the stores against %globaltimer: each thread stores
// 16 bytes per sweep and starts sweep s no earlier than s * ns_per_sweep after it began.  Evict-first stores: the
// cleared rows are not read again before the histogram's scattered writes.
constexpr int kClearThreads = 128;

__device__ __forceinline__ uint64_t global_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__global__ void __launch_bounds__(kClearThreads, 16)
clear_kernel(uint4* __restrict__ p, int64_t n16, unsigned char* __restrict__ tail, int tail_bytes,
             unsigned ns_per_sweep) {
    const int64_t stride = (int64_t)gridDim.x * kClearThreads;
    const uint64_t t0 = ns_per_sweep ? global_ns() : 0;
    uint64_t due = t0;
    for (int64_t i = (int64_t)blockIdx.x * kClearThreads + threadIdx.x; i < n16; i += stride) {
        __stcs(p + i, make_uint4(0u, 0u, 0u, 0u));
        if (ns_per_sweep) {
            due += ns_per_sweep;
            while (global_ns() < due) __nanosleep(64);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < tail_bytes) tail[threadIdx.x] = 0;
}

// One CTA walks images (grid-stride).  Per image: the ids are read ONCE into registers (up to WPT per thread;
// longer images re-read the tail from L2), min/max for the numpy-compat edges (32-bit redux), shared-memory atomic
// counts, then the row is written with 128-bit stores while the counters are cleared in the same sweep (no
// separate zeroing phase); the NEXT image's ids are already in flight during the write-out.  ZEROED (the row was
// cleared beforehand): only the image's distinct bins are written, see write_distinct_bins.  The Okapi weight
// depends only on (tf, dl): the weights of tf = 1..kTfTable are computed once per image by 32 threads and the
// write-out looks them up -- with the FP64 divisions inlined in the write-out the first version was
// instruction-bound (6.1 k warp instructions per image, 0.44 of HBM peak; profiles/r01_findings.md section 9).
// Ids must fit in int32 (k < 2^31 is checked by the entry point; other values cannot come out of the assign).
constexpr int kTfTable = 32;

// out-of-line on purpose: inlined, the compiler if-converts `tf <= table ? table[tf] : weight(tf)` and runs the FP64
// division for EVERY non-zero (ncu: 45 % of the kernel's instructions were that speculated DFMA chain)
__device__ __noinline__ double okapi_weight_rare(double tf, double k1, double k2, double b, double ratio) {
    return okapi_weight(tf, k1, k2, b, ratio);
}

// Write-out of one image into a row that was cleared beforehand: at BoVW sizes ~97 % of a row is zeros, so writing
// only the image's distinct bins saves nearly all of the row's bytes.  The nt threads of the group (warp or CTA)
// walk their own ids, not the k counters.  A held id (bins[i], -1 = none) whose atomicAdd saw 0 (bit i of `first`)
// was its bin's first hit: that thread writes the bin, and after `sync` resets its counter, so only touched counters
// are reset.  With `whole` (k a multiple of the bins per 32-byte sector, 32-byte aligned rows) the owner writes the
// whole aligned sector around its bin, every value taken from the final counts: a scattered 8-byte store into a row
// that is not in L2 is a partial sector, which the memory side has to read, merge and write back.  Two owners in one
// sector write the same bytes.  Ids past the WPT * nt held ones were re-read and kept no flags: once the held owners
// are done, an atomicExch picks one writer for each bin still counted.
template <int WPT, typename OutT, typename BinOf, typename Weight, typename Sync>
__device__ __forceinline__ void write_distinct_bins(const int (&bins)[WPT], unsigned first, int* s_cnt, OutT* orow,
                                                    bool whole, const int64_t* __restrict__ words, int64_t lo,
                                                    int64_t hi, int t, int nt, BinOf bin_of, Weight weight, Sync sync) {
    constexpr int G = 32 / (int)sizeof(OutT);   // bins per 32-byte sector
#pragma unroll
    for (int i = 0; i < WPT; ++i)
        if (first & (1u << i)) {
            if (whole) {
                const int g = bins[i] & ~(G - 1);
                auto val = [&](int u) -> double {
                    const int c = s_cnt[g + u];
                    return c ? weight(c) : 0.0;
                };
#pragma unroll
                for (int u = 0; u < G; u += 4) store4(orow + g + u, val(u), val(u + 1), val(u + 2), val(u + 3));
            } else {
                orow[bins[i]] = (OutT)weight(s_cnt[bins[i]]);
            }
        }
    sync();
#pragma unroll
    for (int i = 0; i < WPT; ++i)
        if (first & (1u << i)) s_cnt[bins[i]] = 0;
    if (lo + WPT * nt < hi) {
        sync();
        for (int64_t j = lo + t + WPT * nt; j < hi; j += nt) {
            const int bin = bin_of((int)__ldg(words + j));
            if (bin >= 0) {
                const int c = atomicExch(&s_cnt[bin], 0);
                if (c) orow[bin] = (OutT)weight(c);
            }
        }
    }
}

template <typename OutT, bool SMEM, bool ZEROED>
__global__ void __launch_bounds__(kThreads, 8)
histogram_kernel(const int64_t* __restrict__ words, const int64_t* __restrict__ off, int64_t n_img, int k, int mode,
                 OutT* __restrict__ out, int okapi, double k1, double k2, double b, double avgdl_in) {
    static_assert(SMEM || !ZEROED, "without shared-memory counters the counts are added into the cleared row itself");
    constexpr int WPT = 4;                       // ids held in registers per thread (covers 512 per image)
    extern __shared__ int s_cnt[];
    __shared__ int s_mn, s_mx;
    __shared__ double s_w[kTfTable + 1];
    // np.mean(dl) over the batch being transformed (utils.py:196); a caller that feeds the batch in
    // several launches passes the whole batch's mean explicitly
    const double avgdl = avgdl_in >= 0.0 ? avgdl_in : (double)(off[n_img] - off[0]) / (double)n_img;
    if (SMEM) {
        for (int j = threadIdx.x; j < k; j += kThreads) s_cnt[j] = 0;
    }
    if (threadIdx.x == 0) { s_mn = INT_MAX; s_mx = INT_MIN; }
    int w[WPT];
    int64_t lo = 0, hi = 0;
    auto fetch = [&](int64_t img) {
        lo = off[img]; hi = off[img + 1];
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int64_t j = lo + threadIdx.x + i * kThreads;
            w[i] = j < hi ? (int)__ldg(words + j) : 0;
        }
    };
    if (blockIdx.x < n_img) fetch(blockIdx.x);
    __syncthreads();
    const bool vec_ok = (k % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const bool whole = ZEROED && k % (32 / (int)sizeof(OutT)) == 0 && (reinterpret_cast<uintptr_t>(out) & 31) == 0;
    for (int64_t img = blockIdx.x; img < n_img; img += gridDim.x) {
        const int64_t cnt = hi - lo;
        OutT* orow = out + img * (int64_t)k;
        const double ratio = __ddiv_rn((double)cnt, avgdl);  // rep / avgdl
        if (okapi && threadIdx.x >= kThreads - kTfTable)     // the last warp: usually holds no ids
            s_w[threadIdx.x - (kThreads - kTfTable) + 1] =
                okapi_weight((double)(threadIdx.x - (kThreads - kTfTable) + 1), k1, k2, b, ratio);
        NumpyBins nb;
        if (mode == ISE_HIST_NUMPY_COMPAT && cnt > 0) {
            int mn = INT_MAX, mx = INT_MIN;
#pragma unroll
            for (int i = 0; i < WPT; ++i)
                if (lo + threadIdx.x + i * kThreads < hi) { mn = min(mn, w[i]); mx = max(mx, w[i]); }
            for (int64_t j = lo + threadIdx.x + WPT * kThreads; j < hi; j += kThreads) {
                const int v = (int)words[j];
                mn = min(mn, v); mx = max(mx, v);
            }
            mn = __reduce_min_sync(0xffffffffu, mn);
            mx = __reduce_max_sync(0xffffffffu, mx);
            if ((threadIdx.x & 31) == 0 && mn <= mx) { atomicMin(&s_mn, mn); atomicMax(&s_mx, mx); }
            __syncthreads();
            nb.setup(s_mn, s_mx, k);
        }
        auto bin_of = [&](int v) -> int {
            int bin;
            if (mode == ISE_HIST_NUMPY_COMPAT) bin = nb.bin(v);
            else bin = (v >= 0 && v < k) ? v : -1;
            return bin >= 0 && bin < k ? bin : -1;
        };
        auto count = [&](int bin) {
            if (SMEM) atomicAdd(&s_cnt[bin], 1);
            else atomicAdd(orow + bin, (OutT)1);  // row was zeroed beforehand (memset or the caller's clear)
        };
        int bins[WPT];
        unsigned first = 0;    // ZEROED: bit i = bins[i] saw its first hit here
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            bins[i] = lo + threadIdx.x + i * kThreads < hi ? bin_of(w[i]) : -1;
            if (bins[i] >= 0) {
                if (ZEROED) first |= atomicAdd(&s_cnt[bins[i]], 1) == 0 ? 1u << i : 0u;
                else count(bins[i]);
            }
        }
        for (int64_t j = lo + threadIdx.x + WPT * kThreads; j < hi; j += kThreads) {
            const int bin = bin_of((int)words[j]);
            if (bin >= 0) count(bin);
        }
        const int64_t img_lo = lo, img_hi = hi;   // fetch() moves lo / hi on to the next image
        // ids of the next image: in flight while this row is written
        if (img + gridDim.x < n_img) fetch(img + gridDim.x);
        __syncthreads();
        if (threadIdx.x == 0) { s_mn = INT_MAX; s_mx = INT_MIN; }   // read by everyone before the barrier above
        auto weight = [&](int c) -> double {
            if (!okapi) return (double)c;
            if (c <= kTfTable) return s_w[c];
            return okapi_weight_rare((double)c, k1, k2, b, ratio);
        };
        if (ZEROED) {
            write_distinct_bins<WPT>(bins, first, s_cnt, orow, whole, words, img_lo, img_hi, threadIdx.x, kThreads,
                                     bin_of, weight, [] { __syncthreads(); });
        } else if (SMEM) {
            if (vec_ok) {
                for (int j = threadIdx.x * 4; j < k; j += kThreads * 4) {
                    const int4 c = *reinterpret_cast<const int4*>(s_cnt + j);
                    double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
                    if ((c.x | c.y | c.z | c.w) != 0) {
                        *reinterpret_cast<int4*>(s_cnt + j) = make_int4(0, 0, 0, 0);
                        if (c.x) v0 = weight(c.x);
                        if (c.y) v1 = weight(c.y);
                        if (c.z) v2 = weight(c.z);
                        if (c.w) v3 = weight(c.w);
                    }
                    store4(orow + j, v0, v1, v2, v3);
                }
            } else {
                for (int j = threadIdx.x; j < k; j += kThreads) {
                    const int c = s_cnt[j];
                    double v = 0.0;
                    if (c != 0) {
                        s_cnt[j] = 0;
                        v = weight(c);
                    }
                    orow[j] = (OutT)v;
                }
            }
        } else if (okapi) {
            for (int j = threadIdx.x; j < k; j += kThreads) {
                const double c = (double)orow[j];
                if (c != 0.0) orow[j] = (OutT)okapi_weight(c, k1, k2, b, ratio);
            }
        }
        __syncthreads();
    }
}

// Warp-per-image variant for SHORT images (the BoVW regime: ~100 descriptors per image, thousands of bins).  The
// CTA-per-image kernel above spends an image on three CTA-wide barriers and is bound by that critical path (0.64 of
// HBM peak at C2); here a warp owns an image end to end -- its own k counters in shared memory, ids in registers,
// `__syncwarp` only -- and twelve warps per SM keep the 32 KB row stores of twelve images in flight.
constexpr int kWarpHistWarps = 4;          // warps per CTA; k * 4 B of counters each
constexpr int kWarpHistMaxBins = 4096;

template <typename OutT, bool ZEROED>
__global__ void __launch_bounds__(kWarpHistWarps * 32)
histogram_warp_kernel(const int64_t* __restrict__ words, const int64_t* __restrict__ off, int64_t n_img, int k, int mode,
                      OutT* __restrict__ out, int okapi, double k1, double k2, double b, double avgdl_in) {
    constexpr int WPT = 4;                 // ids held in registers per lane (128 per image; longer ones re-read)
    extern __shared__ int s_all[];
    __shared__ double s_wt[kWarpHistWarps][kTfTable + 1];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    int* s_cnt = s_all + wib * k;
    double* s_w = s_wt[wib];
    const double avgdl = avgdl_in >= 0.0 ? avgdl_in : (double)(off[n_img] - off[0]) / (double)n_img;
    for (int j = lane; j < k; j += 32) s_cnt[j] = 0;
    __syncwarp();
    const bool vec_ok = (k % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const bool whole = ZEROED && k % (32 / (int)sizeof(OutT)) == 0 && (reinterpret_cast<uintptr_t>(out) & 31) == 0;
    const int64_t warp = (int64_t)blockIdx.x * kWarpHistWarps + wib, nwarps = (int64_t)gridDim.x * kWarpHistWarps;
    for (int64_t img = warp; img < n_img; img += nwarps) {
        const int64_t lo = __ldg(off + img), hi = __ldg(off + img + 1);
        const int64_t cnt = hi - lo;
        OutT* orow = out + img * (int64_t)k;
        int w[WPT];
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int64_t j = lo + lane + i * 32;
            w[i] = 0;
            if (j < hi) w[i] = (int)__ldg(words + j);
        }
        const double ratio = __ddiv_rn((double)cnt, avgdl);
        if (okapi) s_w[lane + 1] = okapi_weight((double)(lane + 1), k1, k2, b, ratio);     // kTfTable == 32
        NumpyBins nb;
        if (mode == ISE_HIST_NUMPY_COMPAT && cnt > 0) {
            int mn = INT_MAX, mx = INT_MIN;
#pragma unroll
            for (int i = 0; i < WPT; ++i)
                if (lo + lane + i * 32 < hi) { mn = min(mn, w[i]); mx = max(mx, w[i]); }
            for (int64_t j = lo + lane + WPT * 32; j < hi; j += 32) {
                const int v = (int)__ldg(words + j);
                mn = min(mn, v); mx = max(mx, v);
            }
            mn = __reduce_min_sync(0xffffffffu, mn);
            mx = __reduce_max_sync(0xffffffffu, mx);
            nb.setup(mn, mx, k);
        }
        auto bin_of = [&](int v) -> int {
            int bin;
            if (mode == ISE_HIST_NUMPY_COMPAT) bin = nb.bin(v);
            else bin = (v >= 0 && v < k) ? v : -1;
            return bin >= 0 && bin < k ? bin : -1;
        };
        int bins[WPT];
        unsigned first = 0;    // ZEROED: bit i = bins[i] saw its first hit here
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            bins[i] = lo + lane + i * 32 < hi ? bin_of(w[i]) : -1;
            if (bins[i] >= 0) {
                if (ZEROED) first |= atomicAdd(&s_cnt[bins[i]], 1) == 0 ? 1u << i : 0u;
                else atomicAdd(&s_cnt[bins[i]], 1);
            }
        }
        for (int64_t j = lo + lane + WPT * 32; j < hi; j += 32) {
            const int bin = bin_of((int)__ldg(words + j));
            if (bin >= 0) atomicAdd(&s_cnt[bin], 1);
        }
        __syncwarp();
        auto weight = [&](int c) -> double {
            if (!okapi) return (double)c;
            if (c <= kTfTable) return s_w[c];
            return okapi_weight_rare((double)c, k1, k2, b, ratio);
        };
        if (ZEROED) {
            write_distinct_bins<WPT>(bins, first, s_cnt, orow, whole, words, lo, hi, lane, 32, bin_of, weight,
                                     [] { __syncwarp(); });
        } else if (vec_ok) {
            for (int j = lane * 4; j < k; j += 128) {
                const int4 c = *reinterpret_cast<const int4*>(s_cnt + j);
                double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
                if ((c.x | c.y | c.z | c.w) != 0) {
                    *reinterpret_cast<int4*>(s_cnt + j) = make_int4(0, 0, 0, 0);
                    if (c.x) v0 = weight(c.x);
                    if (c.y) v1 = weight(c.y);
                    if (c.z) v2 = weight(c.z);
                    if (c.w) v3 = weight(c.w);
                }
                store4(orow + j, v0, v1, v2, v3);
            }
        } else {
            for (int j = lane; j < k; j += 32) {
                const int c = s_cnt[j];
                double v = 0.0;
                if (c != 0) { s_cnt[j] = 0; v = weight(c); }
                orow[j] = (OutT)v;
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// CSR output: the histogram matrix is ~97 % zeros at BoVW sizes (100-1000 words per image against thousands of
// bins), and OkapiTransformer.transform returns a scipy CSR matrix anyway (utils.py:153-202), so the
// pipeline-level call never has to materialise (or ship over PCIe) the dense [n_img, k] float64 matrix.
//   pass 0  distinct bins per image (atomicAdd's old value == 0 marks a bin's first hit)  -> row_nnz[n_img]
//   scan    exclusive prefix sum                                                          -> indptr[n_img + 1]
//   pass 1  recount, then an ordered compaction of the k counters (thread t owns a contiguous run of bins,
//           block-wide exclusive scan of the per-thread non-zero counts)                  -> indices, data
// Column indices come out sorted, like scipy's dense -> CSR conversion.
// ------------------------------------------------------------------------------------------
template <typename OutT, int PASS>
__global__ void __launch_bounds__(kThreads, 8)
histogram_csr_kernel(const int64_t* __restrict__ words, const int64_t* __restrict__ off, int64_t n_img, int k, int mode,
                     int32_t* __restrict__ row_nnz, const int32_t* __restrict__ indptr, int32_t* __restrict__ indices,
                     OutT* __restrict__ data, int okapi, double k1, double k2, double b, double avgdl_in) {
    extern __shared__ int s_cnt[];
    __shared__ int s_mn, s_mx, s_total;
    __shared__ int s_warp[kThreads / 32];
    __shared__ double s_w[kTfTable + 1];
    const double avgdl = avgdl_in >= 0.0 ? avgdl_in : (double)(off[n_img] - off[0]) / (double)n_img;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    for (int j = threadIdx.x; j < k; j += kThreads) s_cnt[j] = 0;
    if (threadIdx.x == 0) { s_mn = INT_MAX; s_mx = INT_MIN; s_total = 0; }
    __syncthreads();
    for (int64_t img = blockIdx.x; img < n_img; img += gridDim.x) {
        const int64_t lo = off[img], hi = off[img + 1];
        const int64_t cnt = hi - lo;
        NumpyBins nb;
        if (mode == ISE_HIST_NUMPY_COMPAT && cnt > 0) {
            int mn = INT_MAX, mx = INT_MIN;
            for (int64_t j = lo + threadIdx.x; j < hi; j += kThreads) {
                const int v = (int)__ldg(words + j);
                mn = min(mn, v); mx = max(mx, v);
            }
            mn = __reduce_min_sync(0xffffffffu, mn);
            mx = __reduce_max_sync(0xffffffffu, mx);
            if (lane == 0 && mn <= mx) { atomicMin(&s_mn, mn); atomicMax(&s_mx, mx); }
            __syncthreads();
            nb.setup(s_mn, s_mx, k);
        }
        int fresh = 0;
        for (int64_t j = lo + threadIdx.x; j < hi; j += kThreads) {
            const int v = (int)__ldg(words + j);
            int bin;
            if (mode == ISE_HIST_NUMPY_COMPAT) bin = nb.bin(v);
            else bin = (v >= 0 && v < k) ? v : -1;
            if (bin >= 0 && bin < k) fresh += atomicAdd(&s_cnt[bin], 1) == 0 ? 1 : 0;
        }
        if (PASS == 0) {
            fresh = __reduce_add_sync(0xffffffffu, fresh);
            if (lane == 0 && fresh) atomicAdd(&s_total, fresh);
            __syncthreads();
            if (threadIdx.x == 0) { row_nnz[img] = s_total; s_total = 0; s_mn = INT_MAX; s_mx = INT_MIN; }
            // clear only the bins this image touched
            for (int64_t j = lo + threadIdx.x; j < hi; j += kThreads) {
                const int v = (int)__ldg(words + j);
                int bin;
                if (mode == ISE_HIST_NUMPY_COMPAT) bin = nb.bin(v);
                else bin = (v >= 0 && v < k) ? v : -1;
                if (bin >= 0 && bin < k) s_cnt[bin] = 0;
            }
            __syncthreads();
        } else {
            const double ratio = __ddiv_rn((double)cnt, avgdl);
            if (okapi && threadIdx.x >= kThreads - kTfTable)
                s_w[threadIdx.x - (kThreads - kTfTable) + 1] =
                    okapi_weight((double)(threadIdx.x - (kThreads - kTfTable) + 1), k1, k2, b, ratio);
            __syncthreads();
            if (threadIdx.x == 0) { s_mn = INT_MAX; s_mx = INT_MIN; }
            // ordered compaction, bank-conflict free: warp w owns the contiguous bins [w * per_warp, ...), walks them 32
            // at a time (lane = bin) and ranks the non-zeros with ballot + popc; a first sweep counts per warp so
            // that every warp knows where its run starts in the row
            constexpr int NW = kThreads / 32;
            const int per_warp = ((k + NW - 1) / NW + 31) / 32 * 32;
            const int c_lo = wib * per_warp, c_hi = min(k, c_lo + per_warp);
            int mine = 0;
            for (int c0 = c_lo; c0 < c_hi; c0 += 32) {
                const int c = c0 + lane;
                mine += __popc(__ballot_sync(0xffffffffu, c < c_hi && s_cnt[c] != 0));
            }
            if (lane == 0) s_warp[wib] = mine;
            __syncthreads();
            int pos = indptr[img];
#pragma unroll
            for (int i = 0; i < NW; ++i) pos += i < wib ? s_warp[i] : 0;
            for (int c0 = c_lo; c0 < c_hi; c0 += 32) {
                const int c = c0 + lane;
                const int v = c < c_hi ? s_cnt[c] : 0;
                const unsigned mask = __ballot_sync(0xffffffffu, v != 0);
                if (v != 0) {
                    s_cnt[c] = 0;
                    const int p = pos + __popc(mask & ((1u << lane) - 1u));
                    indices[p] = c;
                    double w = (double)v;
                    if (okapi) w = v <= kTfTable ? s_w[v] : okapi_weight_rare((double)v, k1, k2, b, ratio);
                    data[p] = (OutT)w;
                }
                pos += __popc(mask);
            }
            __syncthreads();
        }
    }
}

// exclusive prefix sum of n int32 values -> out[n + 1] (single CTA; n is the number of images)
__global__ void exclusive_scan_i32_kernel(const int32_t* __restrict__ in, int64_t n, int32_t* __restrict__ out) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < n; base += blockDim.x) {
        const int64_t i = base + threadIdx.x;
        const int v = i < n ? in[i] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[wib] = incl;
        __syncthreads();
        int wbase = 0;
        for (int w = 0; w < wib; ++w) wbase += s_warp[w];
        const int carry = s_carry;
        if (i < n) out[i] = carry + wbase + incl - v;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = carry + wbase + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) out[n] = s_carry;
}

// dense in-place Okapi: pass 1 row sums (document lengths), pass 2 weights
template <typename T>
__global__ void row_sum_kernel(const T* __restrict__ h, int64_t n_img, int k, double* __restrict__ dl,
                               double* __restrict__ total) {
    __shared__ double s_part[kThreads / 32];
    for (int64_t img = blockIdx.x; img < n_img; img += gridDim.x) {
        const T* row = h + img * (int64_t)k;
        double acc = 0.0;
        // summed in the same per-thread column order whatever the unrolling: four loads in flight
        int j = threadIdx.x;
        for (; j + 3 * kThreads < k; j += 4 * kThreads) {
            const T a0 = row[j], a1 = row[j + kThreads], a2 = row[j + 2 * kThreads], a3 = row[j + 3 * kThreads];
            acc += (double)a0; acc += (double)a1; acc += (double)a2; acc += (double)a3;
        }
        for (; j < k; j += kThreads) acc += (double)row[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int i = 0; i < kThreads / 32; ++i) t += s_part[i];
            dl[img] = t;
            atomicAdd(total, t);
        }
        __syncthreads();
    }
}

template <typename T>
__global__ void okapi_dense_kernel(T* __restrict__ h, int64_t n_img, int k, double k1, double k2, double b,
                                   double avgdl_in, const double* __restrict__ dl, const double* __restrict__ total) {
    const double avgdl = avgdl_in >= 0.0 ? avgdl_in : __ddiv_rn(*total, (double)n_img);
    for (int64_t img = blockIdx.x; img < n_img; img += gridDim.x) {
        T* row = h + img * (int64_t)k;
        const double ratio = __ddiv_rn(dl[img], avgdl);
        int j = threadIdx.x;
        for (; j + 3 * kThreads < k; j += 4 * kThreads) {
            T a[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) a[u] = row[j + u * kThreads];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if ((double)a[u] != 0.0) row[j + u * kThreads] = (T)okapi_weight((double)a[u], k1, k2, b, ratio);
        }
        for (; j < k; j += kThreads) {
            const double c = (double)row[j];
            if (c != 0.0) row[j] = (T)okapi_weight(c, k1, k2, b, ratio);
        }
    }
}

// ---- OkapiTransformer.transform on a CSR matrix (utils.py:153-202 operates on X.data exactly like this) ----
// one warp per row: document length = sum of the row's stored values
__global__ void csr_row_sum_kernel(const int64_t* __restrict__ indptr, const double* __restrict__ data, int64_t n_rows,
                                   double* __restrict__ dl, double* __restrict__ total) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (kThreads / 32);
    double mine = 0.0;
    for (int64_t r = warp; r < n_rows; r += nwarps) {
        const int64_t lo = indptr[r], hi = indptr[r + 1];
        double acc = 0.0;
        for (int64_t j = lo + lane; j < hi; j += 32) acc += data[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) { dl[r] = acc; mine += acc; }
    }
    if (lane == 0 && mine != 0.0) atomicAdd(total, mine);
}

// weights in place; idf != nullptr / norm != 0 = the opt-in corrected tf-idf mode (the reference computes idf in fit
// and declares norm="l2" but applies neither, utils.py:112-151)
__global__ void csr_okapi_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                 double* __restrict__ data, int64_t n_rows, double k1, double k2, double b,
                                 double avgdl_in, const double* __restrict__ dl, const double* __restrict__ total,
                                 const double* __restrict__ idf, int norm) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (kThreads / 32);
    const double avgdl = avgdl_in >= 0.0 ? avgdl_in : __ddiv_rn(*total, (double)n_rows);
    for (int64_t r = warp; r < n_rows; r += nwarps) {
        const int64_t lo = indptr[r], hi = indptr[r + 1];
        const double ratio = __ddiv_rn(dl[r], avgdl);
        double nrm = 0.0;
        for (int64_t j = lo + lane; j < hi; j += 32) {
            double w = okapi_weight(data[j], k1, k2, b, ratio);     // 0 stays 0 (0 / positive)
            if (idf) w *= idf[indices[j]];
            data[j] = w;
            nrm += norm == 2 ? w * w : fabs(w);
        }
        if (norm) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
            if (norm == 2) nrm = sqrt(nrm);
            if (nrm > 0.0) {
                __syncwarp();
                for (int64_t j = lo + lane; j < hi; j += 32) data[j] = data[j] / nrm;
            }
        }
    }
}

// dense counterpart of the opt-in mode (GPU-resident index build): h[i, j] *= idf[j], then row normalisation
template <typename T>
__global__ void tfidf_finish_kernel(T* __restrict__ h, int64_t n_img, int k, const double* __restrict__ idf, int norm) {
    __shared__ double s_part[kThreads / 32];
    __shared__ double s_nrm;
    for (int64_t img = blockIdx.x; img < n_img; img += gridDim.x) {
        T* row = h + img * (int64_t)k;
        double nrm = 0.0;
        for (int j = threadIdx.x; j < k; j += kThreads) {
            double w = (double)row[j];
            if (w != 0.0) {
                if (idf) { w *= idf[j]; row[j] = (T)w; }
                nrm += norm == 2 ? w * w : fabs(w);
            }
        }
        if (norm) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
            if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = nrm;
            __syncthreads();
            if (threadIdx.x == 0) {
                double t = 0.0;
                for (int i = 0; i < kThreads / 32; ++i) t += s_part[i];
                s_nrm = norm == 2 ? sqrt(t) : t;
            }
            __syncthreads();
            const double t = s_nrm;
            if (t > 0.0)
                for (int j = threadIdx.x; j < k; j += kThreads) {
                    const double w = (double)row[j];
                    if (w != 0.0) row[j] = (T)(w / t);
                }
            __syncthreads();
        }
    }
}

}  // namespace

ISE_EXPORT int ise_clear(ise_ctx* ctx, void* p, size_t bytes, double gb_per_s, void* stream) {
    ISE_CHECK_ARG(ctx && gb_per_s >= 0.0);
    if (bytes == 0) return 0;
    ISE_CHECK_ARG(p && (reinterpret_cast<uintptr_t>(p) & 15) == 0);
    DeviceGuard guard(ctx->device);
    // one sweep = every thread of the grid stores 16 bytes; 1 GB/s = 1 byte per ns
    const double sweep_bytes = (double)ctx->sm_count * kClearThreads * 16;
    const unsigned ns_per_sweep = gb_per_s > 0.0 ? (unsigned)std::min(1e9, std::max(1.0, sweep_bytes / gb_per_s)) : 0u;
    ISE_CUDA(cudaFuncSetAttribute(clear_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
    clear_kernel<<<ctx->sm_count, kClearThreads, 0, (cudaStream_t)stream>>>(
        (uint4*)p, (int64_t)(bytes / 16), (unsigned char*)p + bytes / 16 * 16, (int)(bytes % 16), ns_per_sweep);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_bovw_histogram(ise_ctx* ctx, const int64_t* words, int64_t n_words, const int64_t* img_offsets,
                                  int64_t n_img, int k, int mode, int out_dtype, void* out, int okapi, double k1,
                                  double k2, double b, double avgdl, int zeroed, void* stream) {
    ISE_CHECK_ARG(ctx && n_img >= 0 && k >= 1);   // ids are handled as int32 (k is an int)
    ISE_CHECK_ARG(mode == ISE_HIST_NUMPY_COMPAT || mode == ISE_HIST_BINCOUNT);
    ISE_CHECK_ARG(out_dtype == ISE_OUT_F32 || out_dtype == ISE_OUT_F64);
    if (n_img == 0) return 0;
    ISE_CHECK_ARG(img_offsets && out);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const bool smem = k <= kMaxSmemBins;
    // short images, moderate codebooks: the warp-per-image kernel (n_words / n_img = mean image length)
    // (float64 rows only: measured at C2 size 76 vs 82 us numpy-compat + Okapi, 65 vs 80 us bincount; with float32 rows --
    // half the bytes per image -- the CTA kernel's 52 us beats the warp kernel's 77 us, which is bound by the per-warp
    // chain of id loads, FP64 bin edges and 32 counter sweeps rather than by the stores)
    if (smem && out_dtype == ISE_OUT_F64 && k <= kWarpHistMaxBins && n_img >= 4 * (int64_t)ctx->sm_count && n_words > 0 &&
        n_words <= 256 * n_img && !getenv("ISE_HIST_CTA")) {
        static_assert(kTfTable == 32, "one Okapi table entry per lane");
        const size_t shm_w = (size_t)kWarpHistWarps * k * sizeof(int);
        const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(16, (200 * 1024) / (shm_w + 2048)));
        const int grid_w = (int)std::min<int64_t>(ceil_div64(n_img, kWarpHistWarps), (int64_t)ctx->sm_count * per_sm);
        auto kern = zeroed ? histogram_warp_kernel<double, true> : histogram_warp_kernel<double, false>;
        ISE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm_w));
        kern<<<grid_w, kWarpHistWarps * 32, shm_w, st>>>(words, img_offsets, n_img, k, mode, (double*)out, okapi, k1,
                                                        k2, b, avgdl);
        ISE_LAUNCH_CHECK();
        return 0;
    }
    const int grid = (int)std::min<int64_t>(n_img, (int64_t)ctx->sm_count * 16);
    const size_t elt = out_dtype == ISE_OUT_F64 ? 8 : 4;
    if (!smem && !zeroed) ISE_CUDA(cudaMemsetAsync(out, 0, (size_t)n_img * k * elt, st));
    const size_t shm = smem ? (size_t)k * sizeof(int) : 0;
    if (out_dtype == ISE_OUT_F64) {
        auto kern = !smem ? histogram_kernel<double, false, false>
                          : zeroed ? histogram_kernel<double, true, true> : histogram_kernel<double, true, false>;
        kern<<<grid, kThreads, shm, st>>>(words, img_offsets, n_img, k, mode, (double*)out, okapi, k1, k2, b, avgdl);
    } else {
        auto kern = !smem ? histogram_kernel<float, false, false>
                          : zeroed ? histogram_kernel<float, true, true> : histogram_kernel<float, true, false>;
        kern<<<grid, kThreads, shm, st>>>(words, img_offsets, n_img, k, mode, (float*)out, okapi, k1, k2, b, avgdl);
    }
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_okapi_tf(ise_ctx* ctx, void* h, int out_dtype, int64_t n_img, int k, double k1, double k2,
                            double b, double avgdl, double* dl_workspace, void* stream) {
    ISE_CHECK_ARG(ctx && n_img >= 0 && k >= 1);
    ISE_CHECK_ARG(out_dtype == ISE_OUT_F32 || out_dtype == ISE_OUT_F64);
    if (n_img == 0) return 0;
    ISE_CHECK_ARG(h && dl_workspace);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    double* dl = dl_workspace;
    double* total = dl_workspace + n_img;
    ISE_CUDA(cudaMemsetAsync(total, 0, sizeof(double), st));
    const int grid = (int)std::min<int64_t>(n_img, (int64_t)ctx->sm_count * 16);
    if (out_dtype == ISE_OUT_F64) {
        row_sum_kernel<double><<<grid, kThreads, 0, st>>>((const double*)h, n_img, k, dl, total);
        ISE_LAUNCH_CHECK();
        okapi_dense_kernel<double><<<grid, kThreads, 0, st>>>((double*)h, n_img, k, k1, k2, b, avgdl, dl, total);
    } else {
        row_sum_kernel<float><<<grid, kThreads, 0, st>>>((const float*)h, n_img, k, dl, total);
        ISE_LAUNCH_CHECK();
        okapi_dense_kernel<float><<<grid, kThreads, 0, st>>>((float*)h, n_img, k, k1, k2, b, avgdl, dl, total);
    }
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_bovw_histogram_csr(ise_ctx* ctx, const int64_t* words, const int64_t* img_offsets, int64_t n_img,
                                      int k, int mode, int out_dtype, int32_t* row_nnz, int32_t* indptr,
                                      int32_t* indices, void* data, int okapi, double k1, double k2, double b,
                                      double avgdl, void* stream) {
    ISE_CHECK_ARG(ctx && n_img >= 0 && k >= 1 && k <= kMaxSmemBins);
    ISE_CHECK_ARG(mode == ISE_HIST_NUMPY_COMPAT || mode == ISE_HIST_BINCOUNT);
    ISE_CHECK_ARG(out_dtype == ISE_OUT_F32 || out_dtype == ISE_OUT_F64);
    ISE_CHECK_ARG(indptr != nullptr);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_img == 0) {
        ISE_CUDA(cudaMemsetAsync(indptr, 0, sizeof(int32_t), st));
        return 0;
    }
    ISE_CHECK_ARG(words && img_offsets && row_nnz && indices && data);
    const int grid = (int)std::min<int64_t>(n_img, (int64_t)ctx->sm_count * 16);
    const size_t shm = (size_t)k * sizeof(int);
    histogram_csr_kernel<double, 0><<<grid, kThreads, shm, st>>>(words, img_offsets, n_img, k, mode, row_nnz, nullptr,
                                                                 nullptr, nullptr, 0, k1, k2, b, avgdl);
    ISE_LAUNCH_CHECK();
    exclusive_scan_i32_kernel<<<1, 1024, 0, st>>>(row_nnz, n_img, indptr);
    ISE_LAUNCH_CHECK();
    if (out_dtype == ISE_OUT_F64)
        histogram_csr_kernel<double, 1><<<grid, kThreads, shm, st>>>(words, img_offsets, n_img, k, mode, row_nnz, indptr,
                                                                     indices, (double*)data, okapi, k1, k2, b, avgdl);
    else
        histogram_csr_kernel<float, 1><<<grid, kThreads, shm, st>>>(words, img_offsets, n_img, k, mode, row_nnz, indptr,
                                                                    indices, (float*)data, okapi, k1, k2, b, avgdl);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_okapi_csr(ise_ctx* ctx, const int64_t* indptr, const int32_t* indices, double* data, int64_t n_rows,
                             double k1, double k2, double b, double avgdl, const double* idf, int norm,
                             double* dl_workspace, void* stream) {
    ISE_CHECK_ARG(ctx && n_rows >= 0 && norm >= 0 && norm <= 2);
    if (n_rows == 0) return 0;
    ISE_CHECK_ARG(indptr && data && dl_workspace && (indices || !idf));
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    double* dl = dl_workspace;
    double* total = dl_workspace + n_rows;
    ISE_CUDA(cudaMemsetAsync(total, 0, sizeof(double), st));
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(n_rows, kThreads / 32), (int64_t)ctx->sm_count * 16));
    csr_row_sum_kernel<<<grid, kThreads, 0, st>>>(indptr, data, n_rows, dl, total);
    ISE_LAUNCH_CHECK();
    csr_okapi_kernel<<<grid, kThreads, 0, st>>>(indptr, indices, data, n_rows, k1, k2, b, avgdl, dl, total, idf, norm);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_tfidf_finish(ise_ctx* ctx, void* h, int out_dtype, int64_t n_img, int k, const double* idf, int norm,
                                void* stream) {
    ISE_CHECK_ARG(ctx && n_img >= 0 && k >= 1 && norm >= 0 && norm <= 2);
    ISE_CHECK_ARG(out_dtype == ISE_OUT_F32 || out_dtype == ISE_OUT_F64);
    if (n_img == 0 || (!idf && !norm)) return 0;
    ISE_CHECK_ARG(h != nullptr);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (int)std::min<int64_t>(n_img, (int64_t)ctx->sm_count * 16);
    if (out_dtype == ISE_OUT_F64) tfidf_finish_kernel<double><<<grid, kThreads, 0, st>>>((double*)h, n_img, k, idf, norm);
    else tfidf_finish_kernel<float><<<grid, kThreads, 0, st>>>((float*)h, n_img, k, idf, norm);
    ISE_LAUNCH_CHECK();
    return 0;
}
