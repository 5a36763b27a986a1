// Shared host/device helpers for libise (sm_100a only).
#pragma once

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "../../include/ise.h"

#define ISE_EXPORT extern "C" __attribute__((visibility("default")))

struct ise_ctx {
    int device;
    int sm_count;
    int cc_major, cc_minor;
    size_t smem_optin;
    // cuTensorMapEncodeTiled resolved through the runtime (no link-time libcuda dependency)
    void* encode_tiled;
    // device scratch for the soft lock-step counters of gemm_select (kSyncInts int32, zeroed per launch)
    int32_t* sync_buf;
};
constexpr int kSyncInts = 64 * 1024;

void ise_set_error(const std::string& msg);

#define ISE_FAIL(msg)                                                                  \
    do {                                                                               \
        ise_set_error(std::string(__func__) + ": " + (msg));                           \
        return 1;                                                                      \
    } while (0)

#define ISE_CHECK_ARG(cond)                                                            \
    do {                                                                               \
        if (!(cond)) ISE_FAIL(std::string("invalid argument: ") + #cond);              \
    } while (0)

#define ISE_CUDA(expr)                                                                 \
    do {                                                                               \
        cudaError_t _e = (expr);                                                       \
        if (_e != cudaSuccess)                                                         \
            ISE_FAIL(std::string(#expr) + " -> " + cudaGetErrorString(_e));            \
    } while (0)

#define ISE_LAUNCH_CHECK()                                                             \
    do {                                                                               \
        cudaError_t _e = cudaGetLastError();                                           \
        if (_e != cudaSuccess)                                                         \
            ISE_FAIL(std::string("kernel launch -> ") + cudaGetErrorString(_e));       \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        ok = cudaGetDevice(&prev) == cudaSuccess;
        if (ok && prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// meta layout shared by prepare.cu and gemm_select.cu
enum {
    META_SCALE = 0, META_INV_SCALE = 1, META_LO_NONZERO = 2, META_ABSMAX = 3, META_MAX_NORM_SQ = 4,
    META_WIDE_MANTISSA = 5,   // != 0: some element has more than 11 significant bits (float32 inputs, absmax pass)
    META_MIN_NONZERO = 6,     // 0x7f800000 - bits(min |x| over non-zero elements), 0 = none seen (int, via atomicMax)
    META_NONFINITE = 7,       // != 0: the conversion pass met a NaN or an Inf (Faiss refuses such training sets)
    META_FLOATS = 8
};

#ifdef __CUDACC__

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// The exact FP32 score of one candidate row `brow` (global memory) against the row `s_a` staged as float32 in shared
// memory, for the warp calling it: per-lane sequential FMAs over dimensions lane, lane + 32, ... (float4 steps when
// d and ldb allow), then the warp tree.  IP returns <a,b>; L2 returns Faiss's IndexFlat expansion
// an + *bn - 2<a,b> clamped at 0 (an, *bn: the squared norms; bn is read only for L2).  Every lane returns the same
// value.  The re-score of search results and the radius test of range search both score through it, so their
// distances agree bit for bit.
template <bool L2>
__device__ __forceinline__ float exact_score(const float* s_a, const float* __restrict__ brow, int d, int64_t ldb,
                                             float an, const float* __restrict__ bn, int lane) {
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
    if (!L2) return acc;
    const float dis = an + *bn - 2.f * acc;
    return dis < 0.f ? 0.f : dis;
}

// Canonical ordering shared by every selection kernel: `better(a, b)` is true when candidate a
// must precede b.  LARGEST: bigger score first; ties by smaller id; id < 0 (padding) loses ties.
template <bool LARGEST>
__device__ __forceinline__ bool cand_better(float va, int64_t ia, float vb, int64_t ib) {
    if (va != vb) return LARGEST ? (va > vb) : (va < vb);
    if (ia < 0) return false;
    if (ib < 0) return true;
    return ia < ib;
}

// Rigorous bound on |coarse - exact| for an inner product computed from the FP16 hi planes only.
// With a = hi_a + lo_a, |lo_a| <= 2^-11 |a| (round-to-nearest FP16; 0 when the plane is exact) the
// neglected terms are <= (c_a + c_b + c_a c_b) |a||b| (Cauchy-Schwarz) -- c_a, c_b are the MEASURED relative residuals
// max_rows |x - hi| / |x| when the preparation pass published them (typically 2-3x below 2^-11);
// the truncating FP32 accumulation adds <= (d/16 + 4) 2^-23 |a||b|; FP16 underflow (scaled elements below
// 2^-14 round with absolute error <= 2^-25) adds <= 2^-25/scale * sqrt(d) * |other operand|.
struct CoarseBound {
    float kappa, uf_a, uf_b, nb_max, sq_, ca_;
    // a_exact: the caller knows the A planes are exact in hi (or re-runs the whole tensor when they are not)
    // meta[LO_NONZERO]: 0 = exact in the hi plane; 1.0 = inexact, residual unknown (worst case 2^-11 |x|); any other
    // value = the largest measured |x - hi|^2 / |x|^2 of a row (rows_convert.cuh: publish_lo_residual)
    __device__ __forceinline__ static float rel_residual(float flag) {
        if (flag == 0.f) return 0.f;
        return flag == 1.f ? 4.8828125e-4f : fminf(1.0001f * sqrtf(flag), 4.8828125e-4f);
    }
    __device__ __forceinline__ void init(const float* a_meta, const float* b_meta, int d, bool a_exact = false) {
        const float ca = a_exact ? 0.f : rel_residual(a_meta[META_LO_NONZERO]);
        const float cb = rel_residual(b_meta[META_LO_NONZERO]);
        kappa = 1.02f * (ca + cb) + 2.4e-7f + (float)(d / 16 + 4) * 1.1920929e-7f;
        const float sq = sqrtf((float)d) * 5.9604645e-8f;                         // 2 * 2^-25 * sqrt(d)
        sq_ = sq;
        ca_ = ca;
        uf_a = ca != 0.f ? sq * a_meta[META_INV_SCALE] : 0.f;                     // times |b|
        uf_b = cb != 0.f ? sq * b_meta[META_INV_SCALE] : 0.f;                     // times |a|
        nb_max = sqrtf(b_meta[META_MAX_NORM_SQ]);
    }
    // row operands prepared with a per-row scale (ise_prepare_rows): the FP16-underflow term of the A planes follows
    // the row's own scale instead of the tensor's
    __device__ __forceinline__ void set_a_inv_scale(float a_inv) {
        uf_a = ca_ != 0.f ? sq_ * a_inv : 0.f;
    }
    // every coarse inner product of a row with squared norm `an` is within eps(an) of the exact one
    __device__ __forceinline__ float eps(float an) const {
        const float na = sqrtf(an);
        return kappa * nb_max * na + uf_a * nb_max + uf_b * na;
    }
};

#endif  // __CUDACC__
