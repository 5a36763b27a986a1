// Operand preparation: FP32 / uint8 rows -> scaled FP16 hi/lo planes + exact FP32 row norms,
// and faiss.normalize_L2.  HBM-bound streaming kernels: one warp per row, 128-bit loads.
#include "common.cuh"
#include "rows_convert.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarpsPerBlock = kThreads / 32;

__device__ __forceinline__ float absmax4(float4 v) {
    return fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)));
}

// Besides the absolute maximum, the pass records whether every element would be EXACT in one FP16 plane at the
// power-of-two scale the maximum implies (at most 11 significant bits, and not so small next to the maximum that
// it would leave FP16's normal range): integer-valued descriptors (SIFT, ORB as float) are, and the conversion
// pass then skips the lo plane's stores altogether (a quarter of its HBM traffic).
__device__ __forceinline__ void exact_probe(float v, unsigned& wide, float& mn) {
    const unsigned b = __float_as_uint(v);
    wide |= b & 0x1FFFu;                                   // mantissa bits FP16 cannot hold
    wide |= ((b & 0x7F800000u) == 0x7F800000u) ? 0x80000000u : 0u;   // NaN / Inf: reported through META_NONFINITE
    const float a = fabsf(v);
    mn = (a > 0.f) ? fminf(mn, a) : mn;
}

__global__ void absmax_f32_kernel(const float* __restrict__ x, int64_t n, int d, int64_t ldx, float* meta) {
    const int lane = threadIdx.x & 31;
    float m = 0.f;
    unsigned wide = 0u;
    float mn = 3.402823466e+38f;
    if (ldx == d && ((n * d) % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0)) {
        // contiguous matrix: a flat stream of float4, four independent loads in flight per thread
        const float4* x4 = reinterpret_cast<const float4*>(x);
        const int64_t total = n * d / 4;
        const int64_t stride = (int64_t)gridDim.x * kThreads;
        int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
        for (; i + 3 * stride < total; i += 4 * stride) {
            const float4 a = __ldg(x4 + i), b = __ldg(x4 + i + stride), c = __ldg(x4 + i + 2 * stride),
                         e = __ldg(x4 + i + 3 * stride);
            m = fmaxf(m, fmaxf(fmaxf(absmax4(a), absmax4(b)), fmaxf(absmax4(c), absmax4(e))));
            const float4 q[4] = {a, b, c, e};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                exact_probe(q[u].x, wide, mn); exact_probe(q[u].y, wide, mn);
                exact_probe(q[u].z, wide, mn); exact_probe(q[u].w, wide, mn);
            }
        }
        for (; i < total; i += stride) {
            const float4 a = __ldg(x4 + i);
            m = fmaxf(m, absmax4(a));
            exact_probe(a.x, wide, mn); exact_probe(a.y, wide, mn); exact_probe(a.z, wide, mn); exact_probe(a.w, wide, mn);
        }
    } else {
        const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
        const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
        for (int64_t r = warp; r < n; r += nwarps) {
            const float* row = x + r * ldx;
            for (int c = lane; c < d; c += 32) {
                const float v = __ldg(row + c);
                m = fmaxf(m, fabsf(v));
                exact_probe(v, wide, mn);
            }
        }
    }
    m = warp_max(m);
    wide = __reduce_or_sync(0xffffffffu, wide);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if (lane == 0) {
        if (wide & 0x80000000u) meta[META_NONFINITE] = 1.f;
        if (wide) meta[META_WIDE_MANTISSA] = 1.f;
        if (mn < 3.402823466e+38f)
            atomicMax(reinterpret_cast<int*>(meta + META_MIN_NONZERO), 0x7f800000 - __float_as_int(mn));
    }
    // non-negative finite floats order like their bit patterns; NaN/Inf are rejected by the host API
    if (lane == 0 && m > 0.f) atomicMax(reinterpret_cast<int*>(meta + META_ABSMAX), __float_as_int(m));
}

__device__ __forceinline__ float scale_from_absmax(float absmax) {
    if (!(absmax > 0.f)) return 1.f;
    int e = ilogbf(absmax);  // absmax in [2^e, 2^(e+1))
    int s = 13 - e;          // absmax * 2^s in [2^13, 2^14): inside fp16 range with headroom
    s = max(-100, min(100, s));
    return ldexpf(1.f, s);
}

template <typename T>
__device__ __forceinline__ float load_as_f32(const T* p);
template <>
__device__ __forceinline__ float load_as_f32<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float load_as_f32<uint8_t>(const uint8_t* p) { return (float)__ldg(p); }

// (publish_lo_residual: rows_convert.cuh)

template <typename T>
__global__ void prepare_planes_kernel(const T* __restrict__ x, int64_t n, int d, int64_t ldx,
                                      __half* __restrict__ hi, __half* __restrict__ lo, int64_t ldp,
                                      float* __restrict__ norms, float* meta, bool fixed_unit_scale) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    const float scale = fixed_unit_scale ? 1.f : scale_from_absmax(meta[META_ABSMAX]);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        meta[META_SCALE] = scale;
        meta[META_INV_SCALE] = 1.f / scale;
        if (fixed_unit_scale) meta[META_ABSMAX] = 255.f;
    }
    bool any_lo = false;
    float max_ss = 0.f, max_rs = 0.f;
    const int dp = (int)ldp;
    for (int64_t r = warp; r < n; r += nwarps) {
        const T* row = x + r * ldx;
        __half* hrow = hi + r * ldp;
        __half* lrow = lo ? lo + r * ldp : nullptr;
        float ss = 0.f, rs = 0.f;
        // two columns per lane per step so the plane stores are 32-bit
        for (int c = lane * 2; c < dp; c += 64) {
            float v0 = (c < d) ? load_as_f32<T>(row + c) : 0.f;
            float v1 = (c + 1 < d) ? load_as_f32<T>(row + c + 1) : 0.f;
            ss = fmaf(v0, v0, ss);
            ss = fmaf(v1, v1, ss);
            float s0 = v0 * scale, s1 = v1 * scale;
            __half h0 = __float2half_rn(s0), h1 = __float2half_rn(s1);
            const float e0 = s0 - __half2float(h0), e1 = s1 - __half2float(h1);    // exact residuals of the hi plane
            rs = fmaf(e0, e0, rs);
            rs = fmaf(e1, e1, rs);
            __half l0 = __float2half_rn(e0);
            __half l1 = __float2half_rn(e1);
            *reinterpret_cast<__half2*>(hrow + c) = __halves2half2(h0, h1);
            if (lrow) *reinterpret_cast<__half2*>(lrow + c) = __halves2half2(l0, l1);
            any_lo |= (__half2float(l0) != 0.f) | (__half2float(l1) != 0.f);
        }
        ss = warp_sum(ss);
        if (norms && lane == 0) norms[r] = ss;
        max_ss = fmaxf(max_ss, ss);
        if (__any_sync(0xffffffffu, rs != 0.f)) max_rs = fmaxf(max_rs, warp_sum(rs) / (scale * scale * ss));   // relative
    }
    // largest row norm^2 (non-negative floats order like ints; one atomic per warp): the coarse-pass
    // error bound of ise_rescore_select needs it
    if (lane == 0 && max_ss > 0.f) atomicMax(reinterpret_cast<int*>(meta + META_MAX_NORM_SQ), __float_as_int(max_ss));
    publish_lo_residual(meta, __any_sync(0xffffffffu, any_lo), max_rs, lane);
}

// Fast path, float32 rows with d % 4 == 0 (16-byte aligned rows and planes): a lane converts four consecutive
// columns per step (one 128-bit load, one 64-bit store per plane) and every warp keeps ROWS rows in flight --
// one row per warp iteration leaves ~32 KB of loads in flight per SM, which is what held the first version at
// 0.6 of HBM peak (profiles/r01_findings.md section 9).
// EXACT selects which of the two cases a launch handles; the host launches BOTH instantiations back to back and each
// returns at once unless the absmax pass proved (EXACT) / did not prove (!EXACT) that one FP16 plane holds every
// element exactly -- the decision lives on the device, and the light exact path is not held to the register budget
// of the general one (89 registers -> 2 CTAs per SM when they shared a kernel).
template <int ROWS, bool EXACT>
__global__ void __launch_bounds__(kThreads, EXACT ? 5 : 3) prepare_planes_f32x4_kernel(const float* __restrict__ x, int64_t n, int d, int64_t ldx,
                                            __half* __restrict__ hi, __half* __restrict__ lo, int64_t ldp,
                                            float* __restrict__ norms, float* meta) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    const float scale = scale_from_absmax(meta[META_ABSMAX]);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        meta[META_SCALE] = scale;
        meta[META_INV_SCALE] = 1.f / scale;
    }
    // every element exact in the hi plane (<= 11 significant bits, scaled value in FP16's normal range): the lo plane
    // is all zeros, META_LO_NONZERO stays 0 and nobody will ever read it -- do not write it
    const int mn_code = reinterpret_cast<const int*>(meta)[META_MIN_NONZERO];
    const float mn_abs = mn_code ? __int_as_float(0x7f800000 - mn_code) : 1.f;
    const bool exact = meta[META_WIDE_MANTISSA] == 0.f && mn_abs * scale >= 6.103515625e-05f;
    if (exact != EXACT) return;
    if (EXACT) lo = nullptr;
    bool any_lo = false;
    float max_ss = 0.f, max_rs = 0.f;
    const int d4 = d >> 2, dp4 = (int)(ldp >> 2);
    for (int64_t r0 = warp * ROWS; r0 < n; r0 += nwarps * ROWS) {
        float ss[ROWS], rs[EXACT ? 1 : ROWS];
#pragma unroll
        for (int i = 0; i < ROWS; ++i) ss[i] = 0.f;
#pragma unroll
        for (int i = 0; i < (EXACT ? 1 : ROWS); ++i) rs[i] = 0.f;
        for (int c = lane; c < dp4; c += 32) {
            float4 v[ROWS];
#pragma unroll
            for (int i = 0; i < ROWS; ++i) {
                const int64_t r = r0 + i;
                v[i] = (r < n && c < d4) ? __ldg(reinterpret_cast<const float4*>(x + r * ldx) + c)
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < ROWS; ++i) {
                const int64_t r = r0 + i;
                if (r >= n) continue;
                ss[i] = fmaf(v[i].x, v[i].x, ss[i]); ss[i] = fmaf(v[i].y, v[i].y, ss[i]);
                ss[i] = fmaf(v[i].z, v[i].z, ss[i]); ss[i] = fmaf(v[i].w, v[i].w, ss[i]);
                if (EXACT) {
                    // one packed conversion per two elements, no residual: the float -> half conversions (not HBM)
                    // bound this kernel when every element goes through three of them
                    const __half2 ha = __floats2half2_rn(v[i].x * scale, v[i].y * scale);
                    const __half2 hb = __floats2half2_rn(v[i].z * scale, v[i].w * scale);
                    uint2 hv;
                    hv.x = *reinterpret_cast<const uint32_t*>(&ha); hv.y = *reinterpret_cast<const uint32_t*>(&hb);
                    reinterpret_cast<uint2*>(hi + r * ldp)[c] = hv;
                    continue;
                }
                __half h0, h1, h2, h3, l0, l1, l2, l3;
                split_f16(v[i].x * scale, h0, l0); split_f16(v[i].y * scale, h1, l1);
                split_f16(v[i].z * scale, h2, l2); split_f16(v[i].w * scale, h3, l3);
                if (!EXACT) {   // exact residuals of the hi plane (what the coarse pass neglects)
                    const float e0 = v[i].x * scale - __half2float(h0), e1 = v[i].y * scale - __half2float(h1);
                    const float e2 = v[i].z * scale - __half2float(h2), e3 = v[i].w * scale - __half2float(h3);
                    rs[i] = fmaf(e0, e0, rs[i]); rs[i] = fmaf(e1, e1, rs[i]);
                    rs[i] = fmaf(e2, e2, rs[i]); rs[i] = fmaf(e3, e3, rs[i]);
                }
                const __half2 ha = __halves2half2(h0, h1), hb = __halves2half2(h2, h3);
                const __half2 la = __halves2half2(l0, l1), lb = __halves2half2(l2, l3);
                uint2 hv, lv;
                hv.x = *reinterpret_cast<const uint32_t*>(&ha); hv.y = *reinterpret_cast<const uint32_t*>(&hb);
                lv.x = *reinterpret_cast<const uint32_t*>(&la); lv.y = *reinterpret_cast<const uint32_t*>(&lb);
                reinterpret_cast<uint2*>(hi + r * ldp)[c] = hv;
                if (lo) reinterpret_cast<uint2*>(lo + r * ldp)[c] = lv;
                any_lo |= ((lv.x | lv.y) & 0x7FFF7FFFu) != 0u;
            }
        }
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
            const float t = warp_sum(ss[i]);
            if (r0 + i < n) {
                if (norms && lane == 0) norms[r0 + i] = t;
                max_ss = fmaxf(max_ss, t);
            }
            if (!EXACT && r0 + i < n && t > 0.f) max_rs = fmaxf(max_rs, warp_sum(rs[EXACT ? 0 : i]) / (scale * scale * t));
        }
    }
    if (lane == 0 && max_ss > 0.f) atomicMax(reinterpret_cast<int*>(meta + META_MAX_NORM_SQ), __float_as_int(max_ss));
    if (!EXACT) publish_lo_residual(meta, __any_sync(0xffffffffu, any_lo), max_rs, lane);
}

// ---- single-pass preparation of ROW operands (descriptors / queries) ------------------------------------------------
// The per-tensor scale of the kernels above needs the absolute maximum first, i.e. a second read of the matrix
// (10 B moved per element for 6 B of algorithmic traffic at the C2 assign step).  A row operand does not need a common
// scale: the selection epilogue owns one row per thread and multiplies the accumulator by that row's 1 / scale, and an
// arg-max is invariant to it anyway.  So a warp reads its rows ONCE, takes each row's own absolute maximum with a
// shuffle reduction, and converts from registers: 4 B read + 2 B (+ 2 B when the row is not exact in one FP16 plane)
// written per element.  Rows whose lo part is all zero skip the lo store (integer-valued SIFT / ORB-as-float: all of
// them); they are recorded in lo_skipped[] and zeroed by lo_fixup_kernel only if some other row did need its lo plane.
// NaN / Inf are detected on the way (meta[NONFINITE]) so that k-means training needs no separate validation pass.
// The first version of this kernel ran at 0.56-0.60 of HBM peak and ncu showed why: 146 warp instructions per row
// (ilogbf / ldexpf / a division for the scale, a float NaN test per element, a multiply + three compares per element for
// the exactness test) -- issue-bound, not memory-bound.  Everything that is per-row-uniform is integer bit arithmetic
// now, and the per-element work is four integer min/max/or + one FMA (rows_convert.cuh):
//   * |x| as an unsigned bit pattern orders like the value and keeps NaN / Inf visible (>= 0x7F800000), so one integer
//     max gives both the row's absolute maximum (-> its power-of-two scale: exponent arithmetic) and the non-finite flag;
//   * an element is exact in one FP16 plane iff its low 13 mantissa bits are zero (scaling by a power of two does not
//     change them) and it does not fall below FP16's normal range once scaled: min over (|x| bits - 1) against one
//     per-row threshold (zero wraps to 0xFFFFFFFF and never counts).
template <int ROWS, int NV>
__global__ void __launch_bounds__(kThreads, 4)
prepare_rows_f32_kernel(const float* __restrict__ x, int64_t n, int d, int64_t ldx, __half* __restrict__ hi,
                        __half* __restrict__ lo, int64_t ldp, float* __restrict__ norms, float* __restrict__ row_inv,
                        uint8_t* __restrict__ lo_skipped, float* meta) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    if (blockIdx.x == 0 && threadIdx.x == 0) { meta[META_SCALE] = 1.f; meta[META_INV_SCALE] = 1.f; }
    const int d4 = d >> 2, dp4 = (int)(ldp >> 2);
    RowStats st;
    for (int64_t r0 = warp * ROWS; r0 < n; r0 += nwarps * ROWS)
        convert_row_group<ROWS, NV>(x, n, d4, dp4, ldx, hi, lo, ldp, norms, row_inv, lo_skipped, r0, lane, st);
    commit_row_stats(st, meta, lane);
}

// rows that skipped their (all-zero) lo store get it now -- only when the tensor as a whole has a lo plane in use
__global__ void lo_fixup_kernel(__half* __restrict__ lo, int64_t n, int64_t ldp, const uint8_t* __restrict__ lo_skipped,
                                const float* __restrict__ meta) {
    if (meta[META_LO_NONZERO] == 0.f) return;
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t r0 = warp * 32; r0 < n; r0 += nwarps * 32) {
        const unsigned mask = __ballot_sync(0xffffffffu, r0 + lane < n && lo_skipped[r0 + lane] != 0);
        for (unsigned m = mask; m; m &= m - 1) {
            uint2* row = reinterpret_cast<uint2*>(lo + (r0 + __ffs(m) - 1) * ldp);
            for (int c = lane; c < (int)(ldp >> 2); c += 32) row[c] = make_uint2(0u, 0u);
        }
    }
}

__global__ void fill_row_inv_kernel(float* __restrict__ row_inv, int64_t n, float* meta) {
    const float inv = meta[META_INV_SCALE];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        row_inv[i] = inv;
}

// Fast path, uint8 rows (ORB / BRISK bytes) with d % 16 == 0 and d / 16 a power of two <= 32, contiguous rows and
// planes: the matrix is a flat stream of 16-byte groups; a lane converts one group (16 columns: one 128-bit
// load, two 128-bit stores), and the LPR = d / 16 lanes that share a row reduce its norm with shuffles.
__global__ void prepare_planes_u8x16_kernel(const uint8_t* __restrict__ x, int64_t n, int d, __half* __restrict__ hi,
                                            float* __restrict__ norms, float* meta) {
    const int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        meta[META_SCALE] = 1.f;
        meta[META_INV_SCALE] = 1.f;
        meta[META_ABSMAX] = 255.f;
    }
    const int lpr = d >> 4;                               // lanes per row
    const int64_t groups = n * lpr;
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    const int64_t g_end = (groups + 31) / 32 * 32;        // whole warps stay converged for the shuffles
    float max_ss = 0.f;
    auto convert = [&](int64_t g, const uint4& v) {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        uint32_t out[8];
        float ss = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float b0 = (float)(w[i] & 0xFFu), b1 = (float)((w[i] >> 8) & 0xFFu);
            const float b2 = (float)((w[i] >> 16) & 0xFFu), b3 = (float)(w[i] >> 24);
            ss = fmaf(b0, b0, ss); ss = fmaf(b1, b1, ss); ss = fmaf(b2, b2, ss); ss = fmaf(b3, b3, ss);
            const __half2 p = __floats2half2_rn(b0, b1), q = __floats2half2_rn(b2, b3);
            out[2 * i] = *reinterpret_cast<const uint32_t*>(&p);
            out[2 * i + 1] = *reinterpret_cast<const uint32_t*>(&q);
        }
        if (g < groups) {
            uint4* dst = reinterpret_cast<uint4*>(hi) + 2 * g;
            dst[0] = make_uint4(out[0], out[1], out[2], out[3]);
            dst[1] = make_uint4(out[4], out[5], out[6], out[7]);
        }
        for (int o = lpr >> 1; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (g < groups && (lane & (lpr - 1)) == 0) {
            if (norms) norms[g / lpr] = ss;
            max_ss = fmaxf(max_ss, ss);
        }
    };
    // four independent 128-bit loads in flight per thread
    for (int64_t g = (int64_t)blockIdx.x * kThreads + threadIdx.x; g < g_end; g += 4 * stride) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t gu = g + u * stride;
            v[u] = gu < groups ? __ldg(reinterpret_cast<const uint4*>(x) + gu) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (g + u * stride < g_end) convert(g + u * stride, v[u]);
    }
    max_ss = warp_max(max_ss);
    if (lane == 0 && max_ss > 0.f) atomicMax(reinterpret_cast<int*>(meta + META_MAX_NORM_SQ), __float_as_int(max_ss));
}

// faiss fvec_renorm_L2: x *= 1 / sqrtf(sum x^2), zero rows untouched.  ROWS rows in flight per warp (one row per
// warp iteration keeps too few loads in flight to fill HBM); the second sweep re-reads the rows from L1/L2.
template <int ROWS>
__global__ void normalize_l2_kernel(float* __restrict__ x, int64_t n, int d) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    const bool vec = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    for (int64_t r0 = warp * ROWS; r0 < n; r0 += nwarps * ROWS) {
        float ss[ROWS];
#pragma unroll
        for (int i = 0; i < ROWS; ++i) ss[i] = 0.f;
        if (vec) {
            for (int c = lane; c < d / 4; c += 32) {
                float4 v[ROWS];
#pragma unroll
                for (int i = 0; i < ROWS; ++i)
                    v[i] = r0 + i < n ? reinterpret_cast<const float4*>(x + (r0 + i) * (int64_t)d)[c] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    ss[i] = fmaf(v[i].x, v[i].x, ss[i]); ss[i] = fmaf(v[i].y, v[i].y, ss[i]);
                    ss[i] = fmaf(v[i].z, v[i].z, ss[i]); ss[i] = fmaf(v[i].w, v[i].w, ss[i]);
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < ROWS; ++i)
                if (r0 + i < n)
                    for (int c = lane; c < d; c += 32) { const float v = x[(r0 + i) * (int64_t)d + c]; ss[i] = fmaf(v, v, ss[i]); }
        }
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
            const float t = warp_sum(ss[i]);
            if (r0 + i >= n || !(t > 0.f)) continue;
            const float inv = 1.0f / sqrtf(t);  // fvec_renorm_L2: inv_nr = 1.0 / sqrtf(nr)
            float* row = x + (r0 + i) * (int64_t)d;
            if (vec) {
                float4* row4 = reinterpret_cast<float4*>(row);
                for (int c = lane; c < d / 4; c += 32) {
                    float4 v = row4[c];
                    v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
                    row4[c] = v;
                }
            } else {
                for (int c = lane; c < d; c += 32) row[c] *= inv;
            }
        }
    }
}

int grid_for_rows(const ise_ctx* ctx, int64_t n) {
    int64_t blocks = ceil_div64(n, kWarpsPerBlock);
    int64_t cap = (int64_t)ctx->sm_count * 8;  // 8 resident 256-thread CTAs per SM
    return (int)std::max<int64_t>(1, std::min(blocks, cap));
}

}  // namespace

ISE_EXPORT int ise_prepare_planes(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx,
                                  void* hi, void* lo, int64_t ldp, float* norms, float* meta, void* stream) {
    ISE_CHECK_ARG(ctx && meta && hi);
    ISE_CHECK_ARG(n >= 0 && d > 0 && ldx >= d && ldp >= d && ldp % 8 == 0);
    ISE_CHECK_ARG(dtype == ISE_DTYPE_F32 || dtype == ISE_DTYPE_U8);
    DeviceGuard g(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    ISE_CUDA(cudaMemsetAsync(meta, 0, META_FLOATS * sizeof(float), st));
    if (n == 0) return 0;
    ISE_CHECK_ARG(x != nullptr);
    const int grid = grid_for_rows(ctx, n);
    const bool al16 = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15) == 0;
    if (dtype == ISE_DTYPE_F32) {
        absmax_f32_kernel<<<grid, kThreads, 0, st>>>((const float*)x, n, d, ldx, meta);
        ISE_LAUNCH_CHECK();
        if (d % 4 == 0 && ldx % 4 == 0 && al16) {
            constexpr int ROWS = 4;
            const int g4 = grid_for_rows(ctx, ceil_div64(n, ROWS));
            prepare_planes_f32x4_kernel<ROWS, true><<<g4, kThreads, 0, st>>>((const float*)x, n, d, ldx, (__half*)hi,
                                                                             (__half*)lo, ldp, norms, meta);
            ISE_LAUNCH_CHECK();
            prepare_planes_f32x4_kernel<ROWS, false><<<g4, kThreads, 0, st>>>((const float*)x, n, d, ldx, (__half*)hi,
                                                                              (__half*)lo, ldp, norms, meta);
        } else {
            prepare_planes_kernel<float><<<grid, kThreads, 0, st>>>((const float*)x, n, d, ldx, (__half*)hi,
                                                                    (__half*)lo, ldp, norms, meta, false);
        }
    } else {
        const int lpr = d / 16;
        if (d % 16 == 0 && lpr <= 32 && (lpr & (lpr - 1)) == 0 && ldx == d && ldp == d && al16 && lo == nullptr) {
            const int64_t groups = n * lpr;
            const int gu = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(groups, kThreads), (int64_t)ctx->sm_count * 8));
            prepare_planes_u8x16_kernel<<<gu, kThreads, 0, st>>>((const uint8_t*)x, n, d, (__half*)hi, norms, meta);
        } else {
            prepare_planes_kernel<uint8_t><<<grid, kThreads, 0, st>>>((const uint8_t*)x, n, d, ldx, (__half*)hi,
                                                                      (__half*)lo, ldp, norms, meta, true);
        }
    }
    ISE_LAUNCH_CHECK();
    return 0;
}

// Row-operand preparation (descriptors, queries): one pass, per-row power-of-two scales returned as row_inv[n] =
// 1 / scale.  Shapes the single-pass kernel does not cover (uint8 rows: already one pass with scale 1; float32 rows
// with d % 4 != 0, unaligned, or d > 512) go through ise_prepare_planes and get a constant row_inv.
ISE_EXPORT int ise_prepare_rows(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx, void* hi, void* lo,
                                int64_t ldp, float* norms, float* row_inv, uint8_t* lo_skipped, float* meta, void* stream) {
    ISE_CHECK_ARG(ctx && meta && row_inv);
    ISE_CHECK_ARG(n >= 0 && d > 0 && ldx >= d && ldp >= d && ldp % 8 == 0);
    ISE_CHECK_ARG(dtype == ISE_DTYPE_F32 || dtype == ISE_DTYPE_U8);
    ISE_CHECK_ARG(lo == nullptr || lo_skipped != nullptr);
    DeviceGuard g(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        ISE_CUDA(cudaMemsetAsync(meta, 0, META_FLOATS * sizeof(float), st));
        return 0;
    }
    ISE_CHECK_ARG(x && hi);
    const bool al16 = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15) == 0;
    if (dtype == ISE_DTYPE_F32 && d % 4 == 0 && ldx % 4 == 0 && al16 && ldp <= 512) {
        ISE_CUDA(cudaMemsetAsync(meta, 0, META_FLOATS * sizeof(float), st));
        const int nv = (int)((ldp / 4 + 31) / 32);
#define ISE_ROWS_ARGS (const float*)x, n, d, ldx, (__half*)hi, (__half*)lo, ldp, norms, row_inv, lo_skipped, meta
        if (nv <= 1) prepare_rows_f32_kernel<4, 1><<<grid_for_rows(ctx, ceil_div64(n, 4)), kThreads, 0, st>>>(ISE_ROWS_ARGS);
        else if (nv == 2) prepare_rows_f32_kernel<4, 2><<<grid_for_rows(ctx, ceil_div64(n, 4)), kThreads, 0, st>>>(ISE_ROWS_ARGS);
        else prepare_rows_f32_kernel<2, 4><<<grid_for_rows(ctx, ceil_div64(n, 2)), kThreads, 0, st>>>(ISE_ROWS_ARGS);
#undef ISE_ROWS_ARGS
        ISE_LAUNCH_CHECK();
        if (lo) {
            lo_fixup_kernel<<<grid_for_rows(ctx, ceil_div64(n, 32)), kThreads, 0, st>>>((__half*)lo, n, ldp, lo_skipped, meta);
            ISE_LAUNCH_CHECK();
        }
        return 0;
    }
    if (ise_prepare_planes(ctx, x, dtype, n, d, ldx, hi, lo, ldp, norms, meta, stream)) return 1;
    fill_row_inv_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(n, 256), 1024), 256, 0, st>>>(row_inv, n, meta);
    ISE_LAUNCH_CHECK();
    return 0;
}

// the absmax pass on its own: meta[ABSMAX], meta[NONFINITE] (+ the exactness probes) of a float32 matrix.  Used to
// validate a training set that is about to be sub-sampled (Clustering::train checks ALL of its input for NaN / Inf).
ISE_EXPORT int ise_scan_f32(ise_ctx* ctx, const float* x, int64_t n, int d, int64_t ldx, float* meta, void* stream) {
    ISE_CHECK_ARG(ctx && meta && n >= 0 && d > 0 && ldx >= d);
    DeviceGuard g(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    ISE_CUDA(cudaMemsetAsync(meta, 0, META_FLOATS * sizeof(float), st));
    if (n == 0) return 0;
    ISE_CHECK_ARG(x != nullptr);
    absmax_f32_kernel<<<grid_for_rows(ctx, n), kThreads, 0, st>>>(x, n, d, ldx, meta);
    ISE_LAUNCH_CHECK();
    return 0;
}

ISE_EXPORT int ise_normalize_l2(ise_ctx* ctx, float* x, int64_t n, int d, void* stream) {
    ISE_CHECK_ARG(ctx && d > 0 && n >= 0);
    if (n == 0) return 0;
    ISE_CHECK_ARG(x != nullptr);
    DeviceGuard g(ctx->device);
    normalize_l2_kernel<4><<<grid_for_rows(ctx, ceil_div64(n, 4)), kThreads, 0, (cudaStream_t)stream>>>(x, n, d);
    ISE_LAUNCH_CHECK();
    return 0;
}

// used by ise_assign_fused (gemm_select.cu): gated on the device-side meta[LO_NONZERO] flag
int ise_internal_lo_fixup(ise_ctx* ctx, void* lo, int64_t n, int64_t ldp, const uint8_t* lo_skipped, const float* meta,
                          void* stream) {
    lo_fixup_kernel<<<grid_for_rows(ctx, ceil_div64(n, 32)), kThreads, 0, (cudaStream_t)stream>>>((__half*)lo, n, ldp,
                                                                                                lo_skipped, meta);
    ISE_LAUNCH_CHECK();
    return 0;
}
