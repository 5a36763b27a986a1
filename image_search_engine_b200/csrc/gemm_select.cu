// Fused distance contraction + selection on the Blackwell tensor cores.
//
//   rows  A : m x d   (descriptors for k-means assign / quantisation, queries for kNN)
//   cols  B : n x d   (centroids, database vectors)
//   out     : per row the topk best columns under inner product or squared L2
//
// The m x n score matrix only ever exists as 128 x 256 FP32 accumulator tiles in TMEM.
// A persistent, warp-specialised CTA (one per SM) runs three roles:
//   warp 0   TMA producer : cp.async.bulk.tensor loads of the FP16 hi/lo planes (128B swizzle)
//   warp 1   MMA issuer   : tcgen05.mma kind::f16, split products hi*hi + hi*lo + lo*hi into one
//                           TMEM accumulator (2 accumulators x 256 columns, double buffered)
//   warps 4-7 epilogue    : tcgen05.ld the accumulator, per-row running top-1 / top-k in registers
//                           or thread-local lists while the next tile's MMAs run
// Replaces Faiss knn_inner_product / knn_L2sqr (sgemm + result handler) behind
// reference call sites kmeans_faiss.py:41,49 and engine.py:55.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "sm100_ptx.cuh"
#include "topk_list.cuh"
#include "rows_convert.cuh"

namespace gs {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_N = 256;
constexpr int BLOCK_K = 64;  // fp16 elements = one 128-byte swizzle span
constexpr int UMMA_K = 16;
constexpr int A_TILE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KiB
constexpr int B_TILE_BYTES = BLOCK_N * BLOCK_K * 2;  // 32 KiB
constexpr int EPI_WARP0 = 4;
// One epilogue warp per TMEM lane quadrant.  Two warps per quadrant (each scanning half of a tile's columns) measured
// slower for the coarse top-1 kernels at the d = 128 C2 shape: the split products are MMA-bound (nothing to gain, a
// hand-over to pay) and the one-product coarse pass is bound by the L2 -> shared-memory feed, not by the epilogue's
// TMEM reads (profiles/r01_findings.md section 8).
// The resident-row-tile kernels (ARES: the verified one-product assign at d <= 128) are bound by their epilogue, not by
// the tensor pipe: a single warp per scheduler runs the dependent max / select chains at ~0.27 IPC (ncu, profiles/
// r02_findings.md), so they get two warps per quadrant to interleave.
__host__ __device__ constexpr int epi_halves(bool ares) { return ares ? 2 : 1; }
// conv: four extra warps that convert the NEXT work item's float32 rows into FP16 planes while the current item is
// being multiplied (fused assign, see the CONV template parameter)
__host__ __device__ constexpr int num_threads(int mt = 1, bool conv = false, bool ares = false) {
    return 128 + 128 * epi_halves(ares) * mt + (conv ? 128 : 0);
}
constexpr int TMEM_COLS = 512;  // 2 accumulator stages x BLOCK_N fp32 columns
constexpr int AUX_BYTES = 8192;
constexpr int SMEM_LIMIT = 232448;  // 227 KiB opt-in per CTA on sm_100

// cg = CTAs per MMA (cta_group): with 2, each CTA of the pair stages only half of every B tile
// mt = row tiles per CTA: with 2, one CTA runs two 128-row tiles against every B tile it stages
__host__ __device__ constexpr int stage_bytes(int pa, int pb, int cg = 1, int mt = 1) {
    return mt * pa * A_TILE_BYTES + pb * (B_TILE_BYTES / cg);
}
__host__ __device__ constexpr int num_stages(int pa, int pb, int cg = 1, int mt = 1) {
    int s = (SMEM_LIMIT - AUX_BYTES - 1024) / stage_bytes(pa, pb, cg, mt);
    return s > 6 ? 6 : s;
}

// ARES kernels: two resident A slots of up to two 64-column k-blocks each, stages of B only
__host__ __device__ constexpr int ares_bytes() { return 2 * 2 * A_TILE_BYTES; }
__host__ __device__ constexpr int ares_stage_bytes(int pb, int cg) { return pb * (B_TILE_BYTES / cg); }
__host__ __device__ constexpr int ares_stages(int pb, int cg) {
    int s = (SMEM_LIMIT - AUX_BYTES - 1024 - ares_bytes()) / ares_stage_bytes(pb, cg);
    return s > 8 ? 8 : s;
}

struct Params {
    int64_t m, n;
    int d;
    int n_mtiles;         // ceil(m / 128)
    int n_ntiles;         // ceil(n / 256)
    int tiles_per_split;  // N tiles handled by one work item
    int n_splits;
    int topk;
    int64_t id_base;
    const float* a_meta;
    const float* b_meta;
    const float* a_norms;
    const float* b_norms;
    const float* a_row_inv; // optional [m]: per-row 1 / scale of the A planes (single-pass row preparation); overrides a_meta's
    const float* row_seed;  // optional [m]: a per-row score every kept candidate must beat (real units)
    int32_t* row_count;     // collect mode (KSEL == 0): per-row append counters, out_* are [m, topk] buffers
    int32_t* flag_rows;     // optional (top-1 only): rows whose winner is not provably unique under the
    int32_t* flag_count;    //   coarse error bound are appended here for a full-precision re-run
    float* out_val;    // [n_splits, m, topk]
    int64_t* out_idx;  // [n_splits, m, topk]
    // soft lock-step (optional): the CTAs that walk one column range in the same round check in every `sync_every`
    // column tiles and wait (bounded) for the slowest of them, so that every B tile they share is still in L2 when
    // the last of them asks for it
    int32_t* sync_cnt;  // [rounds * n_splits, sync_ncp] zero-initialised, or nullptr
    int sync_every;
    int sync_ncp;
    // fused assign (CONV kernels): the raw float32 rows and the WRITABLE views of the A operand the converter warps fill
    const float* a_raw;
    int64_t lda_raw;
    __half* a_hi_w;
    __half* a_lo_w;         // nullable
    int64_t lda_w;
    float* a_norms_w;
    float* a_row_inv_w;
    uint8_t* a_lo_skipped;  // nullable (required with a_lo_w)
    float* a_meta_w;
    // regular kernels: return at once when the A operand turned out exact in its hi plane (meta[LO_NONZERO] == 0); the
    // launch that follows an optimistic hi-only fused assign and repeats it with the lo planes only if they exist
    int skip_if_a_exact;
    // verified top-1 pipeline (no host synchronisation between its launches):
    const int32_t* gate;     // optional: the whole launch returns at once unless *gate != 0 (device-side "needed" flag)
    const int32_t* m_dev;    // optional: the number of rows actually present (<= m, which then is the buffers' capacity)
    const int32_t* row_map;  // optional [m]: results of row r are written to out_*[row_map[r]] (compacted re-runs)
};

struct Aux {  // lives after the stage ring in dynamic shared memory
    uint64_t full[8];
    uint64_t empty[8];
    uint64_t tmem_full[2];
    uint64_t tmem_empty[2];
    uint64_t a_ready[2];    // CONV: converter warps -> producer / epilogue, one slot per work-item parity
    uint64_t a_free[2];     // CONV: epilogue -> converter (the converter stays at most two items ahead)
    uint32_t tmem_base;
    uint32_t pad_[3];
    float bnorm[2][BLOCK_N];
    float xbest[3][BLOCK_M];   // column slices 1.. -> slice 0 hand-over of the top-1 state at the end of a work item
    float xrun[3][BLOCK_M];
    int xid[3][BLOCK_M];
};
static_assert(sizeof(Aux) <= AUX_BYTES, "aux area too small");

// selection state per epilogue thread: top-1 scalars, 32 register-resident slots, or a 128-entry sorted
// thread-local list
template <int KSEL> struct SelList { using type = TopKList<KSEL>; };
template <> struct SelList<1> { using type = TopKList<1>; };
template <> struct SelList<0> { using type = TopKList<1>; };   // collect mode keeps no list
template <> struct SelList<32> { using type = RegList32; };

// KSEL: 1 = running top-1 in registers; 0 = COLLECT: append every column beating the row's seed to a
// per-row global buffer (large k: nothing is ordered or evicted on the device, the exact re-score sorts);
// otherwise capacity of the per-thread candidate set.
// VERIFY (top-1 only): also track the exact runner-up and flag rows whose winner is not provably unique.
// CG = 2: CTA PAIRS (cluster of 2 on one TPC, tcgen05 cta_group::2).  The pair owns two adjacent row tiles
//   (M = 256 per MMA); each CTA stages its own A rows and only HALF of every B tile (128 of the 256
//   columns), so the L2 -> smem bytes per MMA cycle drop by ~40 % and stages get smaller (deeper ring).
//   Only the leader CTA issues MMAs; TMA completions of both CTAs signal the leader's `full` barrier;
//   tcgen05.commit multicasts `empty` / `tmem_full` to both CTAs; both epilogues arrive on the leader's
//   `tmem_empty`.  Each CTA's epilogue reads its own 128 TMEM lanes exactly as in the single-CTA case.
// MT = 2 (single CTA, CG == 1): the CTA owns TWO adjacent row tiles and runs both against every B tile it stages
//   (two 256-column accumulators = all of TMEM, so the accumulators are NOT double buffered: the epilogue of a
//   column tile and the MMAs of the next one alternate).  Halves the B bytes per MMA cycle like a CTA pair does,
//   without any cross-CTA signalling; pays off when a tile's MMAs (d / 64 * 512 cycles per row tile) dwarf its
//   epilogue, i.e. for the large-d coarse search pass, which is bound by the L2 -> shared-memory feed.
// CONV (fused assign, top-1 only): the kernel takes the RAW float32 rows.  Four extra warps convert the rows of the work
//   item this CTA will run NEXT into per-row-scaled FP16 planes (rows_convert.cuh: the single-pass preparation, same
//   code) and write planes, norms and per-row scales to global memory -- 32 KB per row tile that the TMA producer reads
//   straight back from L2 -- while the tensor pipe works on the current item.  The separate HBM-bound preparation pass
//   (0.15 ms of a 1.72 ms C2 step) disappears behind the MMAs; the planes / norms / scales stay valid afterwards
//   (re-score, k-means update).  Only the hi plane of A is multiplied: a tensor that turns out NOT to be exact in it
//   sets meta[LO_NONZERO] and the caller's follow-up launch (Params::skip_if_a_exact) repeats the assign with the lo
//   planes -- for descriptors (integer SIFT, ORB / BRISK as float) that launch returns at once.
// CL > 1 (CTA pairs only): CL pairs form ONE cluster of 2 CL CTAs on 2 CL adjacent row tiles and share every B tile:
//   each CTA fetches 1 / CL of its pair's half tile and MULTICASTS it to the CTAs of the same parity in the other pairs,
//   so a B tile is read from L2 once per cluster instead of once per pair (the large-d coarse pass is bound by the
//   L2 -> shared-memory feed: A 16 KB + B 16 KB per stage per SM becomes A 16 KB + B 16 / CL KB).  A stage may only be
//   overwritten when EVERY pair of the cluster has consumed it: each leader's tcgen05.commit of the `empty` barrier is
//   multicast to all 2 CL CTAs (barrier count CL).
// ARES (d <= 128, hi plane of A only): the row tile of a work item stays RESIDENT in shared memory (two slots, loaded with
//   the item's first stage) instead of being re-fetched with every column tile, and the stage ring carries B only.  The
//   one-product coarse pass at d = 128 needs 96 KB of operands per 1024 MMA cycles when A travels with every stage --
//   more than L2 feeds one SM -- and 32 KB (CTA pairs) with A resident.
template <int PA, int PB, bool L2, int KSEL, bool VERIFY, int CG, int MT = 1, bool CONV = false, int CL = 1, bool ARES = false>
__global__ void __launch_bounds__(num_threads(MT, CONV, ARES), 1)
gemm_select_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                   const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                   const Params p) {
    static_assert(MT == 1 || (CG == 1 && epi_halves(ARES) == 1), "two row tiles per CTA: single CTA, one warp per quadrant and tile");
    static_assert(!CONV || (PA == 1 && KSEL == 1 && MT == 1), "fused conversion: top-1, hi plane of A");
    static_assert(!ARES || (PA == 1 && MT == 1 && CL == 1), "resident row tile: hi plane of A, one row tile per CTA, no multicast");
    static_assert(CL == 1 || (CG == 2 && MT == 1 && !CONV && CL == 2), "multicast clusters are made of CTA pairs");
    // uniform over the whole grid, before any barrier / TMEM state exists
    if (!CONV && p.skip_if_a_exact && __ldcg(p.a_meta + META_LO_NONZERO) == 0.f) return;
    if (p.gate != nullptr && __ldcg(p.gate) == 0) return;
    int64_t m_rows = p.m;
    int n_mtiles = p.n_mtiles;
    if (p.m_dev != nullptr) {
        m_rows = min((int64_t)__ldcg(p.m_dev), p.m);
        n_mtiles = (int)((m_rows + BLOCK_M - 1) / BLOCK_M);
    }
    constexpr int A_RES_BYTES = ARES ? ares_bytes() : 0;
    constexpr int STAGES = ARES ? ares_stages(PB, CG) : num_stages(PA, PB, CG, MT);
    constexpr int STAGE_BYTES = ARES ? ares_stage_bytes(PB, CG) : stage_bytes(PA, PB, CG, MT);
    constexpr int A_BLOCK_BYTES = PA * A_TILE_BYTES;      // one row tile's planes inside a stage
    constexpr int B_OFFSET = ARES ? 0 : MT * A_BLOCK_BYTES;   // B planes follow the MT row tiles (ARES: the stage is B only)
    constexpr int CSIZE = CG * CL;                        // CTAs per cluster
    constexpr int GRP = CG * MT * CL;                     // row tiles per work item
    constexpr int B_LOAD_BYTES = B_TILE_BYTES / CG;   // this CTA's share of a B tile (one plane)
    constexpr int B_LOAD_ROWS = BLOCK_N / CG;
    constexpr int B_ISSUE_ROWS = B_LOAD_ROWS / CL;    // ... of which it fetches this many rows itself (CL > 1: multicast)
    constexpr int B_ISSUE_BYTES = B_LOAD_BYTES / CL;
    constexpr int HALVES = epi_halves(ARES);
    constexpr int NUM_EPI_THREADS = 128 * HALVES * MT;
    constexpr int COLS_PER_HALF = BLOCK_N / HALVES;
    static_assert(STAGES >= 2 && STAGES <= 8, "pipeline depth");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem_al = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* a_res = smem_al;                         // ARES: 2 slots x 2 k-blocks x 16 KB
    uint8_t* smem = smem_al + A_RES_BYTES;            // stage ring
    Aux* aux = reinterpret_cast<Aux*>(smem + STAGES * STAGE_BYTES);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_a_hi);
        ptx::prefetch_tensormap(&tm_b_hi);
        if (PA == 2) ptx::prefetch_tensormap(&tm_a_lo);
        if (PB == 2) ptx::prefetch_tensormap(&tm_b_lo);
    }
    const uint32_t cta_rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;     // rank in the cluster: pair (rank >> 1), CTA of the pair (rank & 1)
    const uint32_t pair_cta = cta_rank & 1u, pair_idx = cta_rank >> 1, leader_rank = cta_rank & ~1u;
    const bool leader = pair_cta == 0;
    const uint16_t pair_mask = (uint16_t)(3u << (2 * pair_idx));                        // both CTAs of this pair
    const uint16_t cluster_mask = (uint16_t)((1u << CSIZE) - 1u);                       // every CTA of the cluster
    uint16_t parity_mask = 0;                                                            // this CTA's counterparts in all pairs
#pragma unroll
    for (int pp = 0; pp < CL; ++pp) parity_mask |= (uint16_t)(1u << (2 * pp + pair_cta));
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; ++i) {
            ptx::mbar_init(&aux->full[i], CG);      // one arrival per CTA of the pair (+ their TMA bytes)
            ptx::mbar_init(&aux->empty[i], CL);      // tcgen05.commit of every pair of the cluster (multicast to all its CTAs)
        }
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(&aux->tmem_full[i], 1);
            ptx::mbar_init(&aux->tmem_empty[i], NUM_EPI_THREADS * CG);   // both CTAs' epilogues (leader's copy)
            ptx::mbar_init(&aux->a_ready[i], 128);                       // CONV: the four converter warps
            ptx::mbar_init(&aux->a_free[i], NUM_EPI_THREADS);            // CONV: this CTA's epilogue threads
        }
        ptx::fence_barrier_init();
    }
    if (CG == 2) ptx::cluster_sync_all();            // peer barriers exist before anything signals them
    if (warp == 2) {
        if (CG == 2) ptx::tmem_alloc_2sm(&aux->tmem_base, TMEM_COLS);
        else ptx::tmem_alloc(&aux->tmem_base, TMEM_COLS);
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = aux->tmem_base;

    const int num_kb = (p.d + BLOCK_K - 1) / BLOCK_K;
    // work items are (column split, group of CG adjacent row tiles); a pair walks them together
    const int n_mgroups = (n_mtiles + GRP - 1) / GRP;
    const int total_work = n_mgroups * p.n_splits;
    const int w_begin = blockIdx.x / CSIZE, w_step = gridDim.x / CSIZE;
    // PA / PB are the plane SLOTS of a stage; whether a lo plane is really loaded and multiplied is a
    // run-time property of the data (prepare.cu sets meta[LO_NONZERO]), so callers never have to
    // synchronise with the host to find out that e.g. integer descriptors are exact in one plane.
    const bool use_alo = (PA == 2) && (__ldg(p.a_meta + META_LO_NONZERO) != 0.f);
    const bool use_blo = (PB == 2) && (__ldg(p.b_meta + META_LO_NONZERO) != 0.f);

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t it = 0, item = 0;
            const uint32_t tx_bytes = (ARES ? 0 : MT * A_TILE_BYTES * (1 + (int)use_alo)) + B_LOAD_BYTES * (1 + (int)use_blo);
            for (int w = w_begin; w < total_work; w += w_step, ++item) {
                const int split = w / n_mgroups, mt = (w - split * n_mgroups) * GRP + (int)cta_rank;
                if (CONV) {
                    // this item's planes have been written (generic proxy, this CTA) -- make them visible to the TMA reads
                    ptx::mbar_wait(&aux->a_ready[item & 1], (item >> 1) & 1);
                    asm volatile("fence.proxy.async;" ::: "memory");
                }
                const int nt0 = split * p.tiles_per_split;
                const int nt1 = min(nt0 + p.tiles_per_split, p.n_ntiles);
                // this work item's lock-step group: the items of the same split handled in the same round
                int32_t* cnt = nullptr;
                int gsize = 0;
                if (p.sync_cnt != nullptr && cta_rank == 0) {
                    const int round = (w - w_begin) / w_step;
                    const int g_lo = max(round * w_step, split * n_mgroups);
                    const int g_hi = min(min((round + 1) * w_step, (split + 1) * n_mgroups), total_work);
                    gsize = g_hi - g_lo;
                    if (gsize > 1) cnt = p.sync_cnt + ((int64_t)round * p.n_splits + split) * p.sync_ncp;
                }
                for (int nt = nt0; nt < nt1; ++nt) {
                    if (cnt != nullptr && (nt - nt0) % p.sync_every == 0) {
                        const int cp = (nt - nt0) / p.sync_every;
                        atomicAdd(cnt + cp, 1);
                        if (cp > 0) {
                            // wait until every member has at least STARTED the previous block of tiles; bounded, since
                            // this is a performance hint and co-residency of the group is not guaranteed
                            const volatile int32_t* prev = cnt + cp - 1;
                            for (int spin = 0; spin < 400 && *prev < gsize; ++spin) __nanosleep(100);
                        }
                    }
                    for (int kb = 0; kb < num_kb; ++kb, ++it) {
                        const int s = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        ptx::mbar_wait(&aux->empty[s], ph ^ 1);
                        uint8_t* st = smem + s * STAGE_BYTES;
                        // this CTA's half of the tile; of that, the 1 / CL it fetches itself
                        const int bcol = nt * BLOCK_N + (int)pair_cta * B_LOAD_ROWS + (int)pair_idx * B_ISSUE_ROWS;
                        const int b_sub = (int)pair_idx * B_ISSUE_BYTES;
                        if (ARES) {
                            // the item's row tile rides on its first stage: all k-blocks into this item's resident slot
                            const bool first = nt == nt0 && kb == 0;
                            const uint32_t tx = tx_bytes + (first ? (uint32_t)(num_kb * A_TILE_BYTES) : 0u);
                            uint8_t* slot = a_res + (item & 1) * (2 * A_TILE_BYTES);
                            if (CG == 1) {
                                ptx::mbar_arrive_expect_tx(&aux->full[s], tx);
                                if (first)
                                    for (int k2 = 0; k2 < num_kb; ++k2)
                                        ptx::tma_load_2d(slot + k2 * A_TILE_BYTES, &tm_a_hi, &aux->full[s], k2 * BLOCK_K, mt * BLOCK_M);
                                ptx::tma_load_2d(st, &tm_b_hi, &aux->full[s], kb * BLOCK_K, bcol);
                                if (use_blo) ptx::tma_load_2d(st + B_LOAD_BYTES, &tm_b_lo, &aux->full[s], kb * BLOCK_K, bcol);
                            } else {
                                if (leader) ptx::mbar_arrive_expect_tx(&aux->full[s], 2 * tx);
                                else ptx::mbar_arrive_remote(&aux->full[s], leader_rank);
                                if (first)
                                    for (int k2 = 0; k2 < num_kb; ++k2)
                                        ptx::tma_load_2d_2sm(slot + k2 * A_TILE_BYTES, &tm_a_hi, &aux->full[s], k2 * BLOCK_K, mt * BLOCK_M);
                                ptx::tma_load_2d_2sm(st, &tm_b_hi, &aux->full[s], kb * BLOCK_K, bcol);
                                if (use_blo) ptx::tma_load_2d_2sm(st + B_LOAD_BYTES, &tm_b_lo, &aux->full[s], kb * BLOCK_K, bcol);
                            }
                        } else if (CG == 1) {
                            ptx::mbar_arrive_expect_tx(&aux->full[s], tx_bytes);
#pragma unroll
                            for (int r = 0; r < MT; ++r) {      // rows past m are zero-filled by TMA
                                ptx::tma_load_2d(st + r * A_BLOCK_BYTES, &tm_a_hi, &aux->full[s], kb * BLOCK_K,
                                                 (mt + r) * BLOCK_M);
                                if (use_alo)
                                    ptx::tma_load_2d(st + r * A_BLOCK_BYTES + A_TILE_BYTES, &tm_a_lo, &aux->full[s],
                                                     kb * BLOCK_K, (mt + r) * BLOCK_M);
                            }
                            ptx::tma_load_2d(st + B_OFFSET, &tm_b_hi, &aux->full[s], kb * BLOCK_K, bcol);
                            if (use_blo)
                                ptx::tma_load_2d(st + B_OFFSET + B_LOAD_BYTES, &tm_b_lo, &aux->full[s],
                                                 kb * BLOCK_K, bcol);
                        } else {
                            // both CTAs' bytes are counted on the LEADER's barrier
                            if (leader) ptx::mbar_arrive_expect_tx(&aux->full[s], 2 * tx_bytes);
                            else ptx::mbar_arrive_remote(&aux->full[s], leader_rank);
                            ptx::tma_load_2d_2sm(st, &tm_a_hi, &aux->full[s], kb * BLOCK_K, mt * BLOCK_M);
                            if (use_alo)
                                ptx::tma_load_2d_2sm(st + A_TILE_BYTES, &tm_a_lo, &aux->full[s], kb * BLOCK_K,
                                                     mt * BLOCK_M);
                            if (CL == 1) {
                                ptx::tma_load_2d_2sm(st + PA * A_TILE_BYTES, &tm_b_hi, &aux->full[s], kb * BLOCK_K, bcol);
                                if (use_blo)
                                    ptx::tma_load_2d_2sm(st + PA * A_TILE_BYTES + B_LOAD_BYTES, &tm_b_lo, &aux->full[s],
                                                         kb * BLOCK_K, bcol);
                            } else {
                                ptx::tma_load_2d_2sm_mc(st + PA * A_TILE_BYTES + b_sub, &tm_b_hi, &aux->full[s], kb * BLOCK_K,
                                                        bcol, parity_mask);
                                if (use_blo)
                                    ptx::tma_load_2d_2sm_mc(st + PA * A_TILE_BYTES + B_LOAD_BYTES + b_sub, &tm_b_lo,
                                                            &aux->full[s], kb * BLOCK_K, bcol, parity_mask);
                            }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // the WHOLE warp walks the loops (uniform control flow and operands); one elected lane issues the MMAs / commits
        if (leader) {   // CG == 2: only the leader CTA of a pair issues MMAs
            constexpr uint32_t idesc = ptx::make_idesc_f16_f32(BLOCK_M * CG, BLOCK_N);
            const uint32_t smem_base = ptx::smem_u32(smem);
            uint32_t it = 0, tile = 0, item = 0;
            for (int w = w_begin; w < total_work; w += w_step, ++item) {
                const int split = w / n_mgroups;
                const int nt0 = split * p.tiles_per_split;
                const int nt1 = min(nt0 + p.tiles_per_split, p.n_ntiles);
                for (int nt = nt0; nt < nt1; ++nt, ++tile) {
                    // MT == 2: both accumulators belong to this column tile (no double buffering)
                    const int as = MT == 2 ? 0 : (tile & 1);
                    const uint32_t aph = MT == 2 ? (tile & 1) : ((tile >> 1) & 1);
                    ptx::mbar_wait(&aux->tmem_empty[as], aph ^ 1);
                    ptx::tc_fence_after();
                    const uint32_t tmem_d = tmem_base + as * BLOCK_N;
                    for (int kb = 0; kb < num_kb; ++kb, ++it) {
                        const int s = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        ptx::mbar_wait(&aux->full[s], ph);
                        ptx::tc_fence_after();
                        // descriptor low words (address >> 4): every operand offset is a multiple of 16 bytes and shared
                        // memory ends below 2^18, so the 14-bit field never carries
                        const uint32_t sb = (smem_base + s * STAGE_BYTES) >> 4;
                        const uint32_t a_hi0 = ARES ? (ptx::smem_u32(a_res) + (item & 1) * (2 * A_TILE_BYTES) + kb * A_TILE_BYTES) >> 4 : sb;
                        const uint32_t a_lo0 = sb + (A_TILE_BYTES >> 4);
                        const uint32_t b_hi0 = sb + (B_OFFSET >> 4), b_lo0 = b_hi0 + (B_LOAD_BYTES >> 4);
                        const uint32_t a1_hi0 = sb + (A_BLOCK_BYTES >> 4), a1_lo0 = a1_hi0 + (A_TILE_BYTES >> 4);   // MT == 2
                        const int rem = p.d - kb * BLOCK_K;
                        const int ksteps = rem >= BLOCK_K ? BLOCK_K / UMMA_K : (rem + UMMA_K - 1) / UMMA_K;
                        auto issue = [&](int ks) {
                            // advancing 16 fp16 = 32 bytes inside the 128B swizzle span: +2 in the >>4 address
                            const uint32_t koff = (uint32_t)(ks * ((UMMA_K * 2) >> 4));
                            const uint32_t acc = (uint32_t)((kb | ks) != 0);
                            if (CG == 1) {
                                ptx::umma_f16_ss_lo(tmem_d, a_hi0 + koff, b_hi0 + koff, idesc, acc);
                                if (use_blo) ptx::umma_f16_ss_lo(tmem_d, a_hi0 + koff, b_lo0 + koff, idesc, 1);
                                if (use_alo) ptx::umma_f16_ss_lo(tmem_d, a_lo0 + koff, b_hi0 + koff, idesc, 1);
                                if (MT == 2) {      // second row tile, accumulator in TMEM columns [256, 512)
                                    ptx::umma_f16_ss_lo(tmem_d + BLOCK_N, a1_hi0 + koff, b_hi0 + koff, idesc, acc);
                                    if (use_blo) ptx::umma_f16_ss_lo(tmem_d + BLOCK_N, a1_hi0 + koff, b_lo0 + koff, idesc, 1);
                                    if (use_alo) ptx::umma_f16_ss_lo(tmem_d + BLOCK_N, a1_lo0 + koff, b_hi0 + koff, idesc, 1);
                                }
                            } else {
                                ptx::umma_f16_ss_2sm_lo(tmem_d, a_hi0 + koff, b_hi0 + koff, idesc, acc);
                                if (use_blo) ptx::umma_f16_ss_2sm_lo(tmem_d, a_hi0 + koff, b_lo0 + koff, idesc, 1);
                                if (use_alo) ptx::umma_f16_ss_2sm_lo(tmem_d, a_lo0 + koff, b_hi0 + koff, idesc, 1);
                            }
                        };
                        const bool last_kb = kb == num_kb - 1;
                        if (ptx::elect_one()) {
                            if (ksteps == BLOCK_K / UMMA_K) {       // a full 64-column block: straight-line issue
#pragma unroll
                                for (int ks = 0; ks < BLOCK_K / UMMA_K; ++ks) issue(ks);
                            } else {
                                for (int ks = 0; ks < ksteps; ++ks) issue(ks);
                            }
                            // frees the smem stage (in both CTAs) when these MMAs retire
                            if (CG == 1) ptx::umma_commit(&aux->empty[s]);
                            else ptx::umma_commit_2sm(&aux->empty[s], CL == 1 ? pair_mask : cluster_mask);
                            if (last_kb) {      // accumulator complete -> epilogue (of both CTAs)
                                if (CG == 1) ptx::umma_commit(&aux->tmem_full[as]);
                                else ptx::umma_commit_2sm(&aux->tmem_full[as], pair_mask);
                            }
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + NUM_EPI_THREADS / 32) {
        // ===================== epilogue: selection =====================
        const int ew = warp - EPI_WARP0;
        const int q = ew & 3;      // TMEM lane quadrant this warp may read (== warp % 4)
        const int half = MT == 2 ? 0 : (ew >> 2);  // which half of every tile's columns this warp scans
        const int rt = MT == 2 ? (ew >> 2) : 0;    // MT == 2: which of the CTA's two row tiles this warp serves
        const int et = threadIdx.x - EPI_WARP0 * 32;
        const float b_inv = p.b_meta[META_INV_SCALE];
        const float a_inv_tensor = p.a_meta[META_INV_SCALE];
        CoarseBound bound;
        if (KSEL == 1 && VERIFY) bound.init(p.a_meta, p.b_meta, p.d, CONV);   // CONV: a tensor that is not exact in its hi plane is re-run as a whole
        uint32_t tile = 0, item = 0;
        for (int w = w_begin; w < total_work; w += w_step, ++item) {
            const int split = w / n_mgroups, mt = (w - split * n_mgroups) * GRP + (int)cta_rank + rt;
            const int nt0 = split * p.tiles_per_split;
            const int nt1 = min(nt0 + p.tiles_per_split, p.n_ntiles);
            const int row_in_tile = q * 32 + lane;
            const int64_t row = (int64_t)mt * BLOCK_M + row_in_tile;
            // CONV: this item's norms / per-row scales were written by the converter warps during this launch: wait for
            // them and read them with coherent loads (not the read-only path)
            if (CONV) ptx::mbar_wait(&aux->a_ready[item & 1], (item >> 1) & 1);
            // accumulator -> real units: 1 / (scale of this row's A planes * scale of the B planes)
            const float a_inv = (p.a_row_inv != nullptr && row < m_rows)
                                    ? (CONV ? __ldcg(p.a_row_inv + row) : __ldg(p.a_row_inv + row)) : a_inv_tensor;
            const float inv = a_inv * b_inv;
            const float two_inv = 2.f * inv;
            if (KSEL == 1 && VERIFY) bound.set_a_inv_scale(a_inv);

            // top-1 state: best score / id, the best score among the OTHER columns of the chunk that
            // holds the best (sib) and among all other chunks (m2): max(sib, m2) is the exact runner-up
            float best = -CUDART_INF_F, sib = -CUDART_INF_F, m2 = -CUDART_INF_F;
            int best_id = -1;
            typename SelList<KSEL>::type list;
            float collect_thr = CUDART_INF_F;   // collect mode: rows beyond m never append
            if (KSEL == 0) {
                if (row < m_rows) {
                    const float sr = __ldg(p.row_seed + row);
                    collect_thr = L2 ? (__ldg(p.a_norms + row) - sr) : sr / inv;   // scales are powers of two: exact
                }
            }
            if (KSEL > 1) {
                // seed = score of a column already known to exist (from a pre-pass over a column sample):
                // candidates that cannot beat it are never inserted, which removes almost all list traffic
                float seed = -CUDART_INF_F;
                if (p.row_seed != nullptr && row < m_rows) {
                    const float sr = __ldg(p.row_seed + row);
                    seed = L2 ? (__ldg(p.a_norms + row) - sr) : sr / inv;           // scales are powers of two: exact
                }
                list.init(p.topk, seed);
            }

            for (int nt = nt0; nt < nt1; ++nt, ++tile) {
                const int as = MT == 2 ? 0 : (tile & 1);
                const uint32_t aph = MT == 2 ? (tile & 1) : ((tile >> 1) & 1);
                const int col0 = nt * BLOCK_N;
                const int ncols = (int)min((int64_t)BLOCK_N, p.n - col0);
                if (L2) {
                    for (int c = et; c < BLOCK_N; c += NUM_EPI_THREADS)
                        aux->bnorm[tile & 1][c] = (c < ncols) ? __ldg(p.b_norms + col0 + c) : 0.f;
                    asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_THREADS) : "memory");
                }
                ptx::mbar_wait(&aux->tmem_full[as], aph);
                ptx::tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (MT == 2 ? rt : as) * BLOCK_N;
                const int c_begin = half * COLS_PER_HALF;
                const int c_end = min(c_begin + COLS_PER_HALF, ncols);
                // ROLLED loop over 32-column chunks: one copy of the scan / insertion code (I-cache)
                uint32_t r[32];
#pragma unroll 1
                for (int c = c_begin; c < c_end; c += 32) {
                    {
                        ptx::tmem_ld_32x32b_x32(taddr + c, r);
                        ptx::tmem_ld_wait();
                        float v[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            v[j] = __uint_as_float(r[j]);
                            // maximise 2<a,b> - |b|^2  ==  minimise |a|^2 + |b|^2 - 2<a,b>
                            if (L2) v[j] = fmaf(v[j], two_inv, -aux->bnorm[tile & 1][c + j]);
                        }
                        if (c + 32 > ncols) {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (c + j >= ncols) v[j] = -CUDART_INF_F;
                        }
                        // four groups of eight (3-input maxima), then the chunk maximum: the group maxima are what the
                        // rare top-1 update starts from
                        float g[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            g[i] = ptx::fmax3(ptx::fmax3(v[8 * i], v[8 * i + 1], v[8 * i + 2]),
                                              ptx::fmax3(v[8 * i + 3], v[8 * i + 4], v[8 * i + 5]), fmaxf(v[8 * i + 6], v[8 * i + 7]));
                        const float t01 = fmaxf(g[0], g[1]), t23 = fmaxf(g[2], g[3]);
                        const float mx = fmaxf(t01, t23);
                        if (KSEL == 0) {
                            float cur = mx;
#pragma unroll 1
                            while (cur > collect_thr) {
                                int jj = 31;
#pragma unroll
                                for (int j = 30; j >= 0; --j) jj = (v[j] == cur) ? j : jj;
                                const int pos = atomicAdd(p.row_count + row, 1);
                                if (pos < p.topk) {
                                    const float an_c = L2 ? __ldg(p.a_norms + row) : 0.f;
                                    p.out_val[row * p.topk + pos] = L2 ? fmaxf(an_c - cur, 0.f) : cur * inv;
                                    p.out_idx[row * p.topk + pos] = p.id_base + col0 + c + jj;
                                }
                                float nm = -CUDART_INF_F;
#pragma unroll
                                for (int j = 0; j < 32; ++j) {
                                    v[j] = (j == jj) ? -CUDART_INF_F : v[j];
                                    nm = fmaxf(nm, v[j]);
                                }
                                cur = nm;
                            }
                        } else if (KSEL == 1) {
                            if (mx > best) {  // strict: an equal score in a later column never replaces
                                // a warp takes this branch when ANY of its 32 rows improves (two thirds of the chunks of a
                                // 4096-column codebook), and the epilogue is bound by the half-rate ALU pipe (max / compare /
                                // select): the update is written for few ALU instructions
                                if constexpr (VERIFY) {
                                    // Position and runner-up from maxima over BIT PARTITIONS of the index: the maximum sits
                                    // where the partition maximum equals it, and the second largest value is the largest
                                    // min(side 0, side 1) over the bits (the top two differ in at least one bit).  A duplicated
                                    // maximum gives runner-up == maximum (and an arbitrary position): such a row is never
                                    // accepted by the proof, the split re-run decides it with the exact tie rule.
                                    m2 = fmaxf(m2, best);   // the old best's whole chunk is now "other"
                                    best = mx;
                                    const float u02 = fmaxf(g[0], g[2]), u13 = fmaxf(g[1], g[3]);
                                    const int gi = (t01 != mx ? 2 : 0) + (u02 != mx ? 1 : 0);
                                    const float sib_g = fmaxf(fminf(t01, t23), fminf(u02, u13));
                                    // the winning group's eight values (a trip through local memory instead of these 24
                                    // selects was measured slower: 1.46 vs 1.02 ms at the C2 shape)
                                    const bool ghi = t01 != mx, godd = u02 != mx;
                                    float w[8];
#pragma unroll
                                    for (int e = 0; e < 8; ++e) {
                                        const float lo = godd ? v[8 + e] : v[e], hi = godd ? v[24 + e] : v[16 + e];
                                        w[e] = ghi ? hi : lo;
                                    }
                                    float4 wa, wb;
                                    wa.x = w[0]; wa.y = w[1]; wa.z = w[2]; wa.w = w[3];
                                    wb.x = w[4]; wb.y = w[5]; wb.z = w[6]; wb.w = w[7];
                                    const float p01 = fmaxf(wa.x, wa.y), p23 = fmaxf(wa.z, wa.w);
                                    const float p45 = fmaxf(wb.x, wb.y), p67 = fmaxf(wb.z, wb.w);
                                    const float a2 = fmaxf(p01, p23), b2 = fmaxf(p45, p67);                 // bit 2: 0..3 | 4..7
                                    const float a1 = fmaxf(p01, p45), b1 = fmaxf(p23, p67);                 // bit 1
                                    const float a0 = ptx::fmax3(wa.x, wa.z, fmaxf(wb.x, wb.z));             // bit 0: even | odd
                                    const float b0 = ptx::fmax3(wa.y, wa.w, fmaxf(wb.y, wb.w));
                                    const int ee = (a2 != mx ? 4 : 0) + (a1 != mx ? 2 : 0) + (a0 != mx ? 1 : 0);
                                    sib = fmaxf(ptx::fmax3(fminf(a2, b2), fminf(a1, b1), fminf(a0, b0)), sib_g);
                                    best_id = col0 + c + gi * 8 + ee;
                                } else {
                                    best = mx;
                                    const bool in01 = (g[0] == mx) || (g[1] == mx);
                                    const bool odd = in01 ? (g[0] != mx) : (g[2] != mx);
                                    const int gi = (in01 ? 0 : 2) + (odd ? 1 : 0);
                                    float w[8];
#pragma unroll
                                    for (int e = 0; e < 8; ++e) {
                                        const float lo = odd ? v[8 + e] : v[e], hi = odd ? v[24 + e] : v[16 + e];
                                        w[e] = in01 ? lo : hi;
                                    }
                                    int ee = 7;
#pragma unroll
                                    for (int e = 6; e >= 0; --e)
                                        if (w[e] == mx) ee = e;  // lowest column among equals
                                    best_id = col0 + c + gi * 8 + ee;
                                }
                            } else if (VERIFY) {
                                m2 = fmaxf(m2, mx);
                            }
                        } else {
                            // rare path (a value beating the row's current threshold): extract the chunk's
                            // maxima one by one -- a single copy of the insertion code, lowest column first
                            // among equal values
                            float cur = mx;
#pragma unroll 1
                            while (cur > list.thr) {
                                int jj = 31;
#pragma unroll
                                for (int j = 30; j >= 0; --j) jj = (v[j] == cur) ? j : jj;
                                list.insert(cur, col0 + c + jj);
                                float nm = -CUDART_INF_F;
#pragma unroll
                                for (int j = 0; j < 32; ++j) {
                                    v[j] = (j == jj) ? -CUDART_INF_F : v[j];
                                    nm = fmaxf(nm, v[j]);
                                }
                                cur = nm;
                            }
                        }
                    }
                }
                ptx::tc_fence_before();
                // the MMA issuer (leader CTA) may overwrite this accumulator once every epilogue thread of
                // the pair has drained it
                if (CG == 1 || leader) ptx::mbar_arrive(&aux->tmem_empty[as]);
                else ptx::mbar_arrive_remote(&aux->tmem_empty[as], leader_rank);
            }

            if (KSEL == 1) {
                // combine the two column halves of this row (half 1 hands its state to half 0)
                float runner = fmaxf(sib, m2);
                if (HALVES > 1) {
                    if (half > 0) {
                        aux->xbest[half - 1][row_in_tile] = best;
                        aux->xrun[half - 1][row_in_tile] = runner;
                        aux->xid[half - 1][row_in_tile] = best_id;
                    }
                    asm volatile("bar.sync 2, %0;" ::"n"(NUM_EPI_THREADS) : "memory");
                    if (half == 0) {
#pragma unroll
                        for (int h = 0; h < HALVES - 1; ++h) {      // in column order: an equal score further right never wins
                            const float ob = aux->xbest[h][row_in_tile], orun = aux->xrun[h][row_in_tile];
                            const int oid = aux->xid[h][row_in_tile];
                            const bool other_wins = (oid >= 0) && (best_id < 0 || ob > best || (ob == best && oid < best_id));
                            runner = fmaxf(fmaxf(runner, orun), other_wins ? best : ob);
                            if (other_wins) { best = ob; best_id = oid; }
                        }
                    }
                    asm volatile("bar.sync 2, %0;" ::"n"(NUM_EPI_THREADS) : "memory");
                }
                if (half == 0 && row < m_rows) {
                    const float an = (L2 || VERIFY) ? (CONV ? __ldcg(p.a_norms + row) : __ldg(p.a_norms + row)) : 0.f;
                    const int64_t orow = p.row_map != nullptr ? (int64_t)__ldcg(p.row_map + row) : row;
                    float* ov = p.out_val + ((int64_t)split * p.m + orow) * p.topk;
                    int64_t* oi = p.out_idx + ((int64_t)split * p.m + orow) * p.topk;
                    if (best_id >= 0) {
                        ov[0] = L2 ? fmaxf(an - best, 0.f) : best * inv;
                        oi[0] = p.id_base + best_id;
                        if (VERIFY) {
                            // winner provably unique?  IP scores carry +-eps each, L2 scores (2<a,b> - |b|^2) +-2 eps
                            const float gap = L2 ? (best - runner) : (best - runner) * inv;
                            const float need = (L2 ? 4.f : 2.f) * bound.eps(an);
                            if (!(gap > need)) p.flag_rows[atomicAdd(p.flag_count, 1)] = (int32_t)row;
                        }
                    } else {
                        ov[0] = L2 ? 3.402823466e+38f : -3.402823466e+38f;
                        oi[0] = -1;
                    }
                }
            } else if (KSEL > 1 && row < m_rows) {
                const float an = L2 ? __ldg(p.a_norms + row) : 0.f;
                float* ov = p.out_val + ((int64_t)split * p.m + row) * p.topk;
                int64_t* oi = p.out_idx + ((int64_t)split * p.m + row) * p.topk;
                auto emit = [&](int j, float v, int id) {
                    if (id >= 0) {
                        ov[j] = L2 ? fmaxf(an - v, 0.f) : v * inv;
                        oi[j] = p.id_base + id;
                    } else {
                        ov[j] = L2 ? 3.402823466e+38f : -3.402823466e+38f;
                        oi[j] = -1;
                    }
                };
                if constexpr (KSEL == 32) {
                    list.drain_sorted(emit);
                } else {
#pragma unroll 1
                    for (int j = 0; j < p.topk; ++j) emit(j, list.v[j], list.id[j]);
                }
            }
            if (CONV) ptx::mbar_arrive(&aux->a_free[item & 1]);     // the converter may reuse this parity slot
        }
    } else if (CONV && warp >= EPI_WARP0 + NUM_EPI_THREADS / 32) {
        // ===================== converter: float32 rows -> FP16 planes of the item this CTA runs next =====================
        const int cw = warp - (EPI_WARP0 + NUM_EPI_THREADS / 32);   // 0..3: 32 rows of the 128-row tile each
        const int d4 = p.d >> 2, dp4 = (int)(p.lda_w >> 2);
        RowStats st;
        if (blockIdx.x == 0 && cw == 0 && lane == 0) { p.a_meta_w[META_SCALE] = 1.f; p.a_meta_w[META_INV_SCALE] = 1.f; }
        uint32_t item = 0;
        for (int w = w_begin; w < total_work; w += w_step, ++item) {
            const int split = w / n_mgroups, mt = (w - split * n_mgroups) * GRP + (int)cta_rank;
            ptx::mbar_wait(&aux->a_free[item & 1], ((item >> 1) & 1) ^ 1);
            const int64_t r_base = (int64_t)mt * BLOCK_M + cw * 32;
#pragma unroll 1
            for (int g = 0; g < 32; g += 4)
                if (r_base + g < p.m)
                    convert_row_group<4, 1>(p.a_raw, p.m, d4, dp4, p.lda_raw, p.a_hi_w, p.a_lo_w, p.lda_w, p.a_norms_w,
                                            p.a_row_inv_w, p.a_lo_skipped, r_base + g, lane, st);
            __threadfence();                                       // planes / norms / scales are in L2 ...
            asm volatile("fence.proxy.async;" ::: "memory");       // ... and ordered before the TMA (async proxy) reads
            ptx::mbar_arrive(&aux->a_ready[item & 1]);
        }
        commit_row_stats(st, p.a_meta_w, lane);
    }

    ptx::tc_fence_before();
    if (CG == 2) ptx::cluster_sync_all();   // neither CTA of a pair may retire while the other can still signal it
    else __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        if (CG == 2) ptx::tmem_dealloc_2sm(tmem_base, TMEM_COLS);
        else ptx::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------
// merge of g sorted lists per row: one warp per row, each lane owns lists lane, lane+32, ...
// ------------------------------------------------------------------------------------------
constexpr int MERGE_MAX_LISTS_PER_LANE = 8;

template <bool LARGEST>
__global__ void topk_merge_kernel(const float* __restrict__ vparts, const int64_t* __restrict__ iparts, int g,
                                  int64_t m, int topk, float* __restrict__ out_val, int64_t* __restrict__ out_idx) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= m) return;
    int ptr[MERGE_MAX_LISTS_PER_LANE];
#pragma unroll
    for (int t = 0; t < MERGE_MAX_LISTS_PER_LANE; ++t) ptr[t] = 0;
    const float worst = LARGEST ? -3.402823466e+38f : 3.402823466e+38f;
    for (int j = 0; j < topk; ++j) {
        float bv = worst;
        int64_t bi = -1;
        int bt = -1;
#pragma unroll
        for (int t = 0; t < MERGE_MAX_LISTS_PER_LANE; ++t) {
            const int l = lane + 32 * t;
            if (l < g && ptr[t] < topk) {
                const int64_t off = ((int64_t)l * m + row) * topk + ptr[t];
                const float cv = vparts[off];
                const int64_t ci = iparts[off];
                if (ci >= 0 && (bt < 0 || cand_better<LARGEST>(cv, ci, bv, bi))) {
                    bv = cv; bi = ci; bt = t;
                }
            }
        }
        // warp arg-best on (value, id)
        float wv = bv;
        int64_t wi = bi;
        int wl = bt >= 0 ? lane : -1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, wv, o);
            const int64_t oi = __shfl_xor_sync(0xffffffffu, wi, o);
            const int ol = __shfl_xor_sync(0xffffffffu, wl, o);
            const bool take = (ol >= 0) && (wl < 0 || cand_better<LARGEST>(ov, oi, wv, wi));
            if (take) { wv = ov; wi = oi; wl = ol; }
        }
        if (wl == lane && bt >= 0) {
#pragma unroll
            for (int t = 0; t < MERGE_MAX_LISTS_PER_LANE; ++t)
                if (t == bt) ptr[t]++;
        }
        if (lane == 0) {
            out_val[row * topk + j] = (wl >= 0) ? wv : worst;
            out_idx[row * topk + j] = (wl >= 0) ? wi : -1;
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_plane_map(const ise_ctx* ctx, CUtensorMap* map, const void* base, int64_t rows, int d, int64_t ld,
                          int box_rows) {
    EncodeTiledFn fn = (EncodeTiledFn)ctx->encode_tiled;
    cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        ise_set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
        return 1;
    }
    return 0;
}

struct Plan {
    int n_mtiles, n_ntiles, tiles_per_split, n_splits;
};

// CTA pairs (cta_group::2) for the SPLIT products when there are at least two pairs' worth of row tiles.
// Measured on the B200 (profiles/r01_findings.md section 7): with the lo planes in play a stage is 48-64 KB per
// CTA and carries 8-12 MMAs, and pairs win 4-6 % (C2 assign 1.36 vs 1.41 ms, C3 split top-1 92 vs 98 ms);
// for the coarse pass (hi planes only, 4 MMAs per 32 KB stage) the cross-CTA signalling round trip is
// exposed and pairs lose 3-20 %, so the coarse top-1 pass stays single-CTA.
// Coarse top-k / collect passes at large d: with the soft lock-step keeping the column range in L2, halving the
// B bytes per MMA cycle pays (C3 seeded top-32 35.5 -> 33.0 ms), so they use pairs too.
static int pick_cg(int64_t m, bool split_products, int d, int topk) {
    const bool pairs = split_products || (topk != 1 && d >= 1024);
    return (pairs && ceil_div64(m, BLOCK_M) >= 4) ? 2 : 1;
}

// Two row tiles per CTA (MT = 2) for the coarse TOP-1 pass (hi planes only) when the MMAs of a tile pair outlast its
// epilogue by a wide margin (d >= 1024: >= 16 k MMA cycles against ~2 k of scan) and there are enough row tiles to go
// round: C3-shaped top-1 30.9 vs 35.5 ms.  The top-k list epilogues lose with it (seeded top-32 40.8 vs 35.4 ms,
// profiles/r01_findings.md section 13), so they keep one row tile and double-buffered accumulators.
static int pick_mt(int64_t m, int d, bool split_products, int topk) {
    return (!split_products && topk == 1 && d >= 1024 && ceil_div64(m, BLOCK_M) >= 2) ? 2 : 1;
}

// The launch variant (CTAs per MMA, row tiles per CTA) is decided in ONE place: the tensor maps (B box height), the
// work plan and the kernel instantiation must agree, or a TMA box delivers fewer bytes than the barrier expects.
struct Variant {
    int cg, mt, cl;
};
// Pairs per multicast cluster (CL) for the coarse top-k / collect pass at large d, where CTA pairs are used and the pass
// is bound by the L2 -> shared-memory feed: 2 pairs (clusters of 4 CTAs) when there are enough row tiles.
// Measured on the C3 coarse pass (10 k x 1 M x 2048, ncu, profiles/r02_findings.md): clusters of 2 pairs read 11.7 GB
// from DRAM instead of 31.9 GB (L2 traffic 263 vs 380 GB) in the same 30.8 ms; 4 pairs 7.0 GB but 3 % slower (only 15
// clusters of 8 whole-SM CTAs are co-resident: 120 of 148 SMs).  Small column sets (the 1/64 sample pre-pass) keep plain
// pairs: nothing to share, and the cluster-wide stage hand-shake costs.
static int pick_cl(int64_t m, int64_t n, int d, bool split_products, int topk, int cg) {
    if (cg != 2 || split_products || topk == 1) return 1;
    if (n * (int64_t)d * 2 < (256ll << 20)) return 1;                    // B plane below 256 MB
    return ceil_div64(m, BLOCK_M) >= 2 * 2 * 2 ? 2 : 1;                  // at least two clusters' worth of row tiles
}
static Variant pick_variant(int64_t m, int64_t n, int d, bool split_products, int topk) {
    Variant v;
    v.mt = pick_mt(m, d, split_products, topk);
    v.cg = v.mt == 2 ? 1 : pick_cg(m, split_products, d, topk);
    v.cl = pick_cl(m, n, d, split_products, topk, v.cg);
    return v;
}

// co-resident clusters of `csize` (1, 2 or 4) whole-SM CTAs (clusters of 4 do not tile every GPC: 33 on the B200
// instead of 37); the answer is the same for every gemm_select instantiation (one CTA per SM), so one of them is asked
// once
static int cluster_slots(const ise_ctx* ctx, int csize) {
    if (csize <= 2) return std::max(1, ctx->sm_count / csize);
    static int cached = 0;
    if (cached == 0) {
        int got = 0;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(csize * (ctx->sm_count / csize)));
        cfg.blockDim = dim3((unsigned)num_threads());
        cfg.dynamicSmemBytes = (size_t)(num_stages(1, 1, 2) * stage_bytes(1, 1, 2) + AUX_BYTES + 1024);
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = csize; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        auto kern = gemm_select_kernel<1, 1, false, 32, false, 2, 1, false, 2>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.dynamicSmemBytes);
        cudaOccupancyMaxActiveClusters(&got, kern, &cfg);
        cached = got > 0 ? got : std::max(1, ctx->sm_count / csize);
    }
    return cached;
}

static Plan make_plan(const ise_ctx* ctx, int64_t m, int64_t n, int d, int topk, bool single_split = false,
                      bool split_products = false) {
    Plan pl;
    pl.n_mtiles = (int)ceil_div64(m, BLOCK_M);
    pl.n_ntiles = (int)std::max<int64_t>(1, ceil_div64(n, BLOCK_N));
    const Variant var = pick_variant(m, n, d, split_products, topk);
    const int cg = var.cg * var.cl;                      // CTAs that walk a work item together (pair / cluster)
    const int grp = var.cg * var.mt * var.cl;
    const int groups = (pl.n_mtiles + grp - 1) / grp;    // work is scheduled per CTA pair (cluster) / per two-tile CTA
    const int slots = cluster_slots(ctx, cg);
    // enough work items for ~4 waves of the persistent grid, but never less than 8 column tiles per
    // item (a fresh item restarts its selection threshold) and at most 256 partial lists per row
    int64_t want = ceil_div64((int64_t)4 * slots, std::max(1, groups));
    int64_t max_by_tiles = std::max<int64_t>(1, pl.n_ntiles / 8);
    int64_t s_hi = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(2 * want, max_by_tiles), 256));
    if (single_split) s_hi = 1;  // top-1 verification keeps one runner-up per row, so columns are not split
    // pick the split count with the smallest makespan = waves x column tiles per item
    int64_t best_s = 1, best_cost = -1;
    for (int64_t s = 1; s <= s_hi; ++s) {
        const int64_t tps = ceil_div64(pl.n_ntiles, s);
        const int64_t ns = ceil_div64(pl.n_ntiles, tps);
        const int64_t waves = ceil_div64((int64_t)groups * ns, slots);
        const int64_t cost = waves * tps;
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_s = ns; }
    }
    pl.tiles_per_split = (int)ceil_div64(pl.n_ntiles, best_s);
    pl.n_splits = (int)ceil_div64(pl.n_ntiles, pl.tiles_per_split);
    return pl;
}


// soft lock-step set-up: worth it only when one work item streams more B than a slice of L2 can keep around for the
// slowest CTA of its group
static void setup_sync(const ise_ctx* ctx, Params& p, int d, bool split_products, int cg, int mt, cudaStream_t st) {
    p.sync_cnt = nullptr;
    p.sync_every = 0;
    p.sync_ncp = 0;
    if (!ctx->sync_buf) return;
    const int64_t tile_bytes = (int64_t)BLOCK_N * ((d + BLOCK_K - 1) / BLOCK_K * BLOCK_K) * 2 * (split_products ? 2 : 1);
    if (tile_bytes * p.tiles_per_split < (24ll << 20)) return;
    const int every = (int)std::max<int64_t>(1, (16ll << 20) / tile_bytes);         // ~16 MB of B between check-ins
    const int ncp = (p.tiles_per_split + every - 1) / every;
    const int grp = cg * mt;
    const int n_mgroups = (p.n_mtiles + grp - 1) / grp;
    const int64_t total = (int64_t)n_mgroups * p.n_splits;
    const int slots = cluster_slots(ctx, cg);
    const int64_t rounds = ceil_div64(total, std::min<int64_t>(total, slots));
    const int64_t ints = rounds * p.n_splits * ncp;
    if (ints > kSyncInts) return;
    if (cudaMemsetAsync(ctx->sync_buf, 0, (size_t)ints * sizeof(int32_t), st) != cudaSuccess) return;
    p.sync_cnt = ctx->sync_buf;
    p.sync_every = every;
    p.sync_ncp = ncp;
}

template <int PA, int PB, bool L2, int KSEL, bool VERIFY, int CG, int MT = 1, bool CONV = false, int CL = 1, bool ARES = false>
static int launch_cg(const ise_ctx* ctx, const CUtensorMap* maps, const Params& p, cudaStream_t st) {
    auto kern = gemm_select_kernel<PA, PB, L2, KSEL, VERIFY, CG, MT, CONV, CL, ARES>;
    const int smem = (ARES ? ares_bytes() + ares_stages(PB, CG) * ares_stage_bytes(PB, CG)
                           : num_stages(PA, PB, CG, MT) * stage_bytes(PA, PB, CG, MT)) + AUX_BYTES + 1024;
    ISE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    constexpr int CSIZE = CG * CL;
    const int groups = (p.n_mtiles + CSIZE * MT - 1) / (CSIZE * MT);
    const int total = groups * p.n_splits;
    Params pp = p;
    setup_sync(ctx, pp, p.d, PB == 2, CSIZE, MT, st);
    int slots = std::max(1, ctx->sm_count / CSIZE);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(CSIZE * slots));
    cfg.blockDim = dim3((unsigned)num_threads(MT, CONV, ARES));
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;   // CG == 2: the two CTAs of a pair form a cluster
    attr[0].val.clusterDim.x = CG * CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    slots = cluster_slots(ctx, CSIZE);
    const int grid = CSIZE * std::min(total, slots);
    cfg.gridDim = dim3((unsigned)grid);
    ISE_CUDA(cudaLaunchKernelEx(&cfg, kern, maps[0], maps[1], maps[2], maps[3], pp));
    return 0;
}

template <int PA, int PB, bool L2, int KSEL, bool VERIFY = false>
static int launch(const ise_ctx* ctx, const CUtensorMap* maps, const Params& p, cudaStream_t st) {
    const Variant var = pick_variant(p.m, p.n, p.d, PB == 2, KSEL == 1 ? 1 : 0);
    if constexpr (KSEL == 1 && PA == 1 && PB == 1) {        // coarse top-1: single CTAs, one or two row tiles each
        if (var.cg != 1) ISE_FAIL("internal: CTA pairs picked for the coarse top-1 pass");
        return var.mt == 2 ? launch_cg<PA, PB, L2, KSEL, VERIFY, 1, 2>(ctx, maps, p, st)
                           : launch_cg<PA, PB, L2, KSEL, VERIFY, 1>(ctx, maps, p, st);
    } else {
        if (var.mt != 1) ISE_FAIL("internal: two-row-tile variant picked for a kernel that has none");
        if constexpr (PA == 1 && PB == 1) {       // coarse top-k / collect: multicast clusters of CTA pairs
            if (var.cg == 2 && var.cl == 2) return launch_cg<PA, PB, L2, KSEL, VERIFY, 2, 1, false, 2>(ctx, maps, p, st);
        }
        if (var.cl != 1) ISE_FAIL("internal: multicast cluster picked for a kernel that has none");
        return var.cg == 2 ? launch_cg<PA, PB, L2, KSEL, VERIFY, 2>(ctx, maps, p, st)
                           : launch_cg<PA, PB, L2, KSEL, VERIFY, 1>(ctx, maps, p, st);
    }
}

template <int PA, int PB, bool L2>
static int dispatch_k(const ise_ctx* ctx, const CUtensorMap* maps, const Params& p, cudaStream_t st) {
    if (p.topk == 1) {
        if (p.flag_count != nullptr) {
            if constexpr (PA == 1 && PB == 1) return launch<PA, PB, L2, 1, true>(ctx, maps, p, st);
            ISE_FAIL("top-1 verification is a coarse-pass feature: call with a_lo = b_lo = NULL");
        }
        return launch<PA, PB, L2, 1>(ctx, maps, p, st);
    }
    if (p.topk <= 32) return launch<PA, PB, L2, 32>(ctx, maps, p, st);
    return launch<PA, PB, L2, 128>(ctx, maps, p, st);
}

template <int PA, int PB>
static int dispatch_metric(const ise_ctx* ctx, const CUtensorMap* maps, const Params& p, int metric,
                           cudaStream_t st) {
    return metric == ISE_METRIC_L2 ? dispatch_k<PA, PB, true>(ctx, maps, p, st)
                                   : dispatch_k<PA, PB, false>(ctx, maps, p, st);
}

// the parameters of a plain launch under plan `pl`: every field not set here (the optional inputs and outputs, the
// fused-conversion operand, the verified-pipeline controls) starts zero / null
static Params make_params(const Plan& pl, int64_t m, int64_t n, int d, int topk, int64_t id_base, const float* a_meta,
                          const float* a_norms, const float* a_row_inv, const float* b_meta, const float* b_norms,
                          float* out_val, int64_t* out_idx) {
    Params p{};
    p.m = m; p.n = n; p.d = d;
    p.n_mtiles = pl.n_mtiles; p.n_ntiles = pl.n_ntiles;
    p.tiles_per_split = pl.tiles_per_split; p.n_splits = pl.n_splits;
    p.topk = topk; p.id_base = id_base;
    p.a_meta = a_meta; p.a_norms = a_norms; p.a_row_inv = a_row_inv; p.b_meta = b_meta; p.b_norms = b_norms;
    p.out_val = out_val; p.out_idx = out_idx;
    return p;
}

}  // namespace gs

ISE_EXPORT size_t ise_gemm_select_workspace_bytes(ise_ctx* ctx, int64_t m, int64_t n, int d, int topk) {
    if (!ctx || m <= 0 || topk <= 0) return 0;
    // the split count depends on whether the call will run CTA pairs (lo planes present): size for the larger
    const int ns = std::max(gs::make_plan(ctx, m, n, d, topk, false, false).n_splits, gs::make_plan(ctx, m, n, d, topk, false, true).n_splits);
    if (ns <= 1) return 0;
    return (size_t)ns * (size_t)m * (size_t)topk * (sizeof(float) + sizeof(int64_t)) + 256;
}

ISE_EXPORT int ise_topk_merge(ise_ctx* ctx, const float* val_parts, const int64_t* idx_parts, int g, int64_t m,
                              int topk, int metric, float* out_val, int64_t* out_idx, void* stream) {
    ISE_CHECK_ARG(ctx && g >= 1 && g <= 32 * gs::MERGE_MAX_LISTS_PER_LANE && m >= 0 && topk >= 1);
    if (m == 0) return 0;
    ISE_CHECK_ARG(val_parts && idx_parts && out_val && out_idx);
    DeviceGuard guard(ctx->device);
    const int warps = 8;
    const int grid = (int)ceil_div64(m, warps);
    if (metric == ISE_METRIC_IP)
        gs::topk_merge_kernel<true><<<grid, warps * 32, 0, (cudaStream_t)stream>>>(val_parts, idx_parts, g, m, topk,
                                                                                  out_val, out_idx);
    else
        gs::topk_merge_kernel<false><<<grid, warps * 32, 0, (cudaStream_t)stream>>>(val_parts, idx_parts, g, m, topk,
                                                                                   out_val, out_idx);
    ISE_LAUNCH_CHECK();
    return 0;
}

// shared argument validation + tensor maps
static int setup_maps_var(ise_ctx* ctx, const void* a_hi, const void* a_lo, int64_t lda, const void* b_hi,
                          const void* b_lo, int64_t ldb, int64_t m, int64_t n, int d, gs::Variant var, CUtensorMap* maps);

static int setup_maps(ise_ctx* ctx, const void* a_hi, const void* a_lo, int64_t lda, const void* b_hi,
                      const void* b_lo, int64_t ldb, int64_t m, int64_t n, int d, int topk, CUtensorMap* maps) {
    return setup_maps_var(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, m, n, d, gs::pick_variant(m, n, d, b_lo != nullptr, topk), maps);
}

static int setup_maps_var(ise_ctx* ctx, const void* a_hi, const void* a_lo, int64_t lda, const void* b_hi,
                          const void* b_lo, int64_t ldb, int64_t m, int64_t n, int d, gs::Variant var, CUtensorMap* maps) {
    const int b_box = gs::BLOCK_N / (var.cg * var.cl);   // a CTA of a pair stages half of every B tile (and fetches 1 / CL of that itself)
    ISE_CHECK_ARG(lda >= d && ldb >= d && lda % 8 == 0 && ldb % 8 == 0);
    ISE_CHECK_ARG((reinterpret_cast<uintptr_t>(a_hi) & 15) == 0 && (reinterpret_cast<uintptr_t>(b_hi) & 15) == 0);
    if (gs::make_plane_map(ctx, &maps[0], a_hi, m, d, lda, gs::BLOCK_M)) return 1;
    if (gs::make_plane_map(ctx, &maps[1], a_lo ? a_lo : a_hi, m, d, lda, gs::BLOCK_M)) return 1;
    if (gs::make_plane_map(ctx, &maps[2], b_hi, n, d, ldb, b_box)) return 1;
    if (gs::make_plane_map(ctx, &maps[3], b_lo ? b_lo : b_hi, n, d, ldb, b_box)) return 1;
    return 0;
}

ISE_EXPORT int ise_gemm_collect(ise_ctx* ctx, const void* a_hi, const void* a_lo, int64_t lda, const float* a_meta,
                                const float* a_norms, const float* a_row_inv, const void* b_hi, const void* b_lo, int64_t ldb,
                                const float* b_meta, const float* b_norms, int64_t m, int64_t n, int d, int metric,
                                int64_t id_base, const float* row_seed, int cap, float* cand_val, int64_t* cand_idx,
                                int32_t* row_count, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(m >= 0 && n > 0 && d > 0 && cap >= 1 && n < (int64_t)1 << 31 && m < (int64_t)1 << 31);
    if (m == 0) return 0;
    ISE_CHECK_ARG(a_hi && b_hi && a_meta && b_meta && row_seed && cand_val && cand_idx && row_count);
    if (metric == ISE_METRIC_L2) ISE_CHECK_ARG(a_norms && b_norms);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const gs::Plan pl = gs::make_plan(ctx, m, n, d, 0, false, b_lo != nullptr);
    gs::Params p = gs::make_params(pl, m, n, d, cap, id_base, a_meta, a_norms, a_row_inv, b_meta, b_norms, cand_val, cand_idx);
    p.row_seed = row_seed; p.row_count = row_count;
    // empty slots read as id -1 / count 0
    ISE_CUDA(cudaMemsetAsync(cand_idx, 0xFF, (size_t)m * cap * sizeof(int64_t), st));
    ISE_CUDA(cudaMemsetAsync(row_count, 0, (size_t)m * sizeof(int32_t), st));
    CUtensorMap maps[4];
    if (setup_maps(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, m, n, d, 0, maps)) return 1;
    const int pa = a_lo ? 2 : 1, pb = b_lo ? 2 : 1;
    const bool l2 = metric == ISE_METRIC_L2;
    if (pa == 1 && pb == 1) return l2 ? gs::launch<1, 1, true, 0>(ctx, maps, p, st) : gs::launch<1, 1, false, 0>(ctx, maps, p, st);
    if (pa == 1 && pb == 2) return l2 ? gs::launch<1, 2, true, 0>(ctx, maps, p, st) : gs::launch<1, 2, false, 0>(ctx, maps, p, st);
    if (pa == 2 && pb == 2) return l2 ? gs::launch<2, 2, true, 0>(ctx, maps, p, st) : gs::launch<2, 2, false, 0>(ctx, maps, p, st);
    ISE_FAIL("a_lo without b_lo is not supported: pass a zero b_lo plane");
}

static int gemm_select_impl(ise_ctx* ctx, const void* a_hi, const void* a_lo, int64_t lda, const float* a_meta,
                            const float* a_norms, const float* a_row_inv, const void* b_hi, const void* b_lo, int64_t ldb,
                            const float* b_meta, const float* b_norms, int64_t m, int64_t n, int d, int metric,
                            int topk, int64_t id_base, const float* row_seed, int32_t* flag_rows,
                            int32_t* flag_count, float* out_val, int64_t* out_idx, void* workspace,
                            size_t workspace_bytes, void* stream, int skip_if_a_exact) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(m >= 0 && n >= 0 && d > 0 && topk >= 1 && topk <= 128);
    ISE_CHECK_ARG(n < (int64_t)1 << 31 && m < (int64_t)1 << 31);
    if (m == 0) return 0;
    ISE_CHECK_ARG(a_hi && b_hi && a_meta && b_meta && out_val && out_idx);
    ISE_CHECK_ARG(lda >= d && ldb >= d && lda % 8 == 0 && ldb % 8 == 0);
    ISE_CHECK_ARG((reinterpret_cast<uintptr_t>(a_hi) & 15) == 0 && (reinterpret_cast<uintptr_t>(b_hi) & 15) == 0);
    if (metric == ISE_METRIC_L2) ISE_CHECK_ARG(a_norms && b_norms);
    if (row_seed) ISE_CHECK_ARG(topk > 1);
    ISE_CHECK_ARG(n > 0);  // an empty index is handled by the caller (Faiss pads with -1)
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;

    const gs::Plan pl = gs::make_plan(ctx, m, n, d, topk, flag_count != nullptr, b_lo != nullptr);
    gs::Params p = gs::make_params(pl, m, n, d, topk, id_base, a_meta, a_norms, a_row_inv, b_meta, b_norms, out_val, out_idx);
    p.skip_if_a_exact = skip_if_a_exact;
    p.row_seed = row_seed;
    p.flag_rows = flag_rows;
    p.flag_count = flag_count;
    if (flag_count) {
        ISE_CHECK_ARG(flag_rows && topk == 1 && a_norms);
        ISE_CUDA(cudaMemsetAsync(flag_count, 0, sizeof(int32_t), st));
    }
    float* wv = nullptr;
    int64_t* wi = nullptr;
    if (pl.n_splits > 1) {
        const size_t need = (size_t)pl.n_splits * (size_t)m * (size_t)topk * (sizeof(float) + sizeof(int64_t)) + 256;
        if (!workspace || workspace_bytes < need) ISE_FAIL("workspace too small: need " + std::to_string(need));
        const size_t cnt = (size_t)pl.n_splits * (size_t)m * (size_t)topk;
        wi = reinterpret_cast<int64_t*>(workspace);  // int64 first keeps both arrays aligned
        wv = reinterpret_cast<float*>(wi + cnt);
        p.out_val = wv; p.out_idx = wi;
    }

    const int pa = a_lo ? 2 : 1, pb = b_lo ? 2 : 1;
    CUtensorMap maps[4];
    if (setup_maps(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, m, n, d, topk, maps)) return 1;

    int rc;
    if (pa == 1 && pb == 1) rc = gs::dispatch_metric<1, 1>(ctx, maps, p, metric, st);
    else if (pa == 1 && pb == 2) rc = gs::dispatch_metric<1, 2>(ctx, maps, p, metric, st);
    else if (pa == 2 && pb == 2) rc = gs::dispatch_metric<2, 2>(ctx, maps, p, metric, st);
    else ISE_FAIL("a_lo without b_lo is not supported: pass a zero b_lo plane");
    if (rc) return rc;
    if (pl.n_splits > 1)
        return ise_topk_merge(ctx, wv, wi, pl.n_splits, m, topk, metric, out_val, out_idx, stream);
    return 0;
}

ISE_EXPORT int ise_gemm_select(ise_ctx* ctx, const void* a_hi, const void* a_lo, int64_t lda, const float* a_meta,
                               const float* a_norms, const float* a_row_inv, const void* b_hi, const void* b_lo, int64_t ldb,
                               const float* b_meta, const float* b_norms, int64_t m, int64_t n, int d, int metric,
                               int topk, int64_t id_base, const float* row_seed, int32_t* flag_rows,
                               int32_t* flag_count, float* out_val, int64_t* out_idx, void* workspace,
                               size_t workspace_bytes, void* stream) {
    return gemm_select_impl(ctx, a_hi, a_lo, lda, a_meta, a_norms, a_row_inv, b_hi, b_lo, ldb, b_meta, b_norms, m, n, d,
                            metric, topk, id_base, row_seed, flag_rows, flag_count, out_val, out_idx, workspace,
                            workspace_bytes, stream, 0);
}

int ise_internal_lo_fixup(ise_ctx* ctx, void* lo, int64_t n, int64_t ldp, const uint8_t* lo_skipped, const float* meta,
                          void* stream);   // prepare.cu

// ------------------------------------------------------------------------------------------
// verified top-1 at d <= 128 without a host round trip (quantisation / k-means assign)
// ------------------------------------------------------------------------------------------
namespace gs {

// compacts the hi (/ lo) plane rows, norms and scales of the flagged rows; block 0 publishes the row count of the
// re-run and whether the list overflowed its capacity
__global__ void gather_flagged_kernel(const int32_t* __restrict__ flag_rows, const int32_t* __restrict__ flag_count, int cap,
                                      const __half* __restrict__ a_hi, const __half* __restrict__ a_lo, int64_t lda,
                                      const float* __restrict__ norms, const float* __restrict__ row_inv,
                                      __half* __restrict__ g_hi, __half* __restrict__ g_lo, float* __restrict__ g_norms,
                                      float* __restrict__ g_row_inv, int32_t* __restrict__ m_dev, int32_t* __restrict__ overflow) {
    const int cnt = *flag_count;
    const int n = min(cnt, cap);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        *m_dev = n;
        *overflow = cnt > cap ? 1 : 0;
    }
    const int vecs = (int)(lda >> 3);                 // 8 halves per 16-byte vector (lda % 8 == 0)
    // one row per group of `vecs` (<= 16) consecutive threads, grid-stride
    const int per_block = blockDim.x / vecs;
    const int sub = threadIdx.x / vecs, c = threadIdx.x - sub * vecs;
    if (sub >= per_block) return;
    for (int64_t r = (int64_t)blockIdx.x * per_block + sub; r < n; r += (int64_t)gridDim.x * per_block) {
        const int64_t src = flag_rows[r];
        reinterpret_cast<uint4*>(g_hi + r * lda)[c] = __ldg(reinterpret_cast<const uint4*>(a_hi + src * lda) + c);
        if (a_lo != nullptr) reinterpret_cast<uint4*>(g_lo + r * lda)[c] = __ldg(reinterpret_cast<const uint4*>(a_lo + src * lda) + c);
        if (c == 0) {
            g_norms[r] = norms[src];
            if (row_inv != nullptr) g_row_inv[r] = row_inv[src];
        }
    }
}

struct VerifiedWs {
    int32_t* ctrl;        // [0] flagged rows, [1] rows of the re-run, [2] overflow
    int32_t* flag_rows;   // [m]
    __half* g_hi;
    __half* g_lo;
    float* g_norms;
    float* g_row_inv;
    int64_t cap;
    size_t bytes;
};

static VerifiedWs verified_ws(void* base, int64_t m, int64_t lda) {
    VerifiedWs w;
    // a quarter of the rows may be re-run through the compact path; beyond that the whole launch is repeated
    w.cap = std::min<int64_t>(ceil_div64(m, BLOCK_M) * BLOCK_M, ceil_div64(std::max<int64_t>(m / 4, 1024), BLOCK_M) * BLOCK_M);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return (uint8_t*)base + o; };
    w.ctrl = (int32_t*)take(16);
    w.flag_rows = (int32_t*)take((size_t)m * 4);
    w.g_hi = (__half*)take((size_t)w.cap * lda * 2);
    w.g_lo = (__half*)take((size_t)w.cap * lda * 2);
    w.g_norms = (float*)take((size_t)w.cap * 4);
    w.g_row_inv = (float*)take((size_t)w.cap * 4);
    w.bytes = off;
    return w;
}

// covered: up to two 64-column k-blocks (the resident row tile), enough column tiles to cycle the stage ring within an
// item, and enough row tiles that one unsplit column range fills the machine
static bool verified_covers(const ise_ctx* ctx, int64_t m, int64_t n, int d, int64_t lda) {
    const int num_kb = (d + BLOCK_K - 1) / BLOCK_K;
    if (d > 128 || lda > 128 || n < 2) return false;
    if (ceil_div64(n, BLOCK_N) * num_kb < 8) return false;
    if (m < (int64_t)2 * BLOCK_M * ctx->sm_count) return false;
    return make_plan(ctx, m, n, d, 1, false, true).n_splits == 1;
}

template <bool L2>
static int verified_launches(ise_ctx* ctx, Params p, const float* x, int64_t ldx, void* a_hi, void* a_lo, int64_t lda,
                             uint8_t* a_lo_skipped, float* a_meta_w, const void* b_hi, const void* b_lo, int64_t ldb,
                             const VerifiedWs& w, cudaStream_t st) {
    const int64_t m = p.m, n = p.n;
    const int d = p.d;
    const bool conv = x != nullptr;
    const bool rerun_lo = !conv && a_lo != nullptr;          // prepared rows that may carry a lo plane
    const float* a_norms = p.a_norms;
    const float* a_row_inv = p.a_row_inv;
    ISE_CUDA(cudaMemsetAsync(w.ctrl, 0, 16, st));
    CUtensorMap maps[4];
    Variant pair; pair.cg = 2; pair.mt = 1; pair.cl = 1;   // every launch of the pipeline runs CTA pairs
    // ---- 1. one product per tile, exact runner-up, rows that are not provably decided are listed
    {
        if (setup_maps_var(ctx, a_hi, nullptr, lda, b_hi, nullptr, ldb, m, n, d, pair, maps)) return 1;
        Params q = p;
        q.flag_rows = w.flag_rows; q.flag_count = w.ctrl;
        if (conv) {
            q.a_raw = x; q.lda_raw = ldx; q.a_hi_w = (__half*)a_hi; q.a_lo_w = (__half*)a_lo; q.lda_w = lda;
            q.a_norms_w = const_cast<float*>(a_norms); q.a_row_inv_w = const_cast<float*>(a_row_inv);
            q.a_lo_skipped = a_lo_skipped; q.a_meta_w = a_meta_w;
        }
        const int rc = conv ? launch_cg<1, 1, L2, 1, true, 2, 1, true, 1, true>(ctx, maps, q, st)
                            : launch_cg<1, 1, L2, 1, true, 2, 1, false, 1, true>(ctx, maps, q, st);
        if (rc) return rc;
    }
    // ---- 2. compact the listed rows
    {
        gather_flagged_kernel<<<(unsigned)(4 * ctx->sm_count), 256, 0, st>>>(
            w.flag_rows, w.ctrl, (int)w.cap, (const __half*)a_hi, rerun_lo ? (const __half*)a_lo : nullptr, lda, a_norms,
            a_row_inv, w.g_hi, w.g_lo, w.g_norms, w.g_row_inv, w.ctrl + 1, w.ctrl + 2);
        ISE_LAUNCH_CHECK();
    }
    // ---- 3. split products over the compacted rows (row count read on the device), results scattered back
    {
        Params q = p;
        q.m = w.cap; q.n_mtiles = (int)ceil_div64(w.cap, BLOCK_M);
        q.a_norms = w.g_norms; q.a_row_inv = a_row_inv ? w.g_row_inv : nullptr;
        q.m_dev = w.ctrl + 1; q.row_map = w.flag_rows;
        if (setup_maps_var(ctx, w.g_hi, rerun_lo ? w.g_lo : nullptr, lda, b_hi, b_lo, ldb, w.cap, n, d, pair, maps)) return 1;
        const int rc = rerun_lo ? launch_cg<2, 2, L2, 1, false, 2>(ctx, maps, q, st) : launch_cg<1, 2, L2, 1, false, 2>(ctx, maps, q, st);
        if (rc) return rc;
    }
    // ---- 4. more listed rows than the compact buffers hold (degenerate codebooks): everything again, split products
    {
        Params q = p;
        q.gate = w.ctrl + 2;
        if (setup_maps_var(ctx, a_hi, rerun_lo ? a_lo : nullptr, lda, b_hi, b_lo, ldb, m, n, d, pair, maps)) return 1;
        const int rc = rerun_lo ? launch_cg<2, 2, L2, 1, false, 2>(ctx, maps, q, st) : launch_cg<1, 2, L2, 1, false, 2>(ctx, maps, q, st);
        if (rc) return rc;
    }
    return 0;
}

}  // namespace gs

ISE_EXPORT size_t ise_assign_workspace_bytes(ise_ctx* ctx, int64_t m, int d) {
    if (!ctx || m <= 0 || d <= 0) return 0;
    return gs::verified_ws(nullptr, m, ((int64_t)d + 7) / 8 * 8).bytes;
}

ISE_EXPORT int ise_assign_verified_covers(ise_ctx* ctx, int64_t m, int64_t n, int d) {
    if (!ctx || m <= 0 || n <= 0 || d <= 0) return 0;
    return gs::verified_covers(ctx, m, n, d, ((int64_t)d + 7) / 8 * 8) ? 1 : 0;
}

// Verified top-1 over PREPARED row planes (k-means iterations: the rows are prepared once): ids equal the split
// products'; out_val holds the one-product scores (|error| <= the coarse bound) except for re-run rows.  Returns 2 when
// the shape is not covered.
ISE_EXPORT int ise_assign_verified(ise_ctx* ctx, const void* a_hi, const void* a_lo, int64_t lda, const float* a_meta,
                                   const float* a_norms, const float* a_row_inv, const void* b_hi, const void* b_lo,
                                   int64_t ldb, const float* b_meta, const float* b_norms, int64_t m, int64_t n, int d,
                                   int metric, int64_t id_base, float* out_val, int64_t* out_idx, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(m >= 0 && n > 0 && d > 0 && n < (int64_t)1 << 31 && m < (int64_t)1 << 31);
    if (m == 0) return 0;
    ISE_CHECK_ARG(a_hi && a_meta && a_norms && b_hi && b_meta && out_val && out_idx && workspace);
    if (metric == ISE_METRIC_L2) ISE_CHECK_ARG(b_norms != nullptr);
    ISE_CHECK_ARG(lda >= d && ldb >= d && lda % 8 == 0 && ldb % 8 == 0);
    ISE_CHECK_ARG(((reinterpret_cast<uintptr_t>(a_hi) | reinterpret_cast<uintptr_t>(a_lo) | reinterpret_cast<uintptr_t>(b_hi) |
                    reinterpret_cast<uintptr_t>(b_lo) | reinterpret_cast<uintptr_t>(workspace)) & 15) == 0);
    if (b_lo == nullptr || !gs::verified_covers(ctx, m, n, d, lda)) return 2;
    const gs::VerifiedWs w = gs::verified_ws(workspace, m, lda);
    if (workspace_bytes < w.bytes) ISE_FAIL("workspace too small: need " + std::to_string(w.bytes));
    DeviceGuard guard(ctx->device);
    const gs::Plan pl = gs::make_plan(ctx, m, n, d, 1, true, false);
    const gs::Params p = gs::make_params(pl, m, n, d, 1, id_base, a_meta, a_norms, a_row_inv, b_meta, b_norms, out_val, out_idx);
    return metric == ISE_METRIC_L2
               ? gs::verified_launches<true>(ctx, p, nullptr, 0, const_cast<void*>(a_hi), const_cast<void*>(a_lo), lda, nullptr, nullptr, b_hi, b_lo, ldb, w, (cudaStream_t)stream)
               : gs::verified_launches<false>(ctx, p, nullptr, 0, const_cast<void*>(a_hi), const_cast<void*>(a_lo), lda, nullptr, nullptr, b_hi, b_lo, ldb, w, (cudaStream_t)stream);
}

// Fused assign: raw float32 rows in, nearest column out, with the row operand (planes, norms, per-row scales, meta) as a
// by-product.  Returns 2 (and does nothing) when the shape is outside what the fused kernel covers -- the caller then
// runs ise_prepare_rows + ise_gemm_select.
ISE_EXPORT int ise_assign_fused(ise_ctx* ctx, const float* x, int64_t ldx, int64_t m, int d, void* a_hi, void* a_lo,
                                int64_t lda, float* a_norms, float* a_row_inv, uint8_t* a_lo_skipped, float* a_meta,
                                const void* b_hi, const void* b_lo, int64_t ldb, const float* b_meta, const float* b_norms,
                                int64_t n, int metric, int64_t id_base, float* out_val, int64_t* out_idx, void* workspace,
                                size_t workspace_bytes, void* stream) {
    ISE_CHECK_ARG(ctx != nullptr);
    ISE_CHECK_ARG(metric == ISE_METRIC_IP || metric == ISE_METRIC_L2);
    ISE_CHECK_ARG(m >= 0 && n > 0 && d > 0 && n < (int64_t)1 << 31 && m < (int64_t)1 << 31);
    if (m == 0) return 0;
    ISE_CHECK_ARG(x && a_hi && a_norms && a_row_inv && a_meta && b_hi && b_meta && out_val && out_idx);
    ISE_CHECK_ARG(a_lo == nullptr || a_lo_skipped != nullptr);
    // rows that may be inexact need the split products, and those have no (2, 1) plane combination
    if (a_lo != nullptr && b_lo == nullptr) ISE_FAIL("a_lo without b_lo is not supported: pass a zero b_lo plane");
    if (metric == ISE_METRIC_L2) ISE_CHECK_ARG(b_norms != nullptr);
    ISE_CHECK_ARG(lda >= d && ldb >= d && lda % 8 == 0 && ldb % 8 == 0 && ldx >= d);
    const bool al16 = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(a_hi) | reinterpret_cast<uintptr_t>(a_lo) |
                        reinterpret_cast<uintptr_t>(b_hi)) & 15) == 0;
    gs::Plan pl = gs::make_plan(ctx, m, n, d, 1, false, b_lo != nullptr);
    // covered: 16-byte aligned float32 rows of at most 128 columns (every keypoint descriptor type: SIFT 128, BRISK 64,
    // ORB 32), an unsplit column range (enough row tiles to fill the machine)
    if (d % 4 != 0 || ldx % 4 != 0 || lda > 128 || !al16 || pl.n_splits != 1) return 2;
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    ISE_CUDA(cudaMemsetAsync(a_meta, 0, META_FLOATS * sizeof(float), st));
    gs::Params p = gs::make_params(pl, m, n, d, 1, id_base, a_meta, a_norms, a_row_inv, b_meta, b_norms, out_val, out_idx);
    const bool l2 = metric == ISE_METRIC_L2;
    int rc;
    if (workspace != nullptr && b_lo != nullptr && gs::verified_covers(ctx, m, n, d, lda)) {
        // ids only need ONE product per tile plus a proof: verified coarse pass, compact split re-run of the few rows
        // it cannot decide (out_val: one-product scores except for those rows)
        ISE_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 15) == 0);
        const gs::VerifiedWs w = gs::verified_ws(workspace, m, lda);
        if (workspace_bytes < w.bytes) ISE_FAIL("workspace too small: need " + std::to_string(w.bytes));
        rc = l2 ? gs::verified_launches<true>(ctx, p, x, ldx, a_hi, a_lo, lda, a_lo_skipped, a_meta, b_hi, b_lo, ldb, w, st)
                : gs::verified_launches<false>(ctx, p, x, ldx, a_hi, a_lo, lda, a_lo_skipped, a_meta, b_hi, b_lo, ldb, w, st);
        if (rc) return rc;
        if (a_lo) {     // rows that were NOT exact in their hi plane (device-side flag): the split products over all of them
            if (ise_internal_lo_fixup(ctx, a_lo, m, lda, a_lo_skipped, a_meta, stream)) return 1;
            return gemm_select_impl(ctx, a_hi, a_lo, lda, a_meta, a_norms, a_row_inv, b_hi, b_lo, ldb, b_meta, b_norms, m, n, d,
                                    metric, 1, id_base, nullptr, nullptr, nullptr, out_val, out_idx, nullptr, 0, stream, 1);
        }
        return 0;
    }
    CUtensorMap maps[4];
    if (setup_maps(ctx, a_hi, nullptr, lda, b_hi, b_lo, ldb, m, n, d, 1, maps)) return 1;
    p.a_raw = x; p.lda_raw = ldx; p.a_hi_w = (__half*)a_hi; p.a_lo_w = (__half*)a_lo; p.lda_w = lda;
    p.a_norms_w = a_norms; p.a_row_inv_w = a_row_inv; p.a_lo_skipped = a_lo_skipped; p.a_meta_w = a_meta;
    const int cg = gs::pick_variant(m, n, d, b_lo != nullptr, 1).cg;
    if (b_lo == nullptr) {      // no split products (a_lo is NULL too): CTA pairs are never picked
        if (cg != 1) ISE_FAIL("internal: CTA pairs picked for the fused assign without a B lo plane");
        rc = l2 ? gs::launch_cg<1, 1, true, 1, false, 1, 1, true>(ctx, maps, p, st)
                : gs::launch_cg<1, 1, false, 1, false, 1, 1, true>(ctx, maps, p, st);
    } else if (cg == 2) {
        rc = l2 ? gs::launch_cg<1, 2, true, 1, false, 2, 1, true>(ctx, maps, p, st)
                : gs::launch_cg<1, 2, false, 1, false, 2, 1, true>(ctx, maps, p, st);
    } else {
        rc = l2 ? gs::launch_cg<1, 2, true, 1, false, 1, 1, true>(ctx, maps, p, st)
                : gs::launch_cg<1, 2, false, 1, false, 1, 1, true>(ctx, maps, p, st);
    }
    if (rc) return rc;
    if (a_lo) {
        // the tensor was NOT exact in its hi plane (device-side flag): complete the lo plane of the rows that skipped
        // it and repeat the assign with the lo products; both launches return at once otherwise
        if (ise_internal_lo_fixup(ctx, a_lo, m, lda, a_lo_skipped, a_meta, stream)) return 1;
        return gemm_select_impl(ctx, a_hi, a_lo, lda, a_meta, a_norms, a_row_inv, b_hi, b_lo, ldb, b_meta, b_norms, m, n, d,
                                metric, 1, id_base, nullptr, nullptr, nullptr, out_val, out_idx, nullptr, 0, stream, 1);
    }
    return 0;
}
