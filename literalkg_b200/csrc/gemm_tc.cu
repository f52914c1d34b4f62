// Tensor-core GEMM engine of the path:  C[M,N] = epilogue( A[M,K] @ B[N,K]^T ), fp32-class accuracy.
//
//   lkg_linear_fwd : act(A B^T + bias)                      linear_gat (model.py:309-310) and the h0 @ Q residual terms
//   lkg_gate_fwd   : literal gate, tanh / sigmoid / mix      GateMul / Gate (gate.py:22-28, 45-51)
//   lkg_score      : emb[heads] @ emb[tails]^T (+ min/max)   calc_score / predict_links (model.py:473-491)
//
// sm_100a design
//   * operands live in HBM as fp16 "planes": s*x = hi + lo with hi = fp16(s*x), lo = fp16(s*x - hi)  (2 x 2 bytes,
//     the same footprint as the fp32 value; s = power of two from the operand's scale record, so the split is
//     exact up to 22 significand bits).  Three tcgen05.mma per k-step  hi*hi + lo*hi + hi*lo  accumulate in fp32
//     TMEM; the dropped lo*lo term and the residual of the split are ~2^-22 relative, i.e. fp32-class: the GEMMs
//     that feed LayerNorm over 32 features get amplified on the way to the final embeddings (the fp32 reference
//     itself sits ~1e-4 from fp64 there, SURVEY.md appendix A), so a bf16 split (2^-17) eats the 1e-3 parity
//     budget and a single bf16 pass (2^-9) is far above it;
//   * TMA (cp.async.bulk.tensor.3d, 128-byte swizzle) stages {hi, lo} x 64-wide K chunks of A (128 rows) and
//     B (N-tile rows) into shared memory; a 2-stage mbarrier ring feeds one MMA-issuing thread;
//   * accumulators: 2 x 256 TMEM columns, double buffered so the epilogue of tile i overlaps the MMAs of
//     tile i+1; 4 epilogue warps read them back with tcgen05.ld (32 lanes x 16 columns per instruction);
//   * persistent CTAs (one per SM), static tile round-robin, N fastest so that co-running CTAs share A tiles in L2;
//   * the virtual torch.cat of the reference is a list of K segments, each with its own tensor map.
#include <cstdlib>

#include "tc.cuh"

namespace lkg {
namespace {

using namespace tc;
constexpr int kMaxBN = 256;       // columns per tile (UMMA N)
constexpr int kStages = 4;        // upper bound; a launch uses as many as fit next to its B tile (TcParams::stages)
// Epilogue warp groups of 4 (one warp per TMEM lane quarter), each takes a column range of the tile.  Template
// parameter G of the kernel: 2 for the linear / score epilogues (stores only), 3 for the gate (4 MUFU + ~20 other
// instructions per output channel: with 8 warps the epilogue, not the MMAs, paced the tile -- ncu r02b).
// Thread layout: warps 0-3 epilogue group 0, warp 4 TMA producer, warp 5 MMA issuer, warps 6.. epilogue groups 1..
__host__ __device__ constexpr int threads_for(int groups) { return 64 + 128 * groups; }
constexpr uint32_t kABytes = 2 * kBM * kBK * 2;            // hi + lo planes of one A chunk
constexpr uint32_t kSmemBudget = 227 * 1024;
// Epilogue staging: a warp owns 32 TMEM lanes (= tile rows), one thread per row.  Storing a thread's row straight to
// global memory makes every 16-byte store of the warp hit 32 different lines (32 LSU wavefronts per instruction; ncu
// r02a: the epilogue, not the MMAs or the L2 -> SM fill, set the tile time of every GEMM of the pass).  Each warp
// therefore transposes 32 rows x 32 accumulator columns through shared memory (pitch 33 floats: conflict free both
// ways) and touches global memory with 8 (gate: 4) lanes per row -- whole 128-byte (64-byte) row segments.
constexpr int kStagePitch = 33;
__host__ __device__ constexpr uint32_t epi_stage_bytes(int groups) { return (uint32_t)groups * 4 * 32 * kStagePitch * 4; }
// bn_cta = rows of the B tile one CTA stages (the whole N tile, or half of it in a CTA pair)
__host__ __device__ constexpr uint32_t stage_bytes_for(int bn_cta) { return kABytes + 2u * (uint32_t)bn_cta * kBK * 2u; }
inline int stages_for(int bn_cta, int groups) {
    const int s = (int)((kSmemBudget - 1024 - 256 - epi_stage_bytes(groups)) / stage_bytes_for(bn_cta));
    return s > kStages ? kStages : s;
}

enum EpiKind { kEpiLinear = 0, kEpiGate = 1, kEpiScore = 2, kEpiRank = 3 };

struct TcParams {
    CUtensorMap a_map[LKG_MAX_SEGMENTS];
    CUtensorMap b_map;
    int n_segments;
    int seg_chunks[LKG_MAX_SEGMENTS];   // number of 64-wide chunks of each A segment
    int seg_bcol[LKG_MAX_SEGMENTS];     // first column of the segment inside the packed B planes
    int64_t m;
    int n;                              // valid output columns (GEMM N)
    int bn;                             // N tile (multiple of 16, <= 256)
    int tiles_m, tiles_n;
    int m_fastest;
    int stages;                         // pipeline depth of this launch (2 .. kStages)
    uint32_t stage_bytes;               // kABytes + hi/lo planes of a bn x 64 B tile
    // epilogue
    const float* bias;                  // linear: [n]; gate: interleaved pairs [n]
    int act;
    float* out;
    int64_t ldo;
    float* out2;                        // linear, optional: the columns from split_col (a multiple of 4) on are written
    int64_t ld2;                        //   to out2[row * ld2 + col - split_col] instead (two consumers, two layouts)
    int split_col;
    __half* out_planes;                 // optional hi/lo copy of the output (feeds the next GEMM)
    int64_t ld_planes, plane_stride;
    const float* x_ent;                 // gate mix input
    int64_t ld_ent;
    uint32_t* minmax;                   // score: ordered-encoded running {min, max}
    const float* mul_a;                 // scale records whose [2] (= 1/scale) the accumulator is multiplied by:
    const float* mul_b;                 //   mul_b = packed weight (1/S) or tails; mul_a = heads (score only), nullable
    const float* out_rec;               // scale record of out_planes
    float* gz_out;                      // gate, training: activated (tanh g, sigmoid z) pairs [m, n] (nullable)
    int64_t ld_gz;
    int accumulate;                     // linear: out += result
    // rank epilogue (lkg_score_rank): no score is stored.  Per head row the columns whose score is certainly above the
    // target's are counted; the ones inside the error band around it are listed for an exact re-score
    const float* rank_thr;              // [m][2] {lo, hi} = exact target score -/+ the error bound of the 3-product GEMM
    int* rank_above;                    // [m]   += columns with score > hi
    int* rank_band_cnt;                 // [m]   += columns with lo <= score <= hi
    int* rank_band;                     // [m][rank_band_cap] those columns (first rank_band_cap of them)
    int rank_band_cap;
};

__device__ __forceinline__ uint32_t order_enc(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ---- epilogue of one 32-row x 32-column accumulator block, staged in shared memory as st[row * kStagePitch + col] ----
__device__ __forceinline__ float4 ld4_guard(const float* ptr, int valid, bool vec) {
    if (vec && valid >= 4) return __ldg(reinterpret_cast<const float4*>(ptr));
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid > 0) v.x = __ldg(ptr);
    if (valid > 1) v.y = __ldg(ptr + 1);
    if (valid > 2) v.z = __ldg(ptr + 2);
    if (valid > 3) v.w = __ldg(ptr + 3);
    return v;
}
__device__ __forceinline__ void st4_guard(float* ptr, const float4& v, int valid, bool vec) {
    if (vec && valid >= 4) {
        *reinterpret_cast<float4*>(ptr) = v;
        return;
    }
    if (valid > 0) ptr[0] = v.x;
    if (valid > 1) ptr[1] = v.y;
    if (valid > 2) ptr[2] = v.z;
    if (valid > 3) ptr[3] = v.w;
}
// hi/lo planes of four consecutive values (already multiplied by the plane scale)
__device__ __forceinline__ void st_planes4(__half* hrow, int64_t plane_stride, const float4& v, int valid, bool vec) {
    __align__(8) __half h[4], l[4];
    split_f16(v.x, h[0], l[0]);
    split_f16(v.y, h[1], l[1]);
    split_f16(v.z, h[2], l[2]);
    split_f16(v.w, h[3], l[3]);
    __half* lrow = hrow + plane_stride;
    if (vec && valid >= 4) {
        *reinterpret_cast<uint2*>(hrow) = *reinterpret_cast<const uint2*>(h);
        *reinterpret_cast<uint2*>(lrow) = *reinterpret_cast<const uint2*>(l);
        return;
    }
    for (int j = 0; j < 4; ++j)
        if (j < valid) {
            hrow[j] = h[j];
            lrow[j] = l[j];
        }
}

// Alignment facts of a launch that let the epilogue use 16-byte (planes: 8-byte) accesses; computed once per thread.
struct EpiAlign {
    bool out4, ent4, gz4, planes4, bias4;
};
__device__ __forceinline__ EpiAlign epi_align(const TcParams& p) {
    EpiAlign a;
    a.out4 = ((reinterpret_cast<uintptr_t>(p.out) & 15u) == 0) && (p.ldo % 4 == 0) &&
             (!p.out2 || (((reinterpret_cast<uintptr_t>(p.out2) & 15u) == 0) && (p.ld2 % 4 == 0)));
    a.ent4 = p.x_ent && ((reinterpret_cast<uintptr_t>(p.x_ent) & 15u) == 0) && (p.ld_ent % 4 == 0);
    a.gz4 = p.gz_out && ((reinterpret_cast<uintptr_t>(p.gz_out) & 15u) == 0) && (p.ld_gz % 4 == 0);
    a.planes4 = p.out_planes && ((reinterpret_cast<uintptr_t>(p.out_planes) & 7u) == 0) && (p.ld_planes % 4 == 0) &&
                (p.plane_stride % 4 == 0);
    a.bias4 = p.bias && ((reinterpret_cast<uintptr_t>(p.bias) & 15u) == 0);
    return a;
}

// linear / score: 8 lanes per row (4 columns each), 4 rows per pass, 8 passes.  `old` = prefetched previous values of
// the output (accumulate mode).  col0 = first GEMM column of the block (multiple of 16).
template <int EPI>
__device__ __forceinline__ void epilogue_block(const TcParams& p, const EpiAlign& al, const float* st, int64_t row0,
                                               int col0, int col_end, int lane, float out_scale, float& lo, float& hi) {
    const int c4 = lane & 7, rsub = lane >> 3;
    const int col = col0 + 4 * c4;
    const int valid = col_end - col;             // columns of this lane inside the tile and the matrix (<= 0: none)
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (EPI == kEpiLinear && p.bias && valid > 0) b = ld4_guard(p.bias + col, valid, al.bias4);
    float* obase = p.out + col;
    int64_t ostride = p.ldo;
    if (EPI == kEpiLinear && p.out2 && col >= p.split_col) {
        obase = p.out2 + (col - p.split_col);
        ostride = p.ld2;
    }
    float4 old[8];
    if (EPI == kEpiLinear && p.accumulate) {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int64_t row = row0 + it * 4 + rsub;
            old[it] = (row < p.m && valid > 0) ? ld4_guard(obase + row * ostride, valid, al.out4)
                                               : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int rl = it * 4 + rsub;
        const int64_t row = row0 + rl;
        const float* sp = st + rl * kStagePitch + 4 * c4;
        float4 v = make_float4(sp[0], sp[1], sp[2], sp[3]);
        if (row >= p.m || valid <= 0) continue;
        if (EPI == kEpiLinear) {
            v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
            if (p.act == LKG_ACT_LEAKY_RELU) {
                v.x = leaky(v.x); v.y = leaky(v.y); v.z = leaky(v.z); v.w = leaky(v.w);
            } else if (p.act == LKG_ACT_TANH) {
                v.x = tanh_acc(v.x); v.y = tanh_acc(v.y); v.z = tanh_acc(v.z); v.w = tanh_acc(v.w);
            }
            if (p.accumulate) {
                v.x += old[it].x; v.y += old[it].y; v.z += old[it].z; v.w += old[it].w;
            }
        }
        if (EPI == kEpiScore) {
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (j < valid) {
                    lo = fminf(lo, vv[j]);
                    hi = fmaxf(hi, vv[j]);
                }
        }
        st4_guard(obase + row * ostride, v, valid, al.out4);
        if (EPI == kEpiLinear && p.out_planes) {
            const float4 sv = make_float4(v.x * out_scale, v.y * out_scale, v.z * out_scale, v.w * out_scale);
            st_planes4(p.out_planes + row * p.ld_planes + col, p.plane_stride, sv, valid, al.planes4);
        }
    }
}

// gate: the 32 accumulator columns are 16 (g, z) pairs = 16 output channels; 4 lanes per row (4 channels each),
// 8 rows per pass, 4 passes.  `e` = the lane's x_ent values, loaded by the caller before the accumulator wait.
__device__ __forceinline__ void gate_prefetch(const TcParams& p, const EpiAlign& al, int64_t row0, int col0, int col_end,
                                              int lane, float4 (&e)[4]) {
    const int ch = (col0 >> 1) + 4 * (lane & 3);
    const int valid = (col_end >> 1) - ch;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int64_t row = row0 + it * 8 + (lane >> 2);
        e[it] = (row < p.m && valid > 0) ? ld4_guard(p.x_ent + row * p.ld_ent + ch, valid, al.ent4)
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
__device__ __forceinline__ void gate_block(const TcParams& p, const EpiAlign& al, const float* st, int64_t row0,
                                           int col0, int col_end, int lane, float out_scale, const float4 (&e)[4]) {
    const int q = lane & 3, rsub = lane >> 2;
    const int ch = (col0 >> 1) + 4 * q;          // first output channel of this lane
    const int valid = (col_end >> 1) - ch;       // channels inside the tile and the matrix
    if (valid <= 0) return;
    const float4 b0 = ld4_guard(p.bias + col0 + 8 * q, 2 * valid, al.bias4);          // (g, z) bias pairs
    const float4 b1 = ld4_guard(p.bias + col0 + 8 * q + 4, 2 * valid - 4, al.bias4);
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int rl = it * 8 + rsub;
        const int64_t row = row0 + rl;
        const float* sp = st + rl * kStagePitch + 8 * q;
        const float a0 = sp[0], a1 = sp[1], a2 = sp[2], a3 = sp[3], a4 = sp[4], a5 = sp[5], a6 = sp[6], a7 = sp[7];
        if (row >= p.m) continue;
        float4 g, z, o;
        // tanh_acc / sigmoid_acc keep RELATIVE accuracy near zero (the gate's pre-activations are ~0.05 at the reference's
        // initialisation): a 5-instruction 1 - 2 / (1 + e^{2x}) is 2e-7 ABSOLUTE, 30 x worse there, and the LayerNorms
        // downstream amplify it (bench parity leg: row-error quantiles 3 - 10 x the fp32 reference's).  With 12 epilogue
        // warps the MMAs, not this math, pace the tile.
        g.x = tanh_acc(a0 + b0.x); z.x = sigmoid_acc(a1 + b0.y);
        g.y = tanh_acc(a2 + b0.z); z.y = sigmoid_acc(a3 + b0.w);
        g.z = tanh_acc(a4 + b1.x); z.z = sigmoid_acc(a5 + b1.y);
        g.w = tanh_acc(a6 + b1.z); z.w = sigmoid_acc(a7 + b1.w);
        o.x = (1.f - z.x) * e[it].x + z.x * g.x;
        o.y = (1.f - z.y) * e[it].y + z.y * g.y;
        o.z = (1.f - z.z) * e[it].z + z.z * g.z;
        o.w = (1.f - z.w) * e[it].w + z.w * g.w;
        if (p.gz_out) {
            float* grow = p.gz_out + row * p.ld_gz + col0 + 8 * q;
            st4_guard(grow, make_float4(g.x, z.x, g.y, z.y), 2 * valid, al.gz4);
            st4_guard(grow + 4, make_float4(g.z, z.z, g.w, z.w), 2 * valid - 4, al.gz4);
        }
        st4_guard(p.out + row * p.ldo + ch, o, valid, al.out4);
        if (p.out_planes) {
            const float4 sv = make_float4(o.x * out_scale, o.y * out_scale, o.z * out_scale, o.w * out_scale);
            st_planes4(p.out_planes + row * p.ld_planes + ch, p.plane_stride, sv, valid, al.planes4);
        }
    }
}

// CG = 1: one CTA per 128-row tile.  CG = 2: a CTA pair (cluster of 2) per 256-row tile -- the leader issues
// tcgen05.mma.cta_group::2 (M = 256), every CTA stages its own 128 rows of A and HALF of the B tile (gate GEMM: 586 KB
// instead of 850 KB pulled from L2 per CTA and tile, one more pipeline stage, B read from shared memory once for
// both tensor cores).  Measured (r02c, cfg 3): gate 2.17 -> 2.07 ms, h0 @ Q 0.48 -> 0.43 ms, linear_gat 0.63 -> 0.57 ms;
// bit-identical results.  What took the gate from 2.57 ms to there was the epilogue (coalesced staging, 12 warps):
// ncu then shows the tensor pipe 75 % busy at the power-capped 1.27 GHz -- three products per k-step are the floor.
template <int EPI, int CG, int G>
__global__ void __launch_bounds__(threads_for(G), 1) tc_gemm_kernel(const __grid_constant__ TcParams p) {
    constexpr int kEpiGroups = G;
    constexpr int kEpiWarps = 4 * G;
    constexpr uint32_t kEpiStageBytes = epi_stage_bytes(G);
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const uint32_t kStageBytes = p.stage_bytes;
    const int n_stages = p.stages;
    float* epi_stage = reinterpret_cast<float*>(smem + n_stages * kStageBytes);      // [kEpiWarps][32][kStagePitch]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + n_stages * kStageBytes + kEpiStageBytes);
    uint64_t* full = bars;                 // [kStages]  TMA bytes landed (CG = 2: the leader's counts both CTAs' bytes)
    uint64_t* empty = bars + kStages;      // [kStages]  MMAs that read the stage retired (CG = 2: multicast commit)
    uint64_t* acc_full = bars + 2 * kStages;       // [2]  accumulator complete
    uint64_t* acc_empty = bars + 2 * kStages + 2;  // [2]  accumulator drained by the epilogue warps (of both CTAs)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    const int unit = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;        // tile-scheduling unit: CTA or CTA pair
    const int n_units = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int total_tiles = p.tiles_m * p.tiles_n;
    const int bn_cta = p.bn / CG;          // rows of the B tile this CTA stages
    int n_chunks = 0;
    for (int s = 0; s < p.n_segments; ++s) n_chunks += p.seg_chunks[s];

    if (warp == 4 && lane == 0) {
        for (int s = 0; s < p.n_segments; ++s)
            asm volatile("prefetch.tensormap [%0];" ::"l"(&p.a_map[s]) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&p.b_map) : "memory");
        for (int s = 0; s < n_stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&acc_full[a], 1);
            mbar_init(&acc_empty[a], kEpiWarps * CG);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        if (CG == 2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                         "r"(512));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                         "r"(512));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync_all();       // the peer's barriers are initialised before anything remote touches them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t b_bytes = 2u * (uint32_t)bn_cta * kBK * 2u;

    auto tile_coords = [&](int tile, int& mb, int& nb) {
        if (p.m_fastest) {
            mb = tile % p.tiles_m;
            nb = tile / p.tiles_m;
        } else {
            nb = tile % p.tiles_n;
            mb = tile / p.tiles_n;
        }
    };

    if (warp == 4) {
        // ===== TMA producer (one per CTA) =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int tile = unit; tile < total_tiles; tile += n_units) {
                int mb, nb;
                tile_coords(tile, mb, nb);
                const int a_row = (mb * CG + (int)cta_rank) * kBM;
                const int b_row = nb * p.bn + (int)cta_rank * bn_cta;
                for (int s = 0; s < p.n_segments; ++s) {
                    for (int j = 0; j < p.seg_chunks[s]; ++j) {
                        mbar_wait(&empty[stage], phase ^ 1);
                        uint8_t* st = smem + stage * kStageBytes;
                        if (CG == 2) {
                            // both CTAs' bytes are counted on the leader's barrier: the MMA issuer lives there
                            if (leader) mbar_expect_tx(&full[stage], 2u * (kABytes + b_bytes));
                            const uint32_t bar = mapa_u32(&full[stage], 0);
                            tma_load_3d_cg2(&p.a_map[s], bar, st, j * kBK, a_row, 0);
                            tma_load_3d_cg2(&p.b_map, bar, st + kABytes, p.seg_bcol[s] + j * kBK, b_row, 0);
                        } else {
                            mbar_expect_tx(&full[stage], kABytes + b_bytes);
                            tma_load_3d(&p.a_map[s], &full[stage], st, j * kBK, a_row, 0);
                            tma_load_3d(&p.b_map, &full[stage], st + kABytes, p.seg_bcol[s] + j * kBK, b_row, 0);
                        }
                        if (++stage == (uint32_t)n_stages) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == 5) {
        // ===== MMA issuer (CG = 2: the leader CTA issues for the pair) =====
        if (lane == 0 && leader) {
            const uint32_t idesc = umma_idesc(p.bn, kBM * CG);
            uint32_t stage = 0, phase = 0;
            int it = 0;
            for (int tile = unit; tile < total_tiles; tile += n_units, ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (it >> 1) & 1;
                mbar_wait(&acc_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * kMaxBN;
                for (int c = 0; c < n_chunks; ++c) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_hi = smem_u32(smem + stage * kStageBytes);
                    const uint32_t a_lo = a_hi + kBM * kBK * 2;
                    const uint32_t b_hi = a_hi + kABytes;
                    const uint32_t b_lo = b_hi + (uint32_t)bn_cta * kBK * 2;
#pragma unroll
                    for (int k = 0; k < kBK / 16; ++k) {
                        const uint32_t koff = k * 32;   // 16 fp16 = 32 bytes inside the swizzle row
                        const uint64_t dah = umma_desc(a_hi + koff), dal = umma_desc(a_lo + koff);
                        const uint64_t dbh = umma_desc(b_hi + koff), dbl = umma_desc(b_lo + koff);
                        if (CG == 2) {
                            tc_mma_f16_cg2(tmem_d, dah, dbh, idesc, (c | k) != 0);
                            tc_mma_f16_cg2(tmem_d, dal, dbh, idesc, 1);
                            tc_mma_f16_cg2(tmem_d, dah, dbl, idesc, 1);
                        } else {
                            tc_mma_f16(tmem_d, dah, dbh, idesc, (c | k) != 0);
                            tc_mma_f16(tmem_d, dal, dbh, idesc, 1);
                            tc_mma_f16(tmem_d, dah, dbl, idesc, 1);
                        }
                    }
                    // frees the smem stage (in both CTAs) when these MMAs retire
                    if (CG == 2) tc_commit_cg2(&empty[stage], 3); else tc_commit(&empty[stage]);
                    if (++stage == (uint32_t)n_stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                // accumulator ready for the epilogue warps (of both CTAs)
                if (CG == 2) tc_commit_cg2(&acc_full[acc], 3); else tc_commit(&acc_full[acc]);
            }
        }
    } else {
        // ===== epilogue warps: TMEM lane = tile row of this CTA =====
        int it = 0;
        float lo = INFINITY, hi = -INFINITY;
        // powers of two: the rescale is exact
        const float acc_scale = (p.mul_a ? __ldg(p.mul_a + 2) : 1.f) * (p.mul_b ? __ldg(p.mul_b + 2) : 1.f);
        const float out_scale = (p.out_planes && p.out_rec) ? __ldg(p.out_rec + 1) : 1.f;
        const uint32_t acc_empty_leader0 = CG == 2 ? mapa_u32(&acc_empty[0], 0) : 0u;   // the leader's barriers
        const uint32_t acc_empty_leader1 = CG == 2 ? mapa_u32(&acc_empty[1], 0) : 0u;
        const EpiAlign al = epi_align(p);
        // a warp reads the TMEM lanes of its quarter (warp % 4); every group of four warps takes its own range of the
        // tile's columns, 32 at a time
        const int quarter = warp & 3;
        const int group = warp < 4 ? 0 : 1 + (warp - 6) / 4;
        float* st = epi_stage + (group * 4 + quarter) * 32 * kStagePitch;
        const int c_per = ((p.bn + 32 * kEpiGroups - 1) / (32 * kEpiGroups)) * 32;
        const int c_begin = min(group * c_per, p.bn), c_end = min(c_begin + c_per, p.bn);
        for (int tile = unit; tile < total_tiles; tile += n_units, ++it) {
            int mb, nb;
            tile_coords(tile, mb, nb);
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            const int64_t row0 = ((int64_t)mb * CG + cta_rank) * kBM + quarter * 32;
            float4 e[4];
            const int col_end = min(p.n, (nb + 1) * p.bn);     // accumulator columns past it belong to no output
            if (EPI == kEpiGate && c_begin < c_end) gate_prefetch(p, al, row0, nb * p.bn + c_begin, col_end, lane, e);
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * kMaxBN;
            float2 rthr = make_float2(INFINITY, INFINITY);
            int rank_cnt = 0;
            if (EPI == kEpiRank && row0 + lane < p.m)
                rthr = __ldg(reinterpret_cast<const float2*>(p.rank_thr) + row0 + lane);
            for (int c0 = c_begin; c0 < c_end; c0 += 32) {
                uint32_t raw[32];
                // the accumulator buffers are kMaxBN columns apart: a 32-column read that starts inside the tile
                // stays inside the allocation; columns past the tile are masked by the block epilogues
                tc_ld32_nowait(taddr + c0, raw);
                tc_ld_wait();
                const bool last = c0 + 32 >= c_end;
                if (last) {                // every TMEM read of this tile is done: hand the accumulator back now
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {       // one arrival per epilogue warp, on the barrier the MMA issuer waits on
                        if (CG == 2) mbar_arrive_cluster(acc ? acc_empty_leader1 : acc_empty_leader0);
                        else mbar_arrive(&acc_empty[acc]);
                    }
                }
                const int col0 = nb * p.bn + c0;
                if (EPI == kEpiRank) {     // thread = head row: nothing to store, no transpose
                    const int64_t row = row0 + lane;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float v = __uint_as_float(raw[j]) * acc_scale;
                        const bool in = col0 + j < col_end;
                        rank_cnt += (in && v > rthr.y) ? 1 : 0;
                        if (in && v >= rthr.x && v <= rthr.y) {
                            const int slot = atomicAdd(p.rank_band_cnt + row, 1);
                            if (slot < p.rank_band_cap) p.rank_band[row * p.rank_band_cap + slot] = col0 + j;
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) st[lane * kStagePitch + j] = __uint_as_float(raw[j]) * acc_scale;
                    __syncwarp();
                    if (EPI == kEpiGate) {
                        float4 e_next[4];      // the next block's x_ent rows travel while this block is computed
                        if (!last) gate_prefetch(p, al, row0, col0 + 32, col_end, lane, e_next);
                        gate_block(p, al, st, row0, col0, col_end, lane, out_scale, e);
                        if (!last) {
#pragma unroll
                            for (int i = 0; i < 4; ++i) e[i] = e_next[i];
                        }
                    } else {
                        epilogue_block<EPI>(p, al, st, row0, col0, col_end, lane, out_scale, lo, hi);
                    }
                    __syncwarp();
                }
            }
            if (EPI == kEpiRank && rank_cnt > 0) atomicAdd(p.rank_above + row0 + lane, rank_cnt);
            if (c_begin >= c_end) {        // a group without columns in this launch still owes its arrival
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CG == 2) mbar_arrive_cluster(acc ? acc_empty_leader1 : acc_empty_leader0);
                    else mbar_arrive(&acc_empty[acc]);
                }
            }
        }
        if (EPI == kEpiScore && p.minmax) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo = fminf(lo, __shfl_xor_sync(kFull, lo, o));
                hi = fmaxf(hi, __shfl_xor_sync(kFull, hi, o));
            }
            if (lane == 0 && lo <= hi) {
                atomicMin(p.minmax, order_enc(lo));
                atomicMax(p.minmax + 1, order_enc(hi));
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync_all();       // no CTA leaves (or frees TMEM) while its peer may still signal / read it
    if (warp == 5) {
        tc_fence_after();
        if (CG == 2)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    }
}

// ---- host side ---------------------------------------------------------------------------------------
// planes tensor: fp16 [2 planes][rows][ld] with `plane_stride` elements between the planes; logical width k
int make_map(CUtensorMap* map, const void* base, int64_t rows, int k, int64_t ld, int64_t plane_stride, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) LKG_FAIL(LKG_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    LKG_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15u) == 0 && (ld * 2) % 16 == 0 && (plane_stride * 2) % 16 == 0,
                "fp16 planes must be 16-byte aligned (base, row stride, plane stride)");
    cuuint64_t dims[3] = {(cuuint64_t)k, (cuuint64_t)rows, 2};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)plane_stride * 2};
    cuuint32_t box[3] = {(cuuint32_t)kBK, (cuuint32_t)box_rows, 2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) LKG_FAIL(LKG_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return LKG_OK;
}

int pick_bn(int n, int min_tiles = 1) {
    // smallest number of N tiles, then the smallest tile (multiple of 16) that covers n.  (Measured in round 1: taking
    // more, narrower N tiles to fit a third cta_group::1 stage re-reads A and gains nothing: gate 2.69 -> 2.83 ms.)
    int tiles = (n + kMaxBN - 1) / kMaxBN;
    if (tiles < min_tiles) tiles = min_tiles;
    const int b = ((n + tiles - 1) / tiles + 15) / 16 * 16;
    return b < 16 ? 16 : b;
}

// lkg_gemm_set_cta_group / LKG_GEMM_CG=1|2 force the CTA-group size (A/B measurements, tests); default: pairs whenever
// every SM pair gets a tile
int g_forced_cg = -1;
inline int forced_cg() {
    if (g_forced_cg < 0) {
        const char* e = getenv("LKG_GEMM_CG");
        g_forced_cg = (e && (e[0] == '1' || e[0] == '2')) ? e[0] - '0' : 0;
    }
    return g_forced_cg;
}

template <int EPI, int CG>
int launch_tc_cg(TcParams& p, const lkg_planes* a, int64_t m, const lkg_planes* b, int n, cudaStream_t stream) {
    constexpr int G = EPI == kEpiGate ? 3 : 2;
    constexpr uint32_t kEpiStageBytes = epi_stage_bytes(G);
    constexpr int kThreads = threads_for(G);
    const int bn_cta = p.bn / CG;
    p.stages = stages_for(bn_cta, G);
    p.stage_bytes = stage_bytes_for(bn_cta);
    LKG_REQUIRE(p.stages >= 2, "GEMM tile does not fit shared memory");
    const size_t smem_bytes = (size_t)p.stages * p.stage_bytes + kEpiStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
    p.tiles_m = (int)((m + kBM * CG - 1) / (kBM * CG));
    p.tiles_n = (n + p.bn - 1) / p.bn;
    int bcol = 0;
    for (int s = 0; s < a->n_segments; ++s) {
        LKG_REQUIRE(a->ptr[s] && a->k[s] > 0, "bad A segment %d", s);
        p.seg_chunks[s] = (a->k[s] + kBK - 1) / kBK;
        p.seg_bcol[s] = bcol;
        bcol += p.seg_chunks[s] * kBK;
        if (int rc = make_map(&p.a_map[s], a->ptr[s], m, a->k[s], a->ld[s], a->plane_stride[s], kBM)) return rc;
    }
    LKG_REQUIRE(b->k[0] == bcol || (a->n_segments == 1 && b->k[0] == a->k[0]),
                "B has %d columns, the A segments need %d", b->k[0], bcol);
    if (int rc = make_map(&p.b_map, b->ptr[0], n, b->k[0], b->ld[0], b->plane_stride[0], bn_cta)) return rc;
    auto kern = tc_gemm_kernel<EPI, CG, G>;
    LKG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget));
    const int tiles = p.tiles_m * p.tiles_n;
    const int units = sm_count() / CG;                       // persistent: one CTA (or CTA pair) per SM (pair)
    const int grid = CG * (tiles < units ? tiles : units);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = CG == 2 ? 1 : 0;
    LKG_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
    LKG_LAUNCH_CHECK("tc_gemm_kernel");
    return LKG_OK;
}

template <int EPI>
int launch_tc(TcParams& p, const lkg_planes* a, int64_t m, const lkg_planes* b, int n, cudaStream_t stream) {
    LKG_REQUIRE(a && b && a->n_segments >= 1 && a->n_segments <= LKG_MAX_SEGMENTS && b->n_segments == 1, "bad operands");
    LKG_REQUIRE(m > 0 && n > 0, "empty GEMM");
    p.n_segments = a->n_segments;
    LKG_REQUIRE(b->scale[0] != nullptr, "the B operand needs a scale record");
    p.mul_b = b->scale[0];
    if (EPI == kEpiScore || EPI == kEpiRank) {
        LKG_REQUIRE(a->scale[0] != nullptr, "the heads operand needs a scale record");
        p.mul_a = a->scale[0];
    }
    p.m = m;
    p.n = n;
    p.bn = pick_bn(n);
    // a CTA pair halves the B bytes every CTA stages; worth it once there are enough 256-row tiles for every SM pair
    const int64_t pair_tiles = ((m + 2 * kBM - 1) / (2 * kBM)) * ((n + p.bn - 1) / p.bn);
    int cg = (p.bn % 16 == 0 && pair_tiles >= sm_count() / 2) ? 2 : 1;
    if (forced_cg() == 1 || (forced_cg() == 2 && p.bn % 16 == 0)) cg = forced_cg();
    // one CTA staging a whole 256-column B tile next to the gate's three epilogue groups has room for one pipeline
    // stage only (2 * dim = 256 or 512 at embed_dim 128 / 256): narrower N tiles until two stages fit
    constexpr int G = EPI == kEpiGate ? 3 : 2;
    for (int t = 2; stages_for(p.bn / cg, G) < 2 && t <= (n + 15) / 16; ++t) p.bn = pick_bn(n, t);
    return cg == 2 ? launch_tc_cg<EPI, 2>(p, a, m, b, n, stream) : launch_tc_cg<EPI, 1>(p, a, m, b, n, stream);
}

// ---- operand preparation -------------------------------------------------------------------------------
// Scale record {absmax, scale, 1/scale, counter, seg absmax x4}: scale = 2^e parks absmax * scale in [2^11, 2^12).
__device__ __forceinline__ void write_record(float* rec, float amax) {
    const int e = plane_exp(amax, 60);
    rec[0] = amax;
    rec[1] = ldexpf(1.f, e);
    rec[2] = ldexpf(1.f, -e);
}

// VEC: rows are 16-byte aligned -> the [m, k / 4] matrix of float4 units is walked flat (narrow matrices keep every
// lane busy), four independent loads per thread and step; the k % 4 tail columns and the unaligned case go through
// a scalar loop.  I: index type (uint32 while 4 strides past the end still fit).
// FINISH: the last block to leave turns the absmax into the record (rec was zeroed by the caller); otherwise the
// kernel only raises rec[0] (atomic max on the bits of a non-negative float) and lkg_scale_finish completes it.
template <typename I>
__device__ __forceinline__ float absmax_units(const float* __restrict__ src, int64_t ld, const int64_t* __restrict__ rows,
                                              int64_t m, int k) {
    constexpr int U = 4;
    const I kv = (I)(k >> 2);
    const I total = (I)m * kv;
    const I stride = (I)gridDim.x * blockDim.x;
    float mx = 0.f;
    for (I i = (I)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += U * stride) {
        float4 x[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const I j = i + (I)u * stride;
            x[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j < total) {
                const I r = j / kv;
                const I v = j - r * kv;
                x[u] = __ldg(reinterpret_cast<const float4*>(src + (rows ? rows[r] : (int64_t)r) * ld) + v);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)   // fmaxf drops a NaN operand: NaNs do not poison the scale
            mx = fmaxf(fmaxf(mx, fmaxf(fabsf(x[u].x), fabsf(x[u].y))), fmaxf(fabsf(x[u].z), fabsf(x[u].w)));
    }
    return mx;
}

template <bool VEC, bool FINISH>
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ src, int64_t ld,
                                                     const int64_t* __restrict__ rows, int64_t m, int k, float floor_,
                                                     float* __restrict__ rec) {
    float mx = 0.f;
    const int c_begin = VEC ? (k & ~3) : 0;             // columns the scalar loop covers
    if (VEC)
        mx = (m * (int64_t)(k >> 2) < (int64_t)1 << 30) ? absmax_units<uint32_t>(src, ld, rows, m, k)
                                                        : absmax_units<uint64_t>(src, ld, rows, m, k);
    const int kt = k - c_begin;
    if (kt > 0) {
        const int64_t total = m * kt;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
            const int64_t r = i / kt;
            mx = fmaxf(mx, fabsf(src[(rows ? rows[r] : r) * ld + c_begin + (i - r * kt)]));
        }
    }
    mx = warp_max(mx);
    uint32_t* bits = reinterpret_cast<uint32_t*>(rec);
    if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(bits, __float_as_uint(mx));   // non-negative floats order like uints
    if (!FINISH) return;
    // the last block to finish turns the absmax into the record
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicAdd(bits + 3, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        __threadfence();
        float amax = __uint_as_float(atomicMax(bits, 0u));
        if (!(amax < 3.0e38f)) amax = 3.0e38f;                  // +inf in the data: keep the record finite
        write_record(rec, fmaxf(amax, floor_));
    }
}

// rec[0] holds a raw absmax (producer kernels raise it with atomic max): complete the record in place
__global__ void finish_record_kernel(float floor_, float* rec) {
    float amax = rec[0];
    if (!(amax < 3.0e38f)) amax = amax != amax ? 0.f : 3.0e38f;
    write_record(rec, fmaxf(amax, floor_));
}

__global__ void bound_record_kernel(float bound, const float* __restrict__ other, float* __restrict__ rec) {
    write_record(rec, other ? fmaxf(bound, other[0]) : bound);
}

// VEC: 16-byte aligned rows and planes -> the [m, ld_planes / 8] matrix of 8-column groups is walked flat: two float4
// in, one 16-byte store per plane, two groups per thread and step in flight (narrow operands keep every lane busy;
// a group that lies in the zero padding only stores).
template <typename I>
__device__ __forceinline__ void split_groups(const float* __restrict__ src, int64_t ld, const int64_t* __restrict__ rows,
                                             int64_t m, int k, float scale, __half* __restrict__ dst, int64_t ldp,
                                             int64_t plane_stride) {
    constexpr int U = 2;
    const I groups = (I)(ldp >> 3);
    const I total = (I)m * groups;
    const I stride = (I)gridDim.x * blockDim.x;
    for (I i = (I)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += U * stride) {
        float x[U][8];
        I row[U];
        int col[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const I j = i + (I)u * stride;
            const bool ok = j < total;
            const I r = ok ? j / groups : 0;
            const int c0 = 8 * (int)(j - r * groups);
            row[u] = r;
            col[u] = ok ? c0 : -1;
#pragma unroll
            for (int q = 0; q < 8; ++q) x[u][q] = 0.f;
            if (ok && c0 < k) {
                const float* s = src + (rows ? rows[r] : (int64_t)r) * ld + c0;
                if (c0 + 8 <= k) {
                    const float4 a = __ldg(reinterpret_cast<const float4*>(s));
                    const float4 b = __ldg(reinterpret_cast<const float4*>(s) + 1);
                    x[u][0] = a.x; x[u][1] = a.y; x[u][2] = a.z; x[u][3] = a.w;
                    x[u][4] = b.x; x[u][5] = b.y; x[u][6] = b.z; x[u][7] = b.w;
                } else {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        if (c0 + q < k) x[u][q] = __ldg(s + q);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (col[u] < 0) continue;
            __align__(16) __half h[8], l[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) split_f16(x[u][q] * scale, h[q], l[q]);
            __half* hrow = dst + (int64_t)row[u] * ldp + col[u];
            *reinterpret_cast<uint4*>(hrow) = *reinterpret_cast<const uint4*>(h);
            *reinterpret_cast<uint4*>(hrow + plane_stride) = *reinterpret_cast<const uint4*>(l);
        }
    }
}

template <bool VEC>
__global__ void __launch_bounds__(256) split_planes_kernel(const float* __restrict__ src, int64_t ld,
                                                           const int64_t* __restrict__ rows, int64_t m, int k,
                                                           const float* __restrict__ rec, __half* __restrict__ dst,
                                                           int64_t ldp, int64_t plane_stride) {
    const float scale = __ldg(rec + 1);
    if (VEC) {
        if (m * (ldp >> 3) < (int64_t)1 << 30) split_groups<uint32_t>(src, ld, rows, m, k, scale, dst, ldp, plane_stride);
        else split_groups<uint64_t>(src, ld, rows, m, k, scale, dst, ldp, plane_stride);
    } else {
        const int64_t total = m * ldp;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
            const int64_t r = i / ldp;
            const int c = (int)(i - r * ldp);
            float x = 0.f;
            if (c < k) x = src[(rows ? rows[r] : r) * ld + c] * scale;
            __half h, l;
            split_f16(x, h, l);
            dst[i] = h;
            dst[plane_stride + i] = l;
        }
    }
}

// weight [n, sum(seg_k)] fp32 -> fp16 planes [2][n][sum(ceil64(seg_k))], every segment zero padded to a multiple of
// 64.  Segment i is multiplied by S / a_scale_i so that every product of the GEMM carries the same factor S.
struct PackSegs {
    int n_segments;
    int k[LKG_MAX_SEGMENTS];
    const float* a_rec[LKG_MAX_SEGMENTS];
};
__global__ void seg_absmax_kernel(const float* __restrict__ w, int64_t ldw, int n, int ktot, PackSegs segs,
                                  float* __restrict__ w_rec) {
    float m[LKG_MAX_SEGMENTS] = {0.f, 0.f, 0.f, 0.f};
    const int64_t total = (int64_t)n * ktot;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / ktot;
        int c = (int)(i - r * ktot);
        const float v = fabsf(w[r * ldw + c]);
        int sgm = 0;
        while (sgm < segs.n_segments - 1 && c >= segs.k[sgm]) c -= segs.k[sgm++];
#pragma unroll
        for (int s = 0; s < LKG_MAX_SEGMENTS; ++s)
            if (s == sgm) m[s] = fmaxf(m[s], v == v ? v : 0.f);
    }
    uint32_t* bits = reinterpret_cast<uint32_t*>(w_rec) + 4;
#pragma unroll
    for (int s = 0; s < LKG_MAX_SEGMENTS; ++s) {
        const float x = warp_max(m[s]);
        if ((threadIdx.x & 31) == 0 && x > 0.f) atomicMax(bits + s, __float_as_uint(x));
    }
}
// S = 2^e with max_i (wmax_i / a_scale_i) * S in [2^11, 2^12)
__device__ __forceinline__ float pack_total_scale(const PackSegs& segs, const float* w_rec) {
    float cmax = 0.f;
    for (int s = 0; s < segs.n_segments; ++s) cmax = fmaxf(cmax, w_rec[4 + s] * __ldg(segs.a_rec[s] + 2));
    return ldexpf(1.f, plane_exp(cmax));
}
__global__ void pack_weight_kernel(const float* __restrict__ w, int64_t ldw, int n, PackSegs segs,
                                   __half* __restrict__ dst, int kb, int64_t plane_stride, float* __restrict__ w_rec) {
    const float S = pack_total_scale(segs, w_rec);
    float seg_scale[LKG_MAX_SEGMENTS];
    for (int s = 0; s < LKG_MAX_SEGMENTS; ++s) seg_scale[s] = s < segs.n_segments ? S * __ldg(segs.a_rec[s] + 2) : 0.f;
    const int64_t total = (int64_t)n * kb;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / kb);
        int c = (int)(i - (int64_t)r * kb);
        int src_col = 0;
        float x = 0.f;
        for (int s = 0; s < segs.n_segments; ++s) {
            const int padded = (segs.k[s] + kBK - 1) / kBK * kBK;
            if (c < padded) {
                if (c < segs.k[s]) x = w[(int64_t)r * ldw + src_col + c] * seg_scale[s];
                break;
            }
            c -= padded;
            src_col += segs.k[s];
        }
        __half h, l;
        split_f16(x, h, l);
        dst[i] = h;
        dst[plane_stride + i] = l;
    }
}
// runs after pack_weight_kernel on the same stream: publishes {., S, 1/S} for the GEMM epilogue
__global__ void pack_finalize_kernel(PackSegs segs, float* __restrict__ w_rec) {
    const float S = pack_total_scale(segs, w_rec);
    w_rec[0] = 0.f;
    w_rec[1] = S;
    w_rec[2] = 1.f / S;
}

inline int grid_1d(int64_t n) {
    int64_t b = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

}  // namespace
}  // namespace lkg

using namespace lkg;

namespace lkg {
namespace {
template <bool FINISH>
int launch_absmax(const float* src, int64_t ld, const int64_t* rows, int64_t m, int32_t k, float floor_, float* rec,
                  cudaStream_t stream) {
    if (m > 0 && aligned16(src) && ld % 4 == 0 && k >= 4)
        absmax_kernel<true, FINISH><<<grid_1d(m * (k / 4 + 3) / 4), 256, 0, stream>>>(src, ld, rows, m, k, floor_, rec);
    else
        absmax_kernel<false, FINISH><<<grid_1d(m * k), 256, 0, stream>>>(src, ld, rows, m, k, floor_, rec);
    LKG_LAUNCH_CHECK("absmax_kernel");
    return LKG_OK;
}
}  // namespace
}  // namespace lkg

extern "C" int lkg_scale_from_data(const float* src, int64_t ld, const int64_t* rows, int64_t m, int32_t k,
                                   float floor_, float* rec, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    LKG_REQUIRE(rec && m >= 0 && k > 0 && (m == 0 || src) && floor_ >= 0.f, "bad scale arguments");
    LKG_CUDA(cudaMemsetAsync(rec, 0, LKG_SCALE_FLOATS * sizeof(float), stream));
    return launch_absmax<true>(src, ld, rows, m, k, floor_, rec, stream);
}

extern "C" int lkg_absmax_accumulate(const float* src, int64_t ld, const int64_t* rows, int64_t m, int32_t k,
                                     float* rec, void* stream_) {
    LKG_REQUIRE(rec && m >= 0 && k > 0 && (m == 0 || src), "bad scale arguments");
    if (m == 0) return LKG_OK;
    return launch_absmax<false>(src, ld, rows, m, k, 0.f, rec, (cudaStream_t)stream_);
}

extern "C" int lkg_scale_finish(float floor_, float* rec, void* stream_) {
    LKG_REQUIRE(rec && floor_ >= 0.f, "bad scale arguments");
    finish_record_kernel<<<1, 1, 0, (cudaStream_t)stream_>>>(floor_, rec);
    LKG_LAUNCH_CHECK("finish_record_kernel");
    return LKG_OK;
}

extern "C" int lkg_scale_from_bound(float bound, const float* other, float* rec, void* stream_) {
    LKG_REQUIRE(rec && bound >= 0.f, "bad scale arguments");
    bound_record_kernel<<<1, 1, 0, (cudaStream_t)stream_>>>(bound, other, rec);
    LKG_LAUNCH_CHECK("bound_record_kernel");
    return LKG_OK;
}

extern "C" int lkg_split_planes(const float* src, int64_t ld, const int64_t* rows, int64_t m, int32_t k,
                                const float* rec, uint16_t* planes, int64_t ld_planes, int64_t plane_stride,
                                void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    LKG_REQUIRE(src && rec && planes && m >= 0 && k > 0 && ld_planes >= k && plane_stride >= m * ld_planes,
                "bad split arguments");
    if (m == 0) return LKG_OK;
    if (aligned16(src) && ld % 4 == 0 && aligned16(planes) && ld_planes % 8 == 0 && plane_stride % 8 == 0)
        split_planes_kernel<true><<<grid_1d(m * (ld_planes / 8 + 1) / 2), 256, 0, stream>>>(
            src, ld, rows, m, k, rec, (__half*)planes, ld_planes, plane_stride);
    else
        split_planes_kernel<false><<<grid_1d(m * ld_planes), 256, 0, stream>>>(src, ld, rows, m, k, rec, (__half*)planes,
                                                                            ld_planes, plane_stride);
    LKG_LAUNCH_CHECK("split_planes_kernel");
    return LKG_OK;
}

extern "C" int lkg_packed_weight_cols(const int32_t* seg_k, int32_t n_segments, int32_t* cols) {
    LKG_REQUIRE(seg_k && cols && n_segments >= 1 && n_segments <= LKG_MAX_SEGMENTS, "bad segment list");
    int c = 0;
    for (int s = 0; s < n_segments; ++s) {
        LKG_REQUIRE(seg_k[s] > 0, "bad segment width");
        c += (seg_k[s] + kBK - 1) / kBK * kBK;
    }
    *cols = c;
    return LKG_OK;
}

extern "C" int lkg_pack_weight(const float* w, int64_t ldw, int32_t n, const int32_t* seg_k, int32_t n_segments,
                               const float* const* a_recs, uint16_t* planes, int64_t plane_stride, float* w_rec,
                               void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    int32_t kb = 0;
    if (int rc = lkg_packed_weight_cols(seg_k, n_segments, &kb)) return rc;
    LKG_REQUIRE(w && planes && w_rec && a_recs && n > 0 && plane_stride >= (int64_t)n * kb, "bad pack arguments");
    PackSegs segs{};
    segs.n_segments = n_segments;
    int ktot = 0;
    for (int s = 0; s < n_segments; ++s) {
        LKG_REQUIRE(a_recs[s] != nullptr, "segment %d has no scale record", s);
        segs.k[s] = seg_k[s];
        segs.a_rec[s] = a_recs[s];
        ktot += seg_k[s];
    }
    LKG_CUDA(cudaMemsetAsync(w_rec, 0, LKG_SCALE_FLOATS * sizeof(float), stream));
    seg_absmax_kernel<<<grid_1d((int64_t)n * ktot), 256, 0, stream>>>(w, ldw, n, ktot, segs, w_rec);
    LKG_LAUNCH_CHECK("seg_absmax_kernel");
    pack_weight_kernel<<<grid_1d((int64_t)n * kb), 256, 0, stream>>>(w, ldw, n, segs, (__half*)planes, kb, plane_stride,
                                                                    w_rec);
    LKG_LAUNCH_CHECK("pack_weight_kernel");
    pack_finalize_kernel<<<1, 1, 0, stream>>>(segs, w_rec);
    LKG_LAUNCH_CHECK("pack_finalize_kernel");
    return LKG_OK;
}

extern "C" int lkg_gemm_set_cta_group(int32_t cta_group) {
    LKG_REQUIRE(cta_group >= 0 && cta_group <= 2, "cta_group must be 0 (automatic), 1 or 2");
    g_forced_cg = cta_group;
    return LKG_OK;
}

extern "C" int lkg_linear_fwd_split(const lkg_planes* a, int64_t m, const lkg_planes* b, int32_t n, const float* bias,
                                    int32_t activation, float* out, int64_t ldo, float* out2, int64_t ld2,
                                    int32_t split_col, uint16_t* out_planes, int64_t ld_planes, int64_t plane_stride,
                                    const float* out_rec, void* stream_) {
    LKG_REQUIRE(out && ldo >= (out2 ? split_col : n), "bad linear output");
    LKG_REQUIRE(!out2 || (split_col > 0 && split_col < n && split_col % 4 == 0 && ld2 >= n - split_col),
                "bad split output (split_col %d of %d columns must be a positive multiple of 4)", split_col, n);
    LKG_REQUIRE(!out_planes || out_rec, "out_planes needs a scale record");
    if (m == 0) return LKG_OK;
    TcParams p{};
    p.bias = bias;
    p.act = activation & 0xff;
    p.accumulate = (activation & LKG_ACT_ACCUMULATE) != 0;
    p.out = out;
    p.ldo = ldo;
    p.out2 = out2;
    p.ld2 = ld2;
    p.split_col = split_col;
    p.out_planes = (__half*)out_planes;
    p.ld_planes = ld_planes;
    p.plane_stride = plane_stride;
    p.out_rec = out_rec;
    return launch_tc<kEpiLinear>(p, a, m, b, n, (cudaStream_t)stream_);
}

extern "C" int lkg_linear_fwd(const lkg_planes* a, int64_t m, const lkg_planes* b, int32_t n, const float* bias,
                              int32_t activation, float* out, int64_t ldo, uint16_t* out_planes, int64_t ld_planes,
                              int64_t plane_stride, const float* out_rec, void* stream_) {
    return lkg_linear_fwd_split(a, m, b, n, bias, activation, out, ldo, nullptr, 0, 0, out_planes, ld_planes, plane_stride,
                                out_rec, stream_);
}

extern "C" int lkg_gate_fwd(const lkg_planes* x, int64_t m, const lkg_planes* w_pair, const float* bias_pair,
                            int32_t dim, const float* x_ent, int64_t ld_ent, float* out, int64_t ldo,
                            uint16_t* out_planes, int64_t ld_planes, int64_t plane_stride, const float* out_rec,
                            float* gz_out, int64_t ld_gz, void* stream_) {
    LKG_REQUIRE(bias_pair && x_ent && out && dim > 0 && ldo >= dim, "bad gate arguments");
    LKG_REQUIRE(!gz_out || ld_gz >= 2 * dim, "bad gz_out stride");
    LKG_REQUIRE(!out_planes || out_rec, "out_planes needs a scale record");
    if (m == 0) return LKG_OK;
    TcParams p{};
    p.bias = bias_pair;
    p.out = out;
    p.ldo = ldo;
    p.out_planes = (__half*)out_planes;
    p.ld_planes = ld_planes;
    p.plane_stride = plane_stride;
    p.out_rec = out_rec;
    p.x_ent = x_ent;
    p.ld_ent = ld_ent;
    p.gz_out = gz_out;
    p.ld_gz = ld_gz;
    return launch_tc<kEpiGate>(p, x, m, w_pair, 2 * dim, (cudaStream_t)stream_);
}

extern "C" int lkg_score_rank(const lkg_planes* heads, int64_t n_heads, const lkg_planes* tails, int64_t n_tails,
                              const float* thr, int32_t* above, int32_t* band_cnt, int32_t* band, int32_t band_cap,
                              void* stream_) {
    LKG_REQUIRE(n_heads >= 0 && n_tails >= 0 && n_tails < (1ll << 31), "bad rank shape");
    if (n_heads == 0 || n_tails == 0) return LKG_OK;
    LKG_REQUIRE(thr && above && band_cnt && band && band_cap > 0 && aligned16(thr) == aligned16(thr), "null argument");
    LKG_REQUIRE((reinterpret_cast<uintptr_t>(thr) & 7u) == 0, "thr must be 8-byte aligned");
    LKG_REQUIRE(heads && tails && heads->n_segments == 1 && tails->n_segments == 1 && heads->k[0] == tails->k[0],
                "rank operands must be single-segment planes of equal width");
    TcParams p{};
    p.rank_thr = thr;
    p.rank_above = above;
    p.rank_band_cnt = band_cnt;
    p.rank_band = band;
    p.rank_band_cap = band_cap;
    p.m_fastest = 1;    // all head tiles of one tail tile run together: the tails stream through L2 once
    return launch_tc<kEpiRank>(p, heads, n_heads, tails, (int)n_tails, (cudaStream_t)stream_);
}

extern "C" int lkg_score(const lkg_planes* heads, int64_t n_heads, const lkg_planes* tails, int64_t n_tails,
                         float* scores, int64_t ld_scores, uint32_t* minmax_dev, void* stream_) {
    LKG_REQUIRE(scores && n_heads >= 0 && n_tails >= 0 && n_tails < (1ll << 31) && ld_scores >= n_tails, "bad score shape");
    if (n_heads == 0 || n_tails == 0) return LKG_OK;
    LKG_REQUIRE(heads && tails && heads->n_segments == 1 && tails->n_segments == 1 && heads->k[0] == tails->k[0],
                "score operands must be single-segment planes of equal width");
    TcParams p{};
    p.out = scores;
    p.ldo = ld_scores;
    p.minmax = minmax_dev;
    p.m_fastest = 1;    // all head tiles of one tail tile run together: the big operand streams through L2 once
    return launch_tc<kEpiScore>(p, heads, n_heads, tails, (int)n_tails, (cudaStream_t)stream_);
}
