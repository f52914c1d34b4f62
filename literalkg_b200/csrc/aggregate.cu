// One aggregator layer, forward: CSR SpMM fused with the combine, LeakyReLU, LayerNorm, dropout mask
// and the L2-normalised copy for the concat buffer.
//
// Replaces Aggregator.forward + residual_connection (model.py:90-164) and the F.normalize of
// model.py:305.  The reference runs cuSPARSE SpMM, then 2-4 dense N x d x d GEMMs, ~10 elementwise
// kernels and a LayerNorm, each a full pass over N x d.  Here one warp owns kRows head rows:
//   phase 1  side = sum_j A[row, j] * ego[col_j]   128-bit streaming gathers, kUnroll neighbours in flight
//   phase 2  u-vectors (side | ego+side | ego | ego*side) staged in shared memory, then the folded
//            combine  o = u @ P + r[row]  with lane = output channel (P lives in shared memory)
//   phase 3  leaky / add / LayerNorm / mask / L2 normalise, all in registers + warp shuffles
// Folding (host side, DESIGN.md section 4): linear(res(hi)) = hi @ P + h0 @ Q + c, P = (1-a) M W^T.
// HBM bound: algorithmic bytes = nnz*(4 col + 4 val + 4 d_in) + N*(4 d_in + 8 + r terms + 2*4*d_out).
#include <cuda_fp16.h>

#include "common.cuh"

namespace lkg {
namespace {

constexpr int kRows = 2;  // head rows per warp per step (P is read from shared memory once per kRows rows)

enum Mode { kOneTerm = 0, kTwoTerms = 1, kBi = 2, kBiZ = 3 /* bi-interaction with a pre-projected sum term */ };
static_assert(kOneTerm == LKG_AGG_MODE_ONE_TERM && kTwoTerms == LKG_AGG_MODE_TWO_TERMS && kBi == LKG_AGG_MODE_BI &&
                  kBiZ == LKG_AGG_MODE_BI_Z, "lkg_agg_mode mirrors the kernel modes");

struct AggParams {
    lkg_graph g;
    const float* a_val;
    const float* ego;
    int64_t ld_ego;
    int d_in, d_out, nvec;
    const float* p0;   // term 0 matrix [d_in, d_out]
    const float* p1;   // term 1 matrix (kTwoTerms: side matrix; kBi: product matrix)
    int sum_ego;       // term 0 vector: 1 -> ego + side, 0 -> side   (kOneTerm / kBi);  kTwoTerms: term0 = ego, term1 = side
    const float* r1;
    const float* r2;
    int64_t ld_r;
    const float* ln_w;
    const float* ln_b;
    const float* mask;
    float* x_out;
    int64_t ld_x;
    float* xn_out;
    int64_t ld_xn;
    __half* xn_planes;          // optional scaled hi/lo fp16 copy of xn (operand of the linear_gat tensor-core GEMM)
    int64_t ld_planes, plane_stride;
    const float* xn_rec;        // its scale record (|xn| <= 1)
    int* counter;
    int p_stride;      // padded row stride (floats) of P in shared memory
    const float* z;    // kBiZ: pre-projected neighbour term, z = ego @ Pb ([N, d_out], row stride ld_z): the sum path
    int64_t ld_z;      //       o1 = r1 + sum_j A[row, j] z[col_j] needs no combine matrix in the kernel
    int64_t local_row_base;   // r1 / r2 / mask / xn_out / xn_planes are indexed by (row - local_row_base): the
                              // row partition's local buffers; ego and x_out are indexed by the global row
    float* o_out;      // training: saved pre-activations [o1 | o2] per local row (nullable), row stride ld_o
    int64_t ld_o;
    float* side_out;   // training: saved side = A @ ego per local row (nullable), row stride ld_side
    int64_t ld_side;
    int n_solo;        // narrow kernel: leading rows of row_order that are scheduled one per warp
};

template <int S, int NC, int MODE>
__global__ void __launch_bounds__(512, 1) aggregate_kernel(AggParams p) {
    extern __shared__ __align__(16) float smem[];
    constexpr int UNROLL = S == 1 ? 8 : 4;   // narrow rows: more neighbours in flight
    constexpr int NT = MODE == kOneTerm ? 1 : 2;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    const int d_in = p.d_in, d_out = p.d_out, nvec = p.nvec;
    const int ps = p.p_stride;
    float* sp0 = smem;
    float* sp1 = smem + (size_t)d_in * ps;
    float* stage = smem + (size_t)NT * d_in * ps + (size_t)warp * (kRows * NT * d_in);

    // stage the folded matrices once per CTA
    for (int i = threadIdx.x; i < d_in * d_out; i += blockDim.x) {
        const int d = i / d_out, c = i - d * d_out;
        sp0[d * ps + c] = p.p0[i];
        if (NT == 2) sp1[d * ps + c] = p.p1[i];
    }
    __syncthreads();
    (void)nwarps;

    const int n = (int)(p.g.row_end - p.g.row_begin);      // rows of the partition, taken in row_order
    const int row0 = (int)p.g.row_begin;
    auto row_of = [&](int i) { return p.g.row_order ? __ldg(p.g.row_order + i) : row0 + i; };
    for (;;) {
        int base = 0;
        if (lane == 0) base = atomicAdd(p.counter, kRows);
        base = __shfl_sync(kFull, base, 0);
        if (base >= n) break;

        // ---- phase 1: SpMM + u-vector staging ------------------------------------------------
#pragma unroll
        for (int rr = 0; rr < kRows; ++rr) {
            if (base + rr >= n) break;
            const int row = row_of(base + rr);
            float4 side[S];
#pragma unroll
            for (int s = 0; s < S; ++s) side[s] = make_float4(0, 0, 0, 0);
            const int u0 = p.g.rowptr[row], u1 = p.g.rowptr[row + 1];
            for (int u = u0; u < u1; u += UNROLL) {
                int cl[UNROLL];
                float av[UNROLL];
#pragma unroll
                for (int j = 0; j < UNROLL; ++j) {
                    const bool live = u + j < u1;
                    cl[j] = live ? __ldg(p.g.col + u + j) : -1;
                    av[j] = live ? __ldg(p.a_val + u + j) : 0.f;
                }
                float4 x[UNROLL][S];
#pragma unroll
                for (int j = 0; j < UNROLL; ++j) {
                    const float* src = p.ego + (int64_t)(cl[j] < 0 ? 0 : cl[j]) * p.ld_ego;
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        const int v = lane + 32 * s;
                        x[j][s] = (cl[j] >= 0 && v < nvec) ? ldg_stream4(src + 4 * v) : make_float4(0, 0, 0, 0);
                    }
                }
#pragma unroll
                for (int j = 0; j < UNROLL; ++j) {
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        side[s].x = fmaf(av[j], x[j][s].x, side[s].x);
                        side[s].y = fmaf(av[j], x[j][s].y, side[s].y);
                        side[s].z = fmaf(av[j], x[j][s].z, side[s].z);
                        side[s].w = fmaf(av[j], x[j][s].w, side[s].w);
                    }
                }
            }
            const float* erow = p.ego + (int64_t)row * p.ld_ego;
            float* st = stage + rr * NT * d_in;
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const int v = lane + 32 * s;
                if (v < nvec) {
                    const float4 sd = side[s];
                    if (p.side_out)
                        reinterpret_cast<float4*>(p.side_out + (row - p.local_row_base) * p.ld_side)[v] = sd;
                    float4 eg = make_float4(0, 0, 0, 0);
                    if (MODE != kOneTerm || p.sum_ego) eg = __ldg(reinterpret_cast<const float4*>(erow) + v);
                    float4 t0, t1;
                    if (MODE == kTwoTerms) {
                        t0 = eg;
                        t1 = sd;
                    } else {
                        t0 = p.sum_ego ? make_float4(eg.x + sd.x, eg.y + sd.y, eg.z + sd.z, eg.w + sd.w) : sd;
                        t1 = make_float4(eg.x * sd.x, eg.y * sd.y, eg.z * sd.z, eg.w * sd.w);
                    }
                    reinterpret_cast<float4*>(st)[v] = t0;
                    if (NT == 2) reinterpret_cast<float4*>(st + d_in)[v] = t1;
                }
            }
        }
        __syncwarp();

        // ---- phase 2: folded combine, lane = output channel ----------------------------------
        float acc1[kRows][NC], acc2[kRows][NC];
#pragma unroll
        for (int rr = 0; rr < kRows; ++rr) {
            const int64_t lrow = row_of(min(base + rr, n - 1)) - p.local_row_base;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                acc1[rr][c] = (ch < d_out && p.r1) ? __ldg(p.r1 + lrow * p.ld_r + ch) : 0.f;
                acc2[rr][c] = (MODE == kBi && ch < d_out && p.r2) ? __ldg(p.r2 + lrow * p.ld_r + ch) : 0.f;
            }
        }
        for (int d4 = 0; d4 < nvec; ++d4) {
            float4 u[kRows][NT];
#pragma unroll
            for (int rr = 0; rr < kRows; ++rr)
#pragma unroll
                for (int t = 0; t < NT; ++t)
                    u[rr][t] = reinterpret_cast<const float4*>(stage + (rr * NT + t) * d_in)[d4];
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                const int chc = ch < d_out ? ch : 0;
                float w0[4], w1[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    w0[i] = sp0[(4 * d4 + i) * ps + chc];
                    w1[i] = NT == 2 ? sp1[(4 * d4 + i) * ps + chc] : 0.f;
                }
#pragma unroll
                for (int rr = 0; rr < kRows; ++rr) {
                    float a = acc1[rr][c];
                    a = fmaf(u[rr][0].x, w0[0], a);
                    a = fmaf(u[rr][0].y, w0[1], a);
                    a = fmaf(u[rr][0].z, w0[2], a);
                    a = fmaf(u[rr][0].w, w0[3], a);
                    if (MODE == kTwoTerms) {
                        a = fmaf(u[rr][1].x, w1[0], a);
                        a = fmaf(u[rr][1].y, w1[1], a);
                        a = fmaf(u[rr][1].z, w1[2], a);
                        a = fmaf(u[rr][1].w, w1[3], a);
                    }
                    acc1[rr][c] = a;
                    if (MODE == kBi) {
                        float b = acc2[rr][c];
                        b = fmaf(u[rr][1].x, w1[0], b);
                        b = fmaf(u[rr][1].y, w1[1], b);
                        b = fmaf(u[rr][1].z, w1[2], b);
                        b = fmaf(u[rr][1].w, w1[3], b);
                        acc2[rr][c] = b;
                    }
                }
            }
        }
        __syncwarp();   // staging buffer is reused by the next step

        // ---- phase 3: activation, LayerNorm, mask, L2 normalise --------------------------------
#pragma unroll
        for (int rr = 0; rr < kRows; ++rr) {
            if (base + rr >= n) break;
            const int row = row_of(base + rr);
            const int64_t lrow = row - p.local_row_base;
            float emb[NC];
            float s1 = 0.f;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                if (p.o_out && ch < d_out) {
                    p.o_out[lrow * p.ld_o + ch] = acc1[rr][c];
                    if (MODE == kBi) p.o_out[lrow * p.ld_o + d_out + ch] = acc2[rr][c];
                }
                float e = leaky(acc1[rr][c]);
                if (MODE == kBi) e += leaky(acc2[rr][c]);
                emb[c] = ch < d_out ? e : 0.f;
                s1 += emb[c];
            }
            const float mean = warp_sum(s1) / (float)d_out;
            float s2 = 0.f;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                const float dlt = ch < d_out ? emb[c] - mean : 0.f;
                s2 = fmaf(dlt, dlt, s2);
            }
            const float rstd = rsqrtf(warp_sum(s2) / (float)d_out + 1e-5f);
            float sq = 0.f;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                float x = 0.f;
                if (ch < d_out) {
                    x = (emb[c] - mean) * rstd * __ldg(p.ln_w + ch) + __ldg(p.ln_b + ch);
                    if (p.mask) x *= __ldg(p.mask + lrow * d_out + ch);
                    p.x_out[(int64_t)row * p.ld_x + ch] = x;
                }
                emb[c] = x;
                sq = fmaf(x, x, sq);
            }
            if (p.xn_out || p.xn_planes) {
                const float inv = 1.f / fmaxf(sqrtf(warp_sum(sq)), 1e-12f);
                const float pscale = p.xn_planes ? __ldg(p.xn_rec + 1) : 1.f;
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    const int ch = lane + 32 * c;
                    if (ch < d_out) {
                        const float xn = emb[c] * inv;
                        if (p.xn_out) p.xn_out[lrow * p.ld_xn + ch] = xn;
                        if (p.xn_planes) {
                            const float xs = xn * pscale;
                            const __half h = __float2half_rn(xs);
                            const __half l = __float2half_rn(xs - __half2float(h));
                            p.xn_planes[lrow * p.ld_planes + ch] = h;
                            p.xn_planes[p.plane_stride + lrow * p.ld_planes + ch] = l;
                        }
                    }
                }
            }
        }
    }
}

// ---- narrow rows (d_in = 16 / 32 / 64): LPR = d_in / 4 lanes own one head row, 32 / LPR rows per warp ----
// Layers >= 2 gather 128-byte rows: with one warp per row 24 of the 32 lanes idle and the kernel is latency
// bound (ncu r01a: 0.9 TB/s, 22 % occupancy).  Here every lane holds one float4 of its row; the neighbour list is
// loaded LPR entries at a time (one coalesced load per group) and broadcast with width-LPR shuffles, all LPR
// gathers of a chunk in flight together.  Batches come from the degree-sorted row_order, so the rows that share
// a warp have similar lengths; a batch whose heaviest row exceeds kCoopDegree is processed row by row with the
// whole warp splitting the row's neighbour list (then summed across groups).  The folded combine keeps the
// u-vectors in registers: lane gl owns the output channels [4 gl, 4 gl + 4) (+ 4 LPR i), u[d] arrives by shuffle
// from the lane that holds it and P rows are read from shared memory as float4.
constexpr int kCoopDegree = 96;

__device__ __forceinline__ float4 f4_fma(float a, float4 w, float4 c) {
    return make_float4(fmaf(a, w.x, c.x), fmaf(a, w.y, c.y), fmaf(a, w.z, c.z), fmaf(a, w.w, c.w));
}

// RB = rows per lane group and unit (register blocking of the combine): a unit is RB batches of RPW rows, walked one
// after the other in phase 1 (same neighbour order as with RB = 1: results are bit identical) and TOGETHER in phase 2,
// where every 16-byte read of a combine matrix then feeds RB rows.  ncu r02v: 103 M of the kernel's 137 M LSU
// wavefronts were those reads (one per 4 FMAs and quarter warp) and the LSU pipe was 77 % busy at 1.89 GHz -- inside
// the pass, where the GPU sits at its power cap, the kernel ran 30 % slower than alone.
template <int LPR, int MODE, int CPL, int RB, int MINB>   // CPL = float4 channel chunks per lane = ceil(d_out / (4 LPR))
__global__ void __launch_bounds__(256, MINB) aggregate_narrow_kernel(AggParams p) {
    extern __shared__ __align__(16) float smem[];
    constexpr int RPW = 32 / LPR;
    constexpr int NT = MODE == kOneTerm ? 1 : 2;
    constexpr int U = LPR < 8 ? LPR : 8;
    const int lane = threadIdx.x & 31;
    const int grp = lane / LPR, gl = lane % LPR;
    const int d_in = 4 * LPR, d_out = p.d_out;
    float* sp0 = smem;
    float* sp1 = smem + d_in * d_out;
    for (int i = threadIdx.x; i < d_in * d_out; i += blockDim.x) {
        sp0[i] = p.p0[i];
        if (NT == 2) sp1[i] = p.p1[i];
    }
    __syncthreads();

    const int n = (int)(p.g.row_end - p.g.row_begin);
    const int row0 = (int)p.g.row_begin;
    // Work units from the dynamic counter: the first n_solo rows of the (degree sorted) order are so long that one
    // of them is a unit of its own -- the whole warp walks its neighbour list -- instead of four of them queueing
    // behind each other in one warp (a 4 096-neighbour row is ~128 dependent round trips); after them, RB * RPW rows
    // each: batch rr of a unit = rows [base + rr RPW, base + (rr + 1) RPW) of the order, one per lane group.
    const int n_solo = RPW > 1 ? min(p.n_solo, n) : 0;
    // The header of a unit is a chain of dependent round trips (counter -> row_order -> rowptr) in front of the index
    // and gather round trips; with ~20 neighbours per row that chain was most of a unit's time (ncu r02: long
    // scoreboard on top, DRAM at 37 %).  It is software pipelined: the unit after next is claimed, the next unit's
    // row ids are loaded while this unit gathers and its extents while this unit runs the combine.
    auto claim = [&]() {
        int u = 0;
        if (lane == 0) u = atomicAdd(p.counter, 1);
        return u;                                            // lane 0's value, broadcast where it is used
    };
    auto unit_base = [&](int unit, bool& is_solo) {
        is_solo = unit < n_solo;
        return is_solo ? unit : n_solo + (unit - n_solo) * (RB * RPW);
    };
    auto row_live = [&](int base_, bool solo_, int rr) {
        return solo_ ? (rr == 0 && grp == 0 && base_ < n) : base_ + rr * RPW + grp < n;
    };
    auto unit_row = [&](int base_, int rr, bool live_) {
        const int pos = base_ + rr * RPW + grp;
        return live_ ? (p.g.row_order ? __ldg(p.g.row_order + pos) : row0 + pos) : 0;
    };
    bool solo;
    int base = unit_base(__shfl_sync(kFull, claim(), 0), solo);
    int claimed = claim();
    bool live[RB];
    int row[RB], u0[RB], u1[RB];
#pragma unroll
    for (int rr = 0; rr < RB; ++rr) {
        live[rr] = row_live(base, solo, rr);
        row[rr] = unit_row(base, rr, live[rr]);
    }
#pragma unroll
    for (int rr = 0; rr < RB; ++rr) {
        u0[rr] = live[rr] ? __ldg(p.g.rowptr + row[rr]) : 0;
        u1[rr] = live[rr] ? __ldg(p.g.rowptr + row[rr] + 1) : 0;
    }
    const float* ego_l = p.ego + 4 * gl;
    while (base < n) {
        bool solo_n;
        const int base_n = unit_base(__shfl_sync(kFull, claimed, 0), solo_n);
        bool live_n[RB];
        int row_n[RB];
#pragma unroll
        for (int rr = 0; rr < RB; ++rr) {
            live_n[rr] = row_live(base_n, solo_n, rr);
            row_n[rr] = unit_row(base_n, rr, live_n[rr]);
        }
        claimed = claim();

        // ---- phase 1: side = sum_j A[row, j] * ego[col_j], this lane's float4, batch after batch ------------
        float4 side[RB];
#pragma unroll
        for (int rr = 0; rr < RB; ++rr) {
            side[rr] = make_float4(0, 0, 0, 0);
            int max_deg = u1[rr] - u0[rr];
#pragma unroll
            for (int o = LPR; o < 32; o <<= 1) max_deg = max(max_deg, __shfl_xor_sync(kFull, max_deg, o));
            max_deg = __shfl_sync(kFull, max_deg, 0);
            const bool coop = RPW > 1 && (solo || max_deg > kCoopDegree);
            for (int pass = 0; pass < (coop ? (solo ? 1 : RPW) : 1); ++pass) {
                // group mode: every group walks its own row, LPR neighbours per step; coop mode: the warp walks the
                // row of group `pass`, 32 neighbours per step (group g takes neighbours [g LPR, (g+1) LPR) of the step)
                const int b0 = coop ? __shfl_sync(kFull, u0[rr], pass * LPR) : u0[rr];
                const int b1 = coop ? __shfl_sync(kFull, u1[rr], pass * LPR) : u1[rr];
                const int my = coop ? lane : gl;
                const int step = coop ? 32 : LPR;
                const int trips = coop ? (b1 - b0 + 31) / 32 : (max_deg + LPR - 1) / LPR;
                float4 acc = make_float4(0, 0, 0, 0);
                // the (column, value) pair of the NEXT step is loaded before the gathers of this one are issued
                int cl_n = -1;
                float av_n = 0.f;
                if (trips > 0 && b0 + my < b1) {
                    cl_n = __ldg(p.g.col + b0 + my);
                    av_n = __ldg(p.a_val + b0 + my);
                }
                for (int it = 0; it < trips; ++it) {
                    const int cl = cl_n;
                    const float av = av_n;
                    const int un = b0 + (it + 1) * step + my;
                    const bool okn = it + 1 < trips && un < b1;
                    cl_n = okn ? __ldg(p.g.col + un) : -1;
                    av_n = okn ? __ldg(p.a_val + un) : 0.f;
#pragma unroll
                    for (int j0 = 0; j0 < LPR; j0 += U) {
                        float4 x[U];
                        float a[U];
#pragma unroll
                        for (int j = 0; j < U; ++j) {
                            const int c = __shfl_sync(kFull, cl, j0 + j, LPR);
                            a[j] = __shfl_sync(kFull, av, j0 + j, LPR);
                            x[j] = c >= 0 ? ldg_stream4(ego_l + (int64_t)c * p.ld_ego) : make_float4(0, 0, 0, 0);
                        }
#pragma unroll
                        for (int j = 0; j < U; ++j) acc = f4_fma(a[j], x[j], acc);
                    }
                }
                if (coop) {
#pragma unroll
                    for (int o = LPR; o < 32; o <<= 1) {
                        acc.x += __shfl_xor_sync(kFull, acc.x, o);
                        acc.y += __shfl_xor_sync(kFull, acc.y, o);
                        acc.z += __shfl_xor_sync(kFull, acc.z, o);
                        acc.w += __shfl_xor_sync(kFull, acc.w, o);
                    }
                    if (grp == pass) side[rr] = acc;
                } else {
                    side[rr] = acc;
                }
            }
        }

        // the next unit's extents: in flight during the combine
        int u0_n[RB], u1_n[RB];
#pragma unroll
        for (int rr = 0; rr < RB; ++rr) {
            u0_n[rr] = live_n[rr] ? __ldg(p.g.rowptr + row_n[rr]) : 0;
            u1_n[rr] = live_n[rr] ? __ldg(p.g.rowptr + row_n[rr] + 1) : 0;
        }

        // ---- phase 2: folded combine in registers, all RB batches per matrix read ----------------------------
        int64_t lrow[RB];
        float4 t0[RB], t1[RB];
        float4 acc1[RB][CPL], acc2[RB][CPL];
#pragma unroll
        for (int rr = 0; rr < RB; ++rr) {
            lrow[rr] = row[rr] - p.local_row_base;
            float4 eg = make_float4(0, 0, 0, 0);
            if (live[rr] && (MODE != kOneTerm || p.sum_ego))
                eg = __ldg(reinterpret_cast<const float4*>(p.ego + (int64_t)row[rr] * p.ld_ego) + gl);
            const float4 sd = side[rr];
            if (p.side_out && live[rr]) reinterpret_cast<float4*>(p.side_out + lrow[rr] * p.ld_side)[gl] = sd;
            if (MODE == kTwoTerms) {
                t0[rr] = eg;
                t1[rr] = sd;
            } else {
                t0[rr] = p.sum_ego ? make_float4(eg.x + sd.x, eg.y + sd.y, eg.z + sd.z, eg.w + sd.w) : sd;
                t1[rr] = make_float4(eg.x * sd.x, eg.y * sd.y, eg.z * sd.z, eg.w * sd.w);
            }
#pragma unroll
            for (int i = 0; i < CPL; ++i) {
                const int ch = 4 * (gl + LPR * i);
                const bool okc = live[rr] && ch < d_out;
                acc1[rr][i] = (okc && p.r1) ? __ldg(reinterpret_cast<const float4*>(p.r1 + lrow[rr] * p.ld_r + ch))
                                            : make_float4(0, 0, 0, 0);
                acc2[rr][i] = (MODE == kBi && okc && p.r2)
                                  ? __ldg(reinterpret_cast<const float4*>(p.r2 + lrow[rr] * p.ld_r + ch))
                                  : make_float4(0, 0, 0, 0);
            }
        }
#pragma unroll 2
        for (int sl = 0; sl < LPR; ++sl) {
            float a0[RB][4], a1[RB][4];
#pragma unroll
            for (int rr = 0; rr < RB; ++rr) {
                a0[rr][0] = __shfl_sync(kFull, t0[rr].x, sl, LPR);
                a0[rr][1] = __shfl_sync(kFull, t0[rr].y, sl, LPR);
                a0[rr][2] = __shfl_sync(kFull, t0[rr].z, sl, LPR);
                a0[rr][3] = __shfl_sync(kFull, t0[rr].w, sl, LPR);
                if (NT == 2) {
                    a1[rr][0] = __shfl_sync(kFull, t1[rr].x, sl, LPR);
                    a1[rr][1] = __shfl_sync(kFull, t1[rr].y, sl, LPR);
                    a1[rr][2] = __shfl_sync(kFull, t1[rr].z, sl, LPR);
                    a1[rr][3] = __shfl_sync(kFull, t1[rr].w, sl, LPR);
                } else {
                    a1[rr][0] = a1[rr][1] = a1[rr][2] = a1[rr][3] = 0.f;
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int d = 4 * sl + c;
#pragma unroll
                for (int i = 0; i < CPL; ++i) {
                    const int ch = 4 * (gl + LPR * i);
                    if (ch < d_out) {
                        const float4 w0 = *reinterpret_cast<const float4*>(sp0 + d * d_out + ch);
#pragma unroll
                        for (int rr = 0; rr < RB; ++rr) acc1[rr][i] = f4_fma(a0[rr][c], w0, acc1[rr][i]);
                        if (NT == 2) {
                            const float4 w1 = *reinterpret_cast<const float4*>(sp1 + d * d_out + ch);
#pragma unroll
                            for (int rr = 0; rr < RB; ++rr) {
                                if (MODE == kTwoTerms) acc1[rr][i] = f4_fma(a1[rr][c], w1, acc1[rr][i]);
                                else acc2[rr][i] = f4_fma(a1[rr][c], w1, acc2[rr][i]);
                            }
                        }
                    }
                }
            }
        }

        // ---- phase 3: activation, LayerNorm, mask, L2 normalise (group-wide reductions), batch after batch ---
#pragma unroll
        for (int rr = 0; rr < RB; ++rr) {
            const bool lv = live[rr];
            const int64_t lr = lrow[rr];
            float4 emb[CPL];
            float s1 = 0.f;
#pragma unroll
            for (int i = 0; i < CPL; ++i) {
                const int ch = 4 * (gl + LPR * i);
                const float4 o1 = acc1[rr][i], o2 = acc2[rr][i];
                if (p.o_out && lv && ch < d_out) {
                    *reinterpret_cast<float4*>(p.o_out + lr * p.ld_o + ch) = o1;
                    if (MODE == kBi) *reinterpret_cast<float4*>(p.o_out + lr * p.ld_o + d_out + ch) = o2;
                }
                float4 e = make_float4(leaky(o1.x), leaky(o1.y), leaky(o1.z), leaky(o1.w));
                if (MODE == kBi) {
                    e.x += leaky(o2.x);
                    e.y += leaky(o2.y);
                    e.z += leaky(o2.z);
                    e.w += leaky(o2.w);
                }
                if (ch >= d_out) e = make_float4(0, 0, 0, 0);
                emb[i] = e;
                s1 += (e.x + e.y) + (e.z + e.w);
            }
#pragma unroll
            for (int o = LPR / 2; o > 0; o >>= 1) s1 += __shfl_xor_sync(kFull, s1, o);
            const float mean = s1 / (float)d_out;
            float s2 = 0.f;
#pragma unroll
            for (int i = 0; i < CPL; ++i) {
                if (4 * (gl + LPR * i) < d_out) {
                    const float dx = emb[i].x - mean, dy = emb[i].y - mean, dz = emb[i].z - mean, dw = emb[i].w - mean;
                    s2 += (dx * dx + dy * dy) + (dz * dz + dw * dw);
                }
            }
#pragma unroll
            for (int o = LPR / 2; o > 0; o >>= 1) s2 += __shfl_xor_sync(kFull, s2, o);
            const float rstd = rsqrtf(s2 / (float)d_out + 1e-5f);
            float sq = 0.f;
#pragma unroll
            for (int i = 0; i < CPL; ++i) {
                const int ch = 4 * (gl + LPR * i);
                float4 x = make_float4(0, 0, 0, 0);
                if (ch < d_out) {
                    const float4 lw = __ldg(reinterpret_cast<const float4*>(p.ln_w + ch));
                    const float4 lb = __ldg(reinterpret_cast<const float4*>(p.ln_b + ch));
                    x.x = (emb[i].x - mean) * rstd * lw.x + lb.x;
                    x.y = (emb[i].y - mean) * rstd * lw.y + lb.y;
                    x.z = (emb[i].z - mean) * rstd * lw.z + lb.z;
                    x.w = (emb[i].w - mean) * rstd * lw.w + lb.w;
                    if (p.mask && lv) {
                        const float4 mk = __ldg(reinterpret_cast<const float4*>(p.mask + lr * d_out + ch));
                        x.x *= mk.x; x.y *= mk.y; x.z *= mk.z; x.w *= mk.w;
                    }
                    if (lv) *reinterpret_cast<float4*>(p.x_out + (int64_t)row[rr] * p.ld_x + ch) = x;
                }
                emb[i] = x;
                sq += (x.x * x.x + x.y * x.y) + (x.z * x.z + x.w * x.w);
            }
            if (p.xn_out || p.xn_planes) {
#pragma unroll
                for (int o = LPR / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(kFull, sq, o);
                const float inv = 1.f / fmaxf(sqrtf(sq), 1e-12f);
                const float pscale = p.xn_planes ? __ldg(p.xn_rec + 1) : 1.f;
#pragma unroll
                for (int i = 0; i < CPL; ++i) {
                    const int ch = 4 * (gl + LPR * i);
                    if (ch < d_out && lv) {
                        const float4 xn = make_float4(emb[i].x * inv, emb[i].y * inv, emb[i].z * inv, emb[i].w * inv);
                        if (p.xn_out) *reinterpret_cast<float4*>(p.xn_out + lr * p.ld_xn + ch) = xn;
                        if (p.xn_planes) {
                            const float v[4] = {xn.x * pscale, xn.y * pscale, xn.z * pscale, xn.w * pscale};
                            __align__(8) __half h[4], l[4];
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                h[c] = __float2half_rn(v[c]);
                                l[c] = __float2half_rn(v[c] - __half2float(h[c]));
                            }
                            __half* hp = p.xn_planes + lr * p.ld_planes + ch;
                            *reinterpret_cast<uint2*>(hp) = *reinterpret_cast<const uint2*>(h);
                            *reinterpret_cast<uint2*>(hp + p.plane_stride) = *reinterpret_cast<const uint2*>(l);
                        }
                    }
                }
            }
        }
        base = base_n;
        solo = solo_n;
#pragma unroll
        for (int rr = 0; rr < RB; ++rr) {
            live[rr] = live_n[rr];
            row[rr] = row_n[rr];
            u0[rr] = u0_n[rr];
            u1[rr] = u1_n[rr];
        }
    }
}

template <int LPR, int MODE, int CPL, int RB, int MINB = 1>
int launch_narrow_rb(const AggParams& p, cudaStream_t stream) {
    auto kern = aggregate_narrow_kernel<LPR, MODE, CPL, RB, MINB>;
    const size_t smem = (size_t)(MODE == kOneTerm ? 1 : 2) * (4 * LPR) * p.d_out * sizeof(float);
    LKG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    LKG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem));
    if (per_sm < 1) LKG_FAIL(LKG_ERR_UNSUPPORTED, "narrow aggregate kernel does not fit (smem %zu)", smem);
    kern<<<sm_count() * per_sm, 256, smem, stream>>>(p);
    LKG_LAUNCH_CHECK("aggregate_narrow_kernel");
    return LKG_OK;
}

template <int LPR, int MODE, int CPL>
int launch_narrow(const AggParams& p, cudaStream_t stream) {
    // Two rows per lane group where the accumulators of both fit (one channel chunk per lane), held to 64 registers
    // (4 CTAs / SM; 32 bytes of spill).  Measured per call inside the cfg 3 pass, same box: 0.75 ms with one row per
    // group (48 registers, 5 CTAs), 0.65 ms with two (80 registers, 3 CTAs), 0.62 vs 0.82 ms for 64 vs 80 registers.
    if constexpr (CPL == 1 && LPR >= 8) return launch_narrow_rb<LPR, MODE, CPL, 2, 4>(p, stream);
    else return launch_narrow_rb<LPR, MODE, CPL, 1>(p, stream);
}

template <int LPR, int CPL>
int dispatch_narrow(int mode, const AggParams& p, cudaStream_t stream) {
    switch (mode) {
        case kOneTerm: return launch_narrow<LPR, kOneTerm, CPL>(p, stream);
        case kTwoTerms: return launch_narrow<LPR, kTwoTerms, CPL>(p, stream);
        default: return launch_narrow<LPR, kBi, CPL>(p, stream);
    }
}

// ---- wide rows (layer 1, d_in = 300): gathered rows stream through a per-warp shared-memory ring --------------------
// Same streaming structure as the attention update (attn.cu): the neighbour list is loaded 32 entries at a time in
// one coalesced step, the 1 200-byte neighbour rows arrive by cp.async.bulk (one TMA-unit copy per row, kRing in
// flight per warp, no registers held), and the schedule record, first index chunk and own ego row of the NEXT row
// are prefetched while the current row streams.  The register-staged kernel above keeps 4 rows in flight behind a
// rowptr -> col -> gather chain of dependent round trips (ncu r01: 66 % of the HBM peak, long_scoreboard on top).
// The folded combine reads the u-vectors (side | ego+side | ego*side) from a per-warp staging buffer and P from
// shared memory in [d/4][channel][4] order: one 16-byte load per matrix feeds four FMAs.
constexpr int kStreamWarps = 16;
// neighbour rows in flight per warp: what fits next to the P tiles (kBiZ keeps one matrix instead of two)
__host__ __device__ constexpr int stream_ring(int mode) { return mode == kBiZ ? 6 : 4; }  // 8 fits (228 KB) but measures slower: 5.95 vs 5.36 ms

template <int S, int NC, int MODE>
__global__ void __launch_bounds__(kStreamWarps * 32, 1) aggregate_stream_kernel(AggParams p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    constexpr bool Z = MODE == kBiZ;                            // sum term pre-projected: only the product term is combined
    constexpr int NT = (MODE == kOneTerm || Z) ? 1 : 2;
    constexpr int kRing = stream_ring(MODE);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int d_in = p.d_in, d_out = p.d_out, nvec = p.nvec;
    const int cpad = 32 * NC;                                   // padded channel count of the P tiles
    const uint32_t row_bytes = (uint32_t)nvec * 16u;
    const uint32_t z_bytes = Z ? (uint32_t)d_out * 4u : 0u;      // a ring slot = neighbour row (+ its z row)
    const uint32_t slot_bytes = row_bytes + z_bytes;
    // layout: P0 [nvec][cpad][4] | P1 | per warp { ring kRing x slot_bytes | stage NT x row_bytes } | barriers
    float4* sp0 = reinterpret_cast<float4*>(smem_raw);
    float4* sp1 = sp0 + (size_t)nvec * cpad;
    const size_t warp_bytes = (size_t)kRing * slot_bytes + (size_t)NT * row_bytes;
    uint8_t* warp_base = smem_raw + (size_t)NT * nvec * cpad * 16 + (size_t)warp * warp_bytes;
    uint8_t* ring = warp_base;
    float4* stage = reinterpret_cast<float4*>(warp_base + (size_t)kRing * slot_bytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)NT * nvec * cpad * 16 +
                                                 (size_t)kStreamWarps * warp_bytes) + warp * kRing;
    // [ego row | z row] stored back to back in one table (model.py lays the gate output and its projection out like
    // that): ONE bulk copy per neighbour instead of two, and the 128-byte z row rides in the DRAM page of its ego row
    const bool zcontig = Z && p.z == p.ego + d_in && p.ld_z == p.ld_ego;
    auto issue = [&](uint32_t slot, int col) {                   // one elected lane: row copy (+ z copy), one barrier
        uint8_t* dst = ring + slot * slot_bytes;
        if (Z && zcontig) {
            ring_issue(dst, p.ego + (int64_t)col * p.ld_ego, slot_bytes, &bars[slot]);
        } else if (Z) {
            ring_expect(&bars[slot], slot_bytes);
            ring_copy(dst, p.ego + (int64_t)col * p.ld_ego, row_bytes, &bars[slot]);
            ring_copy(dst + row_bytes, p.z + (int64_t)col * p.ld_z, z_bytes, &bars[slot]);
        } else {
            ring_issue(dst, p.ego + (int64_t)col * p.ld_ego, row_bytes, &bars[slot]);
        }
    };
    for (int i = threadIdx.x; i < nvec * cpad; i += blockDim.x) {
        const int d4 = i / cpad, c = i - d4 * cpad;
        float w0[4] = {0, 0, 0, 0}, w1[4] = {0, 0, 0, 0};
        if (c < d_out) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                w0[k] = p.p0[(4 * d4 + k) * d_out + c];
                if (NT == 2) w1[k] = p.p1[(4 * d4 + k) * d_out + c];
            }
        }
        sp0[i] = make_float4(w0[0], w0[1], w0[2], w0[3]);
        if (NT == 2) sp1[i] = make_float4(w1[0], w1[1], w1[2], w1[3]);
    }
    if (lane < kRing) ring_bar_init(&bars[lane]);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    const int n_rows = p.g.n_sched > 0 ? (int)p.g.n_sched : (int)(p.g.row_end - p.g.row_begin);   // schedule records
    const int4* sched = reinterpret_cast<const int4*>(p.g.row_sched);
    uint32_t issued = 0, consumed = 0;
    const bool need_ego = MODE != kOneTerm || p.sum_ego;
    const int zvec = d_out >> 2;                                 // float4 per z row

    struct Rec { int row, u0, u1, nseg, ticket, seg; };
    auto fetch_idx = [&]() {
        int i = 0;
        if (lane == 0) i = atomicAdd(p.counter, 1);
        return i;
    };
    auto load_rec = [&](int i) {
        Rec r{0, 0, 0, 0, 0, 0};
        if (i < n_rows) {
            const int4 a = __ldg(sched + 2 * i);
            const int4 b = __ldg(sched + 2 * i + 1);
            r.row = a.x; r.u0 = a.w;
            r.u1 = b.x; r.nseg = b.y; r.ticket = b.z; r.seg = b.w;
        }
        return r;
    };
    struct Head { int col; float val; float4 eg[S]; bool live; };
    auto load_head = [&](const Rec& r, bool live) {
        Head h;
        h.live = live;
        const int cn = min(32, r.u1 - r.u0);
        h.col = (live && lane < cn) ? __ldg(p.g.col + r.u0 + lane) : 0;
        h.val = (live && lane < cn) ? __ldg(p.a_val + r.u0 + lane) : 0.f;
        const float4* erow = reinterpret_cast<const float4*>(p.ego + (int64_t)r.row * p.ld_ego);
#pragma unroll
        for (int s = 0; s < S; ++s) {
            const int v = lane + 32 * s;
            h.eg[s] = (live && need_ego && v < nvec) ? __ldg(erow + v) : make_float4(0, 0, 0, 0);
        }
        return h;
    };

    int idx = __shfl_sync(kFull, fetch_idx(), 0);
    Rec rec = load_rec(idx);
    int idx1 = __shfl_sync(kFull, fetch_idx(), 0);
    Rec rec1 = load_rec(idx1);
    Head head = load_head(rec, idx < n_rows);
    int pre_issued = 0;                              // copies of this row's first chunk issued during the previous row

    while (idx < n_rows) {
        int idx2 = fetch_idx();
        const int row = rec.row, u0 = rec.u0, u1 = rec.u1;
        const int64_t lrow = row - p.local_row_base;
        Rec rec2{0, 0, 0, 0, 0, 0};
        Head head1;
        bool fetched = false;
        auto prefetch_rows = [&]() {                 // with this row's copies in flight: loads of the rows to come
            idx2 = __shfl_sync(kFull, idx2, 0);
            rec2 = load_rec(idx2);
            head1 = load_head(rec1, idx1 < n_rows);
            fetched = true;
        };

        // ---- phase 1: side = sum_j A[row, j] * ego[col_j] ---------------------------------------------------
        float4 side[S];
        float4 zside = make_float4(0, 0, 0, 0);                  // kBiZ: lane q < zvec holds channels [4q, 4q + 4)
#pragma unroll
        for (int s = 0; s < S; ++s) side[s] = make_float4(0, 0, 0, 0);
        for (int c0 = u0; c0 < u1; c0 += 32) {
            const int cn = min(32, u1 - c0);
            int my_col;
            float my_val;
            if (c0 == u0) {
                my_col = head.col; my_val = head.val;
            } else {
                my_col = lane < cn ? __ldg(p.g.col + c0 + lane) : 0;
                my_val = lane < cn ? __ldg(p.a_val + c0 + lane) : 0.f;
            }
            const int first = min(cn, kRing);
            const int done = c0 == u0 ? pre_issued : 0;          // the first chunk's copies may already be in flight
            if (lane >= done && lane < first) {
                issue((issued + lane - done) % kRing, my_col);
            }
            issued += first - done;
            if (!fetched) prefetch_rows();
            for (int e = 0; e < cn; ++e) {
                const float a = __shfl_sync(kFull, my_val, e);
                const uint32_t slot = consumed % kRing;
                ring_wait(&bars[slot], (consumed / kRing) & 1);
                const float4* nrow = reinterpret_cast<const float4*>(ring + slot * slot_bytes);
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    const int v = lane + 32 * s;
                    if (v < nvec) {
                        const float4 x = nrow[v];
                        side[s].x = fmaf(a, x.x, side[s].x);
                        side[s].y = fmaf(a, x.y, side[s].y);
                        side[s].z = fmaf(a, x.z, side[s].z);
                        side[s].w = fmaf(a, x.w, side[s].w);
                    }
                }
                if (Z && lane < zvec) {
                    const float4 x = nrow[nvec + lane];
                    zside.x = fmaf(a, x.x, zside.x);
                    zside.y = fmaf(a, x.y, zside.y);
                    zside.z = fmaf(a, x.z, zside.z);
                    zside.w = fmaf(a, x.w, zside.w);
                }
                ++consumed;
                __syncwarp();                                    // every lane has read the slot before it is refilled
                const int nxt = e + kRing;
                if (nxt < cn) {
                    if (lane == nxt) issue(slot, my_col);
                    ++issued;
                }
            }
        }
        if (!fetched) prefetch_rows();                           // row without neighbours
        // the ring is empty: start the next row's first copies now, they land while this row is combined
        pre_issued = 0;
        if (idx1 < n_rows) {
            pre_issued = min(kRing, min(32, rec1.u1 - rec1.u0));
            if (lane < pre_issued) issue((issued + lane) % kRing, head1.col);
            issued += pre_issued;
        }

        // ---- segmented row: park this piece's partial sums; the piece that arrives last adds them up (in segment
        //      order: the result does not depend on which warp that is) and finishes the row ------------------------
        bool finish = true;
        if (rec.nseg > 0) {
            float4* slot = reinterpret_cast<float4*>(p.g.seg_scratch +
                                                     ((int64_t)rec.ticket * LKG_MAX_SEGS + rec.seg) * p.g.seg_stride);
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const int v = lane + 32 * s;
                if (v < nvec) __stcg(slot + v, side[s]);
            }
            if (Z && lane < zvec) __stcg(slot + nvec + lane, zside);
            __threadfence();
            __syncwarp();
            int t = 0;
            if (lane == 0) {
                t = atomicAdd(p.g.seg_tickets + rec.ticket, 1);
                if (t == rec.nseg - 1) p.g.seg_tickets[rec.ticket] = 0;    // ready for the next launch
            }
            t = __shfl_sync(kFull, t, 0);
            finish = t == rec.nseg - 1;
            if (finish) {
                __threadfence();
#pragma unroll
                for (int s = 0; s < S; ++s) side[s] = make_float4(0, 0, 0, 0);
                zside = make_float4(0, 0, 0, 0);
                for (int q = 0; q < rec.nseg; ++q) {
                    const float4* src = reinterpret_cast<const float4*>(
                        p.g.seg_scratch + ((int64_t)rec.ticket * LKG_MAX_SEGS + q) * p.g.seg_stride);
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        const int v = lane + 32 * s;
                        if (v < nvec) {
                            const float4 x = __ldcg(src + v);
                            side[s].x += x.x; side[s].y += x.y; side[s].z += x.z; side[s].w += x.w;
                        }
                    }
                    if (Z && lane < zvec) {
                        const float4 x = __ldcg(src + nvec + lane);
                        zside.x += x.x; zside.y += x.y; zside.z += x.z; zside.w += x.w;
                    }
                }
            }
        }

        // ---- phase 2: u-vectors to the staging buffer, folded combine with lane = output channel -------------
        if (finish) {
#pragma unroll
        for (int s = 0; s < S; ++s) {
            const int v = lane + 32 * s;
            if (v < nvec) {
                const float4 sd = side[s], eg = head.eg[s];
                if (p.side_out) reinterpret_cast<float4*>(p.side_out + lrow * p.ld_side)[v] = sd;
                float4 t0, t1;
                if (Z) {
                    t0 = make_float4(eg.x * sd.x, eg.y * sd.y, eg.z * sd.z, eg.w * sd.w);
                    t1 = t0;
                } else if (MODE == kTwoTerms) {
                    t0 = eg;
                    t1 = sd;
                } else {
                    t0 = p.sum_ego ? make_float4(eg.x + sd.x, eg.y + sd.y, eg.z + sd.z, eg.w + sd.w) : sd;
                    t1 = make_float4(eg.x * sd.x, eg.y * sd.y, eg.z * sd.z, eg.w * sd.w);
                }
                stage[v] = t0;
                if (NT == 2) stage[nvec + v] = t1;
            }
        }
        __syncwarp();
        float acc1[NC], acc2[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const int ch = lane + 32 * c;
            // kBiZ: acc1 accumulates the product path (r2 + (ego * side) @ P2); the sum path is r1 + zside
            const float* rp = Z ? p.r2 : p.r1;
            acc1[c] = (ch < d_out && rp) ? __ldg(rp + lrow * p.ld_r + ch) : 0.f;
            acc2[c] = (MODE == kBi && ch < d_out && p.r2) ? __ldg(p.r2 + lrow * p.ld_r + ch) : 0.f;
            if (Z) {
                const int src = (ch >> 2) & 31;
                const float zx = __shfl_sync(kFull, zside.x, src), zy = __shfl_sync(kFull, zside.y, src);
                const float zz = __shfl_sync(kFull, zside.z, src), zw = __shfl_sync(kFull, zside.w, src);
                const int comp = ch & 3;
                const float zv = comp == 0 ? zx : (comp == 1 ? zy : (comp == 2 ? zz : zw));
                acc2[c] = ((ch < d_out && p.r1) ? __ldg(p.r1 + lrow * p.ld_r + ch) : 0.f) + zv;
            }
        }
#pragma unroll 5
        for (int d4 = 0; d4 < nvec; ++d4) {
            const float4 ua = stage[d4];
            float4 ub = make_float4(0, 0, 0, 0);
            if (NT == 2) ub = stage[nvec + d4];
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const float4 w0 = sp0[d4 * cpad + lane + 32 * c];
                float x = acc1[c];
                x = fmaf(ua.x, w0.x, x);
                x = fmaf(ua.y, w0.y, x);
                x = fmaf(ua.z, w0.z, x);
                x = fmaf(ua.w, w0.w, x);
                if (NT == 2) {
                    const float4 w1 = sp1[d4 * cpad + lane + 32 * c];
                    if (MODE == kTwoTerms) {
                        x = fmaf(ub.x, w1.x, x);
                        x = fmaf(ub.y, w1.y, x);
                        x = fmaf(ub.z, w1.z, x);
                        x = fmaf(ub.w, w1.w, x);
                    } else {
                        float y = acc2[c];
                        y = fmaf(ub.x, w1.x, y);
                        y = fmaf(ub.y, w1.y, y);
                        y = fmaf(ub.z, w1.z, y);
                        y = fmaf(ub.w, w1.w, y);
                        acc2[c] = y;
                    }
                }
                acc1[c] = x;
            }
        }
        __syncwarp();   // the staging buffer is reused by the next row

        // ---- phase 3: activation, LayerNorm, mask, L2 normalise ------------------------------------------------
        {
            float emb[NC];
            float s1 = 0.f;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                if (p.o_out && ch < d_out) {     // kBiZ: acc1 is the product path (o2), acc2 the sum path (o1)
                    p.o_out[lrow * p.ld_o + (Z ? d_out : 0) + ch] = acc1[c];
                    if (MODE == kBi || Z) p.o_out[lrow * p.ld_o + (Z ? 0 : d_out) + ch] = acc2[c];
                }
                float e = leaky(acc1[c]);
                if (MODE == kBi || Z) e += leaky(acc2[c]);
                emb[c] = ch < d_out ? e : 0.f;
                s1 += emb[c];
            }
            const float mean = warp_sum(s1) / (float)d_out;
            float s2 = 0.f;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                const float dlt = ch < d_out ? emb[c] - mean : 0.f;
                s2 = fmaf(dlt, dlt, s2);
            }
            const float rstd = rsqrtf(warp_sum(s2) / (float)d_out + 1e-5f);
            float sq = 0.f;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int ch = lane + 32 * c;
                float x = 0.f;
                if (ch < d_out) {
                    x = (emb[c] - mean) * rstd * __ldg(p.ln_w + ch) + __ldg(p.ln_b + ch);
                    if (p.mask) x *= __ldg(p.mask + lrow * d_out + ch);
                    p.x_out[(int64_t)row * p.ld_x + ch] = x;
                }
                emb[c] = x;
                sq = fmaf(x, x, sq);
            }
            if (p.xn_out || p.xn_planes) {
                const float inv = 1.f / fmaxf(sqrtf(warp_sum(sq)), 1e-12f);
                const float pscale = p.xn_planes ? __ldg(p.xn_rec + 1) : 1.f;
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    const int ch = lane + 32 * c;
                    if (ch < d_out) {
                        const float xn = emb[c] * inv;
                        if (p.xn_out) p.xn_out[lrow * p.ld_xn + ch] = xn;
                        if (p.xn_planes) {
                            const float xs = xn * pscale;
                            const __half h = __float2half_rn(xs);
                            const __half l = __float2half_rn(xs - __half2float(h));
                            p.xn_planes[lrow * p.ld_planes + ch] = h;
                            p.xn_planes[p.plane_stride + lrow * p.ld_planes + ch] = l;
                        }
                    }
                }
            }
        }
        }   // finish
        idx = idx1; rec = rec1; head = head1;
        idx1 = idx2; rec1 = rec2;
    }
}

template <int S, int NC, int MODE>
int launch_stream(const AggParams& p, size_t smem, cudaStream_t stream) {
    auto kern = aggregate_stream_kernel<S, NC, MODE>;
    LKG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<sm_count(), kStreamWarps * 32, smem, stream>>>(p);
    LKG_LAUNCH_CHECK("aggregate_stream_kernel");
    return LKG_OK;
}

template <int S, int NC>
int dispatch_stream(int mode, const AggParams& p, size_t smem, cudaStream_t stream) {
    switch (mode) {
        case kOneTerm: return launch_stream<S, NC, kOneTerm>(p, smem, stream);
        case kTwoTerms: return launch_stream<S, NC, kTwoTerms>(p, smem, stream);
        case kBiZ: return launch_stream<S, NC, kBiZ>(p, smem, stream);
        default: return launch_stream<S, NC, kBi>(p, smem, stream);
    }
}

template <int S, int NC, int MODE>
int launch(const AggParams& p, int threads, size_t smem, cudaStream_t stream) {
    auto kern = aggregate_kernel<S, NC, MODE>;
    LKG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    LKG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1) LKG_FAIL(LKG_ERR_UNSUPPORTED, "aggregate kernel does not fit (smem %zu)", smem);
    const int grid = sm_count() * per_sm;
    kern<<<grid, threads, smem, stream>>>(p);
    LKG_LAUNCH_CHECK("aggregate_kernel");
    return LKG_OK;
}

template <int S, int NC>
int dispatch_mode(int mode, const AggParams& p, int threads, size_t smem, cudaStream_t stream) {
    switch (mode) {
        case kOneTerm: return launch<S, NC, kOneTerm>(p, threads, smem, stream);
        case kTwoTerms: return launch<S, NC, kTwoTerms>(p, threads, smem, stream);
        default: return launch<S, NC, kBi>(p, threads, smem, stream);
    }
}

// ---- which kernel runs a shape ---------------------------------------------------------------------------------
// One host function decides: lkg_aggregate_fwd launches what it returns and lkg_aggregate_supported answers from it,
// so a caller can ask before it builds operands for a mode (the model picks layer 1's pre-projected z path this way).
constexpr size_t kMaxSmem = 227 * 1024;
enum Route { kRouteNone = 0, kRouteNarrow, kRouteStream, kRouteGeneric };
struct AggRoute {
    Route route;
    size_t smem;   // stream / generic kernel: dynamic shared memory
    int warps;     // generic kernel: warps per CTA
};

// narrow_ok: d_in in {16, 32, 64}, d_out % 4 == 0 and every operand the narrow kernel moves as float4 is aligned;
// stream_ok: d_in >= 128 and the plan has a 16-byte aligned row schedule
AggRoute agg_route(int mode, int d_in, int d_out, bool narrow_ok, bool stream_ok) {
    const int nvec = d_in / 4;
    if (mode != kBiZ && narrow_ok) return {kRouteNarrow, 0, 0};
    if (stream_ok) {
        const int slots_w = (nvec + 31) / 32, nc_w = (d_out + 31) / 32;
        // one 128-wide slot: only the z mode (layer 1 of a bi-interaction model at embed_dim 128); the other modes
        // keep the generic kernel there
        const bool instance = (slots_w == 1 && nc_w == 1 && mode == kBiZ) || (slots_w == 2 && nc_w == 1) ||
                              (slots_w == 3 && nc_w == 1) || (slots_w == 3 && nc_w == 2) || (slots_w == 4 && nc_w == 1);
        const int nt = (mode == kOneTerm || mode == kBiZ) ? 1 : 2;
        const size_t z_bytes = mode == kBiZ ? (size_t)d_out * 4 : 0;
        const size_t smem = (size_t)nt * nvec * 32 * nc_w * 16 +
                            (size_t)kStreamWarps * (stream_ring(mode) * (nvec * 16 + z_bytes) + (size_t)nt * nvec * 16) +
                            kStreamWarps * stream_ring(mode) * 8;
        if (instance && smem <= kMaxSmem) return {kRouteStream, smem, 0};
    }
    if (mode == kBiZ) return {kRouteNone, 0, 0};           // only the stream kernel gathers z
    const int nt = mode == kOneTerm ? 1 : 2;
    const size_t p_bytes = (size_t)nt * d_in * ((d_out + 3) / 4 * 4) * sizeof(float);
    const size_t stage_per_warp = (size_t)kRows * nt * d_in * sizeof(float);
    int warps = 16;
    while (warps > 4 && p_bytes + warps * stage_per_warp > 200 * 1024) warps /= 2;
    const size_t smem = p_bytes + warps * stage_per_warp;
    if (smem > kMaxSmem) return {kRouteNone, smem, warps};
    return {kRouteGeneric, smem, warps};
}

}  // namespace
}  // namespace lkg

using namespace lkg;

extern "C" int lkg_aggregate_workspace_bytes(size_t* bytes) {
    LKG_REQUIRE(bytes != nullptr, "bytes is null");
    *bytes = 256;
    return LKG_OK;
}

extern "C" int lkg_aggregate_fwd(const lkg_graph* g, const float* a_values, const float* ego, int64_t ld_ego,
                                 int32_t d_in, int32_t d_out, const float* pa, const float* pb, const float* p2,
                                 const float* r1, const float* r2, int64_t ld_r, const float* ln_weight,
                                 const float* ln_bias, const float* drop_mask, float* x_out, int64_t ld_x,
                                 float* xn_out, int64_t ld_xn, uint16_t* xn_planes, int64_t ld_planes,
                                 int64_t plane_stride, const float* xn_rec, int64_t local_row_base, const float* z,
                                 int64_t ld_z, float* o_out, int64_t ld_o, float* side_out, int64_t ld_side,
                                 void* workspace, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    LKG_REQUIRE(g && ego && (pb || z) && ln_weight && ln_bias && x_out && workspace, "null argument");
    LKG_REQUIRE(!z || (p2 && !pa && !pb && d_out % 4 == 0 && ld_z % 4 == 0 && aligned16(z) && d_in >= 128 && g->row_sched),
                "a pre-projected sum term (z) needs the bi-interaction product matrix p2, no pa / pb, wide rows and a "
                "plan with a row schedule");
    LKG_REQUIRE(g->nnz == 0 || a_values != nullptr, "a_values is null");
    LKG_REQUIRE(!xn_planes || xn_rec, "xn_planes needs a scale record");
    LKG_REQUIRE(g->row_begin >= 0 && g->row_begin <= g->row_end && g->row_end <= g->n_entities, "bad row range");
    LKG_REQUIRE(d_in > 0 && d_in % 4 == 0, "d_in must be a positive multiple of 4 (got %d)", d_in);
    LKG_REQUIRE(ld_ego % 4 == 0 && aligned16(ego), "ego rows must be 16-byte aligned");
    LKG_REQUIRE(d_out > 0, "d_out must be positive");
    LKG_REQUIRE(!(p2 && pa && pa != pb), "bi-interaction takes one shared sum matrix (pa == pb or pa NULL)");
    if (d_in > 512) LKG_FAIL(LKG_ERR_UNSUPPORTED, "aggregate d_in %d > 512", d_in);
    if (d_out > 64) LKG_FAIL(LKG_ERR_UNSUPPORTED, "aggregate d_out %d > 64", d_out);

    AggParams p{};
    p.g = *g;
    p.a_val = a_values;
    p.ego = ego;
    p.ld_ego = ld_ego;
    p.d_in = d_in;
    p.d_out = d_out;
    p.nvec = d_in / 4;
    int mode;
    p.z = z;
    p.ld_z = ld_z;
    if (z) {
        mode = kBiZ;
        p.p0 = p2;
        p.p1 = nullptr;
        p.sum_ego = 0;
    } else if (p2) {
        mode = kBi;
        p.p0 = pb;
        p.p1 = p2;
        p.sum_ego = pa != nullptr;
    } else if (pa && pa != pb) {
        mode = kTwoTerms;
        p.p0 = pa;
        p.p1 = pb;
        p.sum_ego = 0;
    } else {
        mode = kOneTerm;
        p.p0 = pb;
        p.p1 = nullptr;
        p.sum_ego = pa != nullptr;
    }
    p.r1 = r1;
    p.r2 = r2;
    p.ld_r = ld_r;
    p.ln_w = ln_weight;
    p.ln_b = ln_bias;
    p.mask = drop_mask;
    p.x_out = x_out;
    p.ld_x = ld_x;
    p.xn_out = xn_out;
    p.ld_xn = ld_xn;
    p.xn_planes = reinterpret_cast<__half*>(xn_planes);
    p.xn_rec = xn_rec;
    p.ld_planes = ld_planes;
    p.plane_stride = plane_stride;
    p.local_row_base = local_row_base;
    LKG_REQUIRE(!o_out || (ld_o % 4 == 0 && aligned16(o_out)), "o_out rows must be 16-byte aligned");
    LKG_REQUIRE(!side_out || (ld_side % 4 == 0 && aligned16(side_out)), "side_out rows must be 16-byte aligned");
    LKG_REQUIRE(g->n_sched == 0 || !g->seg_tickets ||
                    (g->seg_scratch && g->seg_stride % 4 == 0 && g->seg_stride >= d_in + d_out && aligned16(g->seg_scratch)),
                "the plan's segment scratch is too small for d_in %d + d_out %d", d_in, d_out);
    p.o_out = o_out;
    p.ld_o = ld_o;
    p.side_out = side_out;
    p.ld_side = ld_side;
    p.n_solo = g->row_order ? (int)g->n_solo_rows : 0;
    p.counter = static_cast<int*>(workspace);
    // lane c reads sp[d * ps + c]: any stride is conflict free for 32 consecutive channels; pad to a
    // multiple of 4 floats to keep rows 16-byte aligned
    p.p_stride = (d_out + 3) / 4 * 4;
    // narrow rows: LPR lanes per row (needs 16-byte aligned rows everywhere the kernel moves float4 / 8-byte halves)
    const bool narrow_ok =
        (d_in == 16 || d_in == 32 || d_in == 64) && d_out % 4 == 0 && aligned16(x_out) && ld_x % 4 == 0 &&
        (!xn_out || (aligned16(xn_out) && ld_xn % 4 == 0)) && (!r1 || (aligned16(r1) && ld_r % 4 == 0)) &&
        (!r2 || (aligned16(r2) && ld_r % 4 == 0)) && aligned16(ln_weight) && aligned16(ln_bias) &&
        (!drop_mask || aligned16(drop_mask)) &&
        (!xn_planes || ((reinterpret_cast<uintptr_t>(xn_planes) & 7u) == 0 && ld_planes % 4 == 0 && plane_stride % 4 == 0));
    // wide rows with a schedule: the shared-memory ring kernel
    const bool stream_ok = d_in >= 128 && g->row_sched && aligned16(g->row_sched);
    const AggRoute rt = agg_route(mode, d_in, d_out, narrow_ok, stream_ok);
    if (rt.route == kRouteNone) {                            // refused before anything is enqueued
        if (z) LKG_FAIL(LKG_ERR_UNSUPPORTED, "aggregate with a pre-projected sum term: d_in %d d_out %d not supported",
                        d_in, d_out);
        LKG_FAIL(LKG_ERR_UNSUPPORTED, "aggregate shapes d_in %d d_out %d need %zu bytes of shared memory (%zu fit)",
                 d_in, d_out, rt.smem, kMaxSmem);
    }
    LKG_CUDA(cudaMemsetAsync(p.counter, 0, sizeof(int), stream));
    if (rt.route == kRouteNarrow) {
        const int chunks = d_out / 4;
#define LKG_NARROW_CASE(LL, CC) \
    if (d_in == 4 * LL && (chunks + LL - 1) / LL == CC) return dispatch_narrow<LL, CC>(mode, p, stream);
        LKG_NARROW_CASE(4, 1) LKG_NARROW_CASE(4, 2) LKG_NARROW_CASE(4, 3) LKG_NARROW_CASE(4, 4)
        LKG_NARROW_CASE(8, 1) LKG_NARROW_CASE(8, 2)
        LKG_NARROW_CASE(16, 1)
#undef LKG_NARROW_CASE
    }
    if (rt.route == kRouteStream) {
        const int slots_w = (p.nvec + 31) / 32, nc_w = (d_out + 31) / 32;
        if (slots_w == 1 && nc_w == 1) return launch_stream<1, 1, kBiZ>(p, rt.smem, stream);
        if (slots_w == 2 && nc_w == 1) return dispatch_stream<2, 1>(mode, p, rt.smem, stream);
        if (slots_w == 3 && nc_w == 1) return dispatch_stream<3, 1>(mode, p, rt.smem, stream);
        if (slots_w == 3 && nc_w == 2) return dispatch_stream<3, 2>(mode, p, rt.smem, stream);
        if (slots_w == 4 && nc_w == 1) return dispatch_stream<4, 1>(mode, p, rt.smem, stream);
    }
    if (rt.route == kRouteGeneric) {
        const int threads = rt.warps * 32;
        const int slots = (p.nvec + 31) / 32;
        const int nc = (d_out + 31) / 32;
#define LKG_AGG_CASE(SS, CC) \
    if (slots == SS && nc == CC) return dispatch_mode<SS, CC>(mode, p, threads, rt.smem, stream);
        LKG_AGG_CASE(1, 1) LKG_AGG_CASE(2, 1) LKG_AGG_CASE(3, 1) LKG_AGG_CASE(4, 1)
        LKG_AGG_CASE(1, 2) LKG_AGG_CASE(2, 2) LKG_AGG_CASE(3, 2) LKG_AGG_CASE(4, 2)
#undef LKG_AGG_CASE
    }
    LKG_FAIL(LKG_ERR_UNSUPPORTED, "aggregate: no kernel instance for d_in %d d_out %d", d_in, d_out);
}

extern "C" int lkg_aggregate_supported(int32_t d_in, int32_t d_out, int32_t mode, int32_t* ok) {
    LKG_REQUIRE(ok != nullptr, "ok is null");
    LKG_REQUIRE(mode >= LKG_AGG_MODE_ONE_TERM && mode <= LKG_AGG_MODE_BI_Z, "unknown aggregate mode %d", mode);
    *ok = 0;
    if (d_in <= 0 || d_in % 4 != 0 || d_in > 512 || d_out <= 0 || d_out > 64) return LKG_OK;
    if (mode == LKG_AGG_MODE_BI_Z && (d_in < 128 || d_out % 4 != 0)) return LKG_OK;
    const bool narrow_ok = (d_in == 16 || d_in == 32 || d_in == 64) && d_out % 4 == 0;
    *ok = agg_route(mode, d_in, d_out, narrow_ok, d_in >= 128).route != kRouteNone;
    return LKG_OK;
}
