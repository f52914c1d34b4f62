// Backward of the full-graph embedding pass: what loss.backward() runs in the reference's pre_training /
// fine_tuning modes (main.py:121-124, 222-226 -> autograd through gat_embeddings, model.py:298-314).
//
// The reference's autograd replays, per layer, a sparse.mm backward (A^T @ grad), 2-4 dense GEMM backwards
// and ~10 elementwise backwards, each a full pass over N x d.  Here the backward of one layer is
//   layer_bwd_rows   LayerNorm / dropout-mask / LeakyReLU / L2-normalise backward of a row, in registers
//   spmm_coo         out += A^T X as a segmented reduction over the transposed COO list (equal nnz per
//                    worker: a tail with 10^5 in-edges costs what 10^5 separate entries cost)
//   bi_bwd_rows      the product path of the bi-interaction aggregator (d_out -> d_in expansion in the kernel)
// plus the tensor-core GEMM engine (gemm_tc.cu) for the N x k x d products and the tensor-core X^T Y reduction
// (xty_tc.cu) for the parameter gradients.  All HBM bound.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include "common.cuh"

namespace lkg {
namespace {

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// ---- transposed plan ---------------------------------------------------------------------------------------
__global__ void nnz_rows_kernel(const int32_t* __restrict__ rowptr, int64_t n, int64_t nnz, int32_t* __restrict__ rows,
                                int32_t* __restrict__ iota) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz) return;
    int64_t lo = 0, hi = n;                       // rowptr[lo] <= i < rowptr[hi]
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(rowptr + mid) <= i) lo = mid; else hi = mid;
    }
    rows[i] = (int32_t)lo;
    iota[i] = (int32_t)i;
}

__global__ void gather_i32_kernel(const int32_t* __restrict__ src, const int32_t* __restrict__ idx, int64_t n,
                                  int32_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __ldg(src + __ldg(idx + i));
}

size_t transpose_cub_bytes(int64_t nnz) {
    size_t a = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (int32_t*)nullptr, (int32_t*)nullptr, (int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)nnz, 0, 32);
    return a;
}

// ---- out += M X over a COO list sorted by output row ------------------------------------------------------------
struct SpmmParams {
    const int32_t* seg;    // [nnz] output row of every entry, non-decreasing
    const int32_t* src;    // [nnz] gathered row of X
    const int32_t* perm;   // [nnz] index of the entry's value (nullable: identity)
    const float* vals;
    int64_t nnz;
    const float* x;
    int64_t ldx;
    float* out;
    int64_t ldo;
    int nvec;              // float4 per row
    int chunk;             // entries per worker
};

// A worker = LPR lanes, each holding S float4 of the row.  It reduces the entries [w chunk, (w + 1) chunk): runs of
// equal output row are summed in registers; a run that lies entirely inside the worker's range is added to the
// output with a plain read-modify-write (no other worker touches that row), a run cut by a range boundary with a
// vector atomic.
template <int LPR, int S>
__global__ void __launch_bounds__(256) spmm_coo_kernel(SpmmParams p) {
    constexpr int U = 4;
    const int lane = threadIdx.x & 31;
    const int gl = lane % LPR;
    const unsigned gmask = LPR == 32 ? kFull : (((1u << LPR) - 1u) << ((lane / LPR) * LPR));
    const int64_t worker = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    const int64_t u0 = worker * p.chunk;
    if (u0 >= p.nnz) return;                               // whole groups leave together
    const int64_t u1 = min(u0 + (int64_t)p.chunk, p.nnz);
    const bool head_open = u0 > 0 && __ldg(p.seg + u0 - 1) == __ldg(p.seg + u0);
    int cur = __ldg(p.seg + u0);
    bool first = true;
    float4 acc[S];
#pragma unroll
    for (int s = 0; s < S; ++s) acc[s] = make_float4(0, 0, 0, 0);

    auto flush = [&](bool atomic) {
#pragma unroll
        for (int s = 0; s < S; ++s) {
            const int v = gl + LPR * s;
            if (v < p.nvec) {
                float4* dst = reinterpret_cast<float4*>(p.out + (int64_t)cur * p.ldo) + v;
                if (atomic) {
                    atomicAdd(dst, acc[s]);
                } else {
                    float4 o = *dst;
                    o.x += acc[s].x; o.y += acc[s].y; o.z += acc[s].z; o.w += acc[s].w;
                    *dst = o;
                }
            }
            acc[s] = make_float4(0, 0, 0, 0);
        }
    };

    for (int64_t c0 = u0; c0 < u1; c0 += LPR) {
        const int64_t u = c0 + gl;
        const bool ok = u < u1;
        const int my_seg = ok ? __ldg(p.seg + u) : -1;
        const int my_src = ok ? __ldg(p.src + u) : 0;
        const float my_val = ok ? __ldg(p.vals + (p.perm ? __ldg(p.perm + u) : (int)u)) : 0.f;
        const int cn = (int)min((int64_t)LPR, u1 - c0);
        for (int j0 = 0; j0 < cn; j0 += U) {
            float4 x[U][S];
            int sg[U];
            float a[U];
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const int e = (j0 + j) % LPR;
                const bool live = j0 + j < cn;
                const int sj = __shfl_sync(gmask, my_src, e, LPR);
                sg[j] = __shfl_sync(gmask, my_seg, e, LPR);
                a[j] = __shfl_sync(gmask, my_val, e, LPR);
                const float* row = p.x + (int64_t)sj * p.ldx;
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    const int v = gl + LPR * s;
                    x[j][s] = (live && v < p.nvec) ? ldg_stream4(row + 4 * v) : make_float4(0, 0, 0, 0);
                }
            }
#pragma unroll
            for (int j = 0; j < U; ++j) {
                if (j0 + j < cn) {
                    if (sg[j] != cur) {
                        flush(first && head_open);
                        first = false;
                        cur = sg[j];
                    }
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        acc[s].x = fmaf(a[j], x[j][s].x, acc[s].x);
                        acc[s].y = fmaf(a[j], x[j][s].y, acc[s].y);
                        acc[s].z = fmaf(a[j], x[j][s].z, acc[s].z);
                        acc[s].w = fmaf(a[j], x[j][s].w, acc[s].w);
                    }
                }
            }
        }
    }
    const bool tail_open = u1 < p.nnz && __ldg(p.seg + u1) == cur;
    flush((first && head_open) || tail_open);
}

template <int LPR, int S>
int launch_spmm(const SpmmParams& p, cudaStream_t stream) {
    const int64_t workers = (p.nnz + p.chunk - 1) / p.chunk;
    const int64_t threads = workers * LPR;
    const int64_t blocks = (threads + 255) / 256;
    if (blocks > 0x7fffffff) LKG_FAIL(LKG_ERR_UNSUPPORTED, "spmm: too many blocks");
    spmm_coo_kernel<LPR, S><<<(unsigned)blocks, 256, 0, stream>>>(p);
    LKG_LAUNCH_CHECK("spmm_coo_kernel");
    return LKG_OK;
}

// Producer-side scale records: a kernel that writes a gradient matrix raises rec[0] (the bits of a non-negative
// float order like unsigned integers) so that no separate absmax pass has to re-read what it wrote; lkg_scale_finish
// completes the record.  NaNs are dropped by fmaxf like in the absmax pass.
__device__ __forceinline__ void raise_absmax(float* rec, float mx) {
    mx = warp_max(mx);
    if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(reinterpret_cast<uint32_t*>(rec), __float_as_uint(mx));
}

// ---- row backward of one aggregator layer ----------------------------------------------------------------------
struct LayerBwdParams {
    int64_t n;
    int c, has_o2;
    const float* y;      int64_t ld_y;       // layer output (after LayerNorm and mask)
    const float* o;      int64_t ld_o;       // saved pre-activations [o1 | o2]
    const float* mask;                       // [n, c] nullable
    const float* dy_in;  int64_t ld_dy;      // gradient w.r.t. y from the next layer (nullable)
    const float* dyn;    int64_t ld_dyn;     // gradient w.r.t. normalize(y) from the concat buffer (nullable)
    const float* ln_w;
    float* d_o;          int64_t ld_do;      // out: [do1 | do2]
    float* dgb;                              // out (accumulated): [dgamma (c) | dbeta (c)]
    float* amax;                             // nullable: raw absmax of d_o (scale record under construction)
    float* amax2;                            // nullable: a second record that covers d_o (the buffer it is a part of)
};

// Lanes per row of a layout: the whole warp for WarpChannels, a group of LPR lanes for GroupQuads
template <class L> constexpr int kLanesPerRow = 32;
template <int LPR, int CPL> constexpr int kLanesPerRow<GroupQuads<LPR, CPL>> = LPR;

// a slot's values at q, or fill in each of its channels where !ok
template <class S>
__device__ __forceinline__ typename S::V ld_or(const float* q, bool ok, float fill) {
    typename S::V v;
#pragma unroll
    for (int k = 0; k < (int)(sizeof(v) / sizeof(float)); ++k) S::at(v, k) = fill;
    return ok ? S::ld(q) : v;
}

// One row per LPR lanes over a lane layout of the forward: WarpChannels<1 | 2> (a warp per row, any rows) or
// GroupQuads<8 | 16, 1> (one 16-byte vector of channels per lane, 32 / LPR rows per warp: a warp moves 512 bytes per
// array, not 128; needs c % 4 == 0 and 16-byte aligned rows).  A lane sums its values in sequence, slot after slot and
// channel after channel (not pairwise like the forward's QuadSlot::add).  An absent dy_in adds +0, an absent mask
// multiplies by 1.
template <class L>
__global__ void __launch_bounds__(256) layer_bwd_rows_kernel(LayerBwdParams p) {
    using S = typename L::Slot;
    using V = typename S::V;
    constexpr int N = L::N, W = sizeof(V) / sizeof(float), LPR = kLanesPerRow<L>, RPW = 32 / LPR, CW = LPR * N * W;
    __shared__ float red[8][2][CW];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const L ly{lane % LPR};
    const int C = p.c;
    const float inv_c = 1.f / (float)C;
    V lw[N], dgam[N], dbet[N];
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int k = 0; k < W; ++k) {
            S::at(lw[i], k) = ly.ch(i) < C ? __ldg(p.ln_w + ly.ch(i) + k) : 0.f;
            S::at(dgam[i], k) = S::at(dbet[i], k) = 0.f;
        }
    float amax = 0.f;
    const int64_t units = (p.n + RPW - 1) / RPW;
    for (int64_t unit = (int64_t)blockIdx.x * 8 + warp; unit < units; unit += (int64_t)gridDim.x * 8) {
        const int64_t row = unit * RPW + lane / LPR;
        const bool live = RPW == 1 || row < p.n;         // a unit of one row is in range by the loop bound
        bool ok[N];
        V o1[N], o2[N], y[N], g[N], dyi[N], mk[N], e[N];
        float s1 = 0.f, sq = 0.f, dot = 0.f;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const int ch = ly.ch(i);
            ok[i] = live && ch < C;
            o1[i] = ld_or<S>(p.o + row * p.ld_o + ch, ok[i], 0.f);
            o2[i] = ld_or<S>(p.o + row * p.ld_o + C + ch, ok[i] && p.has_o2, 0.f);
            y[i] = ld_or<S>(p.y + row * p.ld_y + ch, ok[i], 0.f);
            g[i] = ld_or<S>(p.dyn + row * p.ld_dyn + ch, ok[i] && p.dyn, 0.f);
            dyi[i] = ld_or<S>(p.dy_in + row * p.ld_dy + ch, ok[i] && p.dy_in, 0.f);
            mk[i] = ld_or<S>(p.mask + row * C + ch, ok[i] && p.mask, 1.f);
#pragma unroll
            for (int k = 0; k < W; ++k) {
                const float ek = ok[i] ? leaky(S::at(o1[i], k)) + (p.has_o2 ? leaky(S::at(o2[i], k)) : 0.f) : 0.f;
                S::at(e[i], k) = ek;
                s1 += ek;
                sq = fmaf(S::at(y[i], k), S::at(y[i], k), sq);
                dot = fmaf(S::at(g[i], k), S::at(y[i], k), dot);
            }
        }
        const float mean = ly.reduce(s1) * inv_c;
        float s2 = 0.f;
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
            for (int k = 0; k < W; ++k) {
                const float dlt = ok[i] ? S::at(e[i], k) - mean : 0.f;
                s2 = fmaf(dlt, dlt, s2);
            }
        const float rstd = rsqrtf(ly.reduce(s2) * inv_c + 1e-5f);
        sq = ly.reduce(sq);
        dot = ly.reduce(dot);
        const float nrm = sqrtf(sq);
        const float den = fmaxf(nrm, 1e-12f);
        const float k1 = 1.f / den;
        const float k2 = nrm > 1e-12f ? dot / (den * den * den) : 0.f;    // clamp_min passes no gradient below eps
        V dhat[N], ehat[N];
        float m1 = 0.f, m2 = 0.f;
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
            for (int k = 0; k < W; ++k) {
                float dy = S::at(g[i], k) * k1 - S::at(y[i], k) * k2 + S::at(dyi[i], k);
                dy *= S::at(mk[i], k);
                if (!ok[i]) dy = 0.f;
                const float eh = ok[i] ? (S::at(e[i], k) - mean) * rstd : 0.f;
                S::at(dgam[i], k) = fmaf(dy, eh, S::at(dgam[i], k));
                S::at(dbet[i], k) += dy;
                const float dh = dy * S::at(lw[i], k);
                S::at(ehat[i], k) = eh;
                S::at(dhat[i], k) = dh;
                m1 += dh;
                m2 = fmaf(dh, eh, m2);
            }
        m1 = ly.reduce(m1) * inv_c;
        m2 = ly.reduce(m2) * inv_c;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            if (!ok[i]) continue;
            V d1, d2;
#pragma unroll
            for (int k = 0; k < W; ++k) {
                const float de = (S::at(dhat[i], k) - m1 - S::at(ehat[i], k) * m2) * rstd;
                S::at(d1, k) = de * (S::at(o1[i], k) > 0.f ? 1.f : 0.01f);
                S::at(d2, k) = de * (S::at(o2[i], k) > 0.f ? 1.f : 0.01f);
                amax = fmaxf(amax, fabsf(S::at(d1, k)));
                if (p.has_o2) amax = fmaxf(amax, fabsf(S::at(d2, k)));
            }
            S::st(p.d_o + row * p.ld_do + ly.ch(i), d1);
            if (p.has_o2) S::st(p.d_o + row * p.ld_do + C + ly.ch(i), d2);
        }
    }
    if (p.amax || p.amax2) {
        amax = warp_max(amax);
        if (lane == 0 && amax > 0.f) {
            if (p.amax) atomicMax(reinterpret_cast<uint32_t*>(p.amax), __float_as_uint(amax));
            if (p.amax2) atomicMax(reinterpret_cast<uint32_t*>(p.amax2), __float_as_uint(amax));
        }
    }
    // LayerNorm weight / bias gradients: the rows of the warp, then the 8 warps, then one atomic per channel and CTA
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int k = 0; k < W; ++k) {
            float& dg = S::at(dgam[i], k);
            float& db = S::at(dbet[i], k);
#pragma unroll
            for (int o = LPR; o < 32; o <<= 1) {
                dg += __shfl_xor_sync(kFull, dg, o);
                db += __shfl_xor_sync(kFull, db, o);
            }
            if (lane < LPR) {
                red[warp][0][ly.ch(i) + k] = dg;
                red[warp][1][ly.ch(i) + k] = db;
            }
        }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * CW; i += blockDim.x) {
        const int half = i / CW, c = i % CW;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += red[w][half][c];
        if (c < C) atomicAdd(p.dgb + half * C + c, s);
    }
}

// ---- product path of the bi-interaction layer: V = do2 @ P2^T; W = V * x; dx (+)= V * side; xs = x * side ---------
struct BiBwdParams {
    int64_t n;
    int d, c;
    const float* d_o2;   int64_t ld_do;
    const float* p2;                         // [d, c]
    const float* x;      int64_t ld_x;
    const float* side;   int64_t ld_side;
    float* w_out;        int64_t ld_w;
    float* dx;           int64_t ld_dx;
    float* xs_out;       int64_t ld_xs;      // nullable: x * side, the row operand of d P2 = (x * side)^T do2
    int accumulate;
    int ps;                                  // padded row stride of P2 in shared memory (floats), = 4 * odd
    float* xs_amax;                          // nullable: raw absmax of xs_out
};

// One warp per row.  The row's do2 (<= 64 values) is broadcast from shared memory into registers once; lane i then
// produces V[i], V[i + 32], ...: a row of P2 is 16-byte vector loads (stride 4 * odd floats: conflict free for the 8
// lanes of a quarter warp), one FMA per loaded weight.  Shared-memory bandwidth bound: d * c * 4 bytes per row.
template <int CQ>   // float4 chunks of do2: c <= 4 CQ
__global__ void __launch_bounds__(256) bi_bwd_rows_kernel(BiBwdParams p) {
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ps = p.ps;
    float* sp = smem;
    float* sdo = smem + (size_t)p.d * ps + warp * (4 * CQ);
    for (int i = threadIdx.x; i < p.d * ps; i += blockDim.x) {
        const int r = i / ps, c = i - r * ps;
        sp[i] = c < p.c ? p.p2[r * p.c + c] : 0.f;
    }
    __syncthreads();
    float amax = 0.f;
    const int64_t stride = (int64_t)gridDim.x * 8;
    for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < p.n; row += stride) {
        for (int c = lane; c < 4 * CQ; c += 32) sdo[c] = c < p.c ? __ldg(p.d_o2 + row * p.ld_do + c) : 0.f;
        __syncwarp();
        float4 dq[CQ];
#pragma unroll
        for (int q = 0; q < CQ; ++q) dq[q] = reinterpret_cast<const float4*>(sdo)[q];
        __syncwarp();
        // UN elements per lane and step: every global load of the step is in flight before the first FMA (the kernel
        // is otherwise bound by the x / side / dx round trips, not by shared memory)
        constexpr int UN = 5;
        for (int i0 = lane; i0 < p.d; i0 += 32 * UN) {
            float xv[UN], sv[UN], dv[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int i = i0 + 32 * u;
                const bool ok = i < p.d;
                xv[u] = ok ? __ldg(p.x + row * p.ld_x + i) : 0.f;
                sv[u] = ok ? __ldg(p.side + row * p.ld_side + i) : 0.f;
                dv[u] = (ok && p.accumulate) ? p.dx[row * p.ld_dx + i] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int i = i0 + 32 * u;
                if (i < p.d) {
                    const float4* w = reinterpret_cast<const float4*>(sp + i * ps);
                    float v0 = 0.f, v1 = 0.f;
#pragma unroll
                    for (int q = 0; q < CQ; ++q) {
                        const float4 ww = w[q];
                        v0 = fmaf(dq[q].x, ww.x, v0);
                        v1 = fmaf(dq[q].y, ww.y, v1);
                        v0 = fmaf(dq[q].z, ww.z, v0);
                        v1 = fmaf(dq[q].w, ww.w, v1);
                    }
                    const float v = v0 + v1;
                    p.w_out[row * p.ld_w + i] = v * xv[u];
                    if (p.xs_out) {
                        const float xsv = xv[u] * sv[u];
                        p.xs_out[row * p.ld_xs + i] = xsv;
                        amax = fmaxf(amax, fabsf(xsv));
                    }
                    p.dx[row * p.ld_dx + i] = fmaf(v, sv[u], dv[u]);
                }
            }
        }
    }
    if (p.xs_amax) raise_absmax(p.xs_amax, amax);
}

// Narrow rows (d <= 64): LPR = d / 4 lanes per row hold one float4 of x / side / dx each and the row's do2 chunk by
// chunk; do2[c] arrives by shuffle, P2^T is read from shared memory as [c][4 LPR] (the groups of a warp read the same
// 16-byte words: broadcast).  Needs d % 4 == 0, c % 4 == 0, c <= 4 LPR and 16-byte aligned rows.
template <int LPR>
__global__ void __launch_bounds__(256) bi_bwd_rows_vec_kernel(BiBwdParams p) {
    extern __shared__ __align__(16) float smem[];
    constexpr int RPW = 32 / LPR, DW = 4 * LPR;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / LPR, gl = lane % LPR;
    for (int i = threadIdx.x; i < p.c * DW; i += blockDim.x) {
        const int cc = i / DW, di = i - cc * DW;
        smem[i] = di < p.d ? p.p2[di * p.c + cc] : 0.f;
    }
    __syncthreads();
    const int i0 = 4 * gl;
    const bool oki = i0 < p.d;
    const int chunks = p.c >> 2;
    float amax = 0.f;
    const int64_t units = (p.n + RPW - 1) / RPW;
    for (int64_t unit = (int64_t)blockIdx.x * 8 + warp; unit < units; unit += (int64_t)gridDim.x * 8) {
        const int64_t row = unit * RPW + grp;
        const bool live = row < p.n;
        const float4 dq = ld_or<QuadSlot>(p.d_o2 + row * p.ld_do + 4 * gl, live && gl < chunks, 0.f);
        const float4 xv = ld_or<QuadSlot>(p.x + row * p.ld_x + i0, live && oki, 0.f);
        const float4 sv = ld_or<QuadSlot>(p.side + row * p.ld_side + i0, live && oki, 0.f);
        float4 dv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live && oki && p.accumulate) dv = *reinterpret_cast<const float4*>(p.dx + row * p.ld_dx + i0);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int sl = 0; sl < chunks; ++sl) {
            const float a[4] = {__shfl_sync(kFull, dq.x, sl, LPR), __shfl_sync(kFull, dq.y, sl, LPR),
                                __shfl_sync(kFull, dq.z, sl, LPR), __shfl_sync(kFull, dq.w, sl, LPR)};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 w = *reinterpret_cast<const float4*>(smem + (4 * sl + q) * DW + i0);
                v.x = fmaf(a[q], w.x, v.x);
                v.y = fmaf(a[q], w.y, v.y);
                v.z = fmaf(a[q], w.z, v.z);
                v.w = fmaf(a[q], w.w, v.w);
            }
        }
        if (live && oki) {
            *reinterpret_cast<float4*>(p.w_out + row * p.ld_w + i0) = make_float4(v.x * xv.x, v.y * xv.y, v.z * xv.z, v.w * xv.w);
            if (p.xs_out) {
                const float4 xs = make_float4(xv.x * sv.x, xv.y * sv.y, xv.z * sv.z, xv.w * sv.w);
                *reinterpret_cast<float4*>(p.xs_out + row * p.ld_xs + i0) = xs;
                amax = fmaxf(fmaxf(amax, fmaxf(fabsf(xs.x), fabsf(xs.y))), fmaxf(fabsf(xs.z), fabsf(xs.w)));
            }
            *reinterpret_cast<float4*>(p.dx + row * p.ld_dx + i0) =
                make_float4(fmaf(v.x, sv.x, dv.x), fmaf(v.y, sv.y, dv.y), fmaf(v.z, sv.z, dv.z), fmaf(v.w, sv.w, dv.w));
        }
    }
    if (p.xs_amax) raise_absmax(p.xs_amax, amax);
}

// ---- gate backward, elementwise part (gate.py:22-28): out = (1 - z) e + z g ----------------------------------------
//   d_pre[2j] = dh z (1 - g^2)   d_pre[2j+1] = dh (g - e) z (1 - z)   d_ent = dh (1 - z)
// The interleaved (g, z) pairs and d_pre move as one float2 per channel, or as two float4 per quad of channels.
__device__ __forceinline__ void ld_pairs(const float* q, float& g, float& z) {
    const float2 a = __ldg(reinterpret_cast<const float2*>(q));
    g = a.x;
    z = a.y;
}
__device__ __forceinline__ void ld_pairs(const float* q, float4& g, float4& z) {
    const float4 a0 = __ldg(reinterpret_cast<const float4*>(q)), a1 = __ldg(reinterpret_cast<const float4*>(q) + 1);
    g = make_float4(a0.x, a0.z, a1.x, a1.z);
    z = make_float4(a0.y, a0.w, a1.y, a1.w);
}
__device__ __forceinline__ void st_pairs(float* q, float g, float z) { *reinterpret_cast<float2*>(q) = make_float2(g, z); }
__device__ __forceinline__ void st_pairs(float* q, float4 g, float4 z) {
    reinterpret_cast<float4*>(q)[0] = make_float4(g.x, z.x, g.y, z.y);
    reinterpret_cast<float4*>(q)[1] = make_float4(g.z, z.z, g.w, z.w);
}

// Both elementwise backwards walk [n, c / width of the slot] flat: ScalarSlot for any operands, QuadSlot (16-byte units)
// when every row is 16-byte aligned; 32-bit index arithmetic while it fits.
template <class S, typename I>
__global__ void __launch_bounds__(256) gate_bwd_kernel(const float* __restrict__ dh, int64_t ld_dh,
                                                       const float* __restrict__ gz, int64_t ld_gz,
                                                       const float* __restrict__ ent, int64_t ld_ent, int64_t n, int dim,
                                                       float* __restrict__ d_pre, int64_t ld_pre,
                                                       float* __restrict__ d_ent, int64_t ld_de,
                                                       float* __restrict__ pre_amax) {
    using V = typename S::V;
    constexpr int W = sizeof(V) / sizeof(float);
    const I qv = (I)(dim / W), total = (I)n * qv, stride = (I)gridDim.x * blockDim.x;
    float amax = 0.f;
    for (I i = (I)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const I row = i / qv;
        const int j = W * (int)(i - row * qv);
        V g, z, pg, pz, de;
        ld_pairs(gz + (int64_t)row * ld_gz + 2 * j, g, z);
        const V d = S::ld(dh + (int64_t)row * ld_dh + j), e = S::ld(ent + (int64_t)row * ld_ent + j);
#pragma unroll
        for (int k = 0; k < W; ++k) {
            const float dk = S::at(d, k), gk = S::at(g, k), zk = S::at(z, k);
            S::at(pg, k) = dk * zk * (1.f - gk * gk);
            S::at(pz, k) = dk * (gk - S::at(e, k)) * zk * (1.f - zk);
            S::at(de, k) = dk * (1.f - zk);
            amax = fmaxf(amax, fmaxf(fabsf(S::at(pg, k)), fabsf(S::at(pz, k))));
        }
        st_pairs(d_pre + (int64_t)row * ld_pre + 2 * j, pg, pz);
        S::st(d_ent + (int64_t)row * ld_de + j, de);
    }
    if (pre_amax) raise_absmax(pre_amax, amax);
}

// dpre = g * leaky'(out)   (sign(out) == sign of the pre-activation); two units in flight per thread
template <class S, typename I>
__global__ void __launch_bounds__(256) leaky_bwd_kernel(const float* __restrict__ g, int64_t ld_g,
                                                        const float* __restrict__ out, int64_t ld_out, int64_t n, int c,
                                                        float* __restrict__ d, int64_t ld_d, float* __restrict__ d_amax) {
    using V = typename S::V;
    constexpr int W = sizeof(V) / sizeof(float), U = 2;
    const I cv = (I)(c / W), total = (I)n * cv, stride = (I)gridDim.x * blockDim.x;
    float amax = 0.f;
    for (I i = (I)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += U * stride) {
        V gv[U], ov[U];
        I row[U];
        int col[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const I j = i + (I)u * stride;
            const bool ok = j < total;
            row[u] = ok ? j / cv : 0;
            col[u] = ok ? W * (int)(j - row[u] * cv) : -1;
            if (ok) {
                gv[u] = S::ld(g + (int64_t)row[u] * ld_g + col[u]);
                ov[u] = S::ld(out + (int64_t)row[u] * ld_out + col[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (col[u] < 0) continue;
            V v;
#pragma unroll
            for (int k = 0; k < W; ++k) {
                S::at(v, k) = S::at(gv[u], k) * (S::at(ov[u], k) > 0.f ? 1.f : 0.01f);
                amax = fmaxf(amax, fabsf(S::at(v, k)));
            }
            S::st(d + (int64_t)row[u] * ld_d + col[u], v);
        }
    }
    if (d_amax) raise_absmax(d_amax, amax);
}

inline bool rows16(const void* ptr, int64_t ld) { return ptr == nullptr || (aligned16(ptr) && ld % 4 == 0); }

}  // namespace
}  // namespace lkg

using namespace lkg;

extern "C" int lkg_plan_transpose_workspace_bytes(int64_t nnz, size_t* bytes) {
    LKG_REQUIRE(bytes != nullptr && nnz >= 0, "bad arguments");
    const size_t e = (size_t)(nnz > 0 ? nnz : 1);
    *bytes = 2 * align_up(e * 4) + align_up(transpose_cub_bytes(nnz)) + 256;
    return LKG_OK;
}

extern "C" int lkg_plan_transpose(const lkg_graph* g, int32_t* t_tail, int32_t* t_head, int32_t* t_perm,
                                  void* workspace, size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    LKG_REQUIRE(g && t_tail && t_head && t_perm && workspace, "null argument");
    const int64_t nnz = g->nnz;
    size_t need = 0;
    lkg_plan_transpose_workspace_bytes(nnz, &need);
    if (workspace_bytes < need) LKG_FAIL(LKG_ERR_WORKSPACE, "transpose workspace: %zu < %zu", workspace_bytes, need);
    if (nnz == 0) return LKG_OK;
    const size_t e = (size_t)nnz;
    char* base = static_cast<char*>(workspace);
    int32_t* rows = reinterpret_cast<int32_t*>(base);
    int32_t* iota = reinterpret_cast<int32_t*>(base + align_up(e * 4));
    void* cub_tmp = base + 2 * align_up(e * 4);
    size_t cub_bytes = transpose_cub_bytes(nnz);
    const unsigned blocks = (unsigned)((nnz + 255) / 256);
    nnz_rows_kernel<<<blocks, 256, 0, stream>>>(g->rowptr, g->n_entities, nnz, rows, iota);
    LKG_LAUNCH_CHECK("nnz_rows_kernel");
    int bits = 1;
    while (bits < 32 && (1ll << bits) < g->n_entities) ++bits;
    // stable LSD radix sort by tail: inside one tail the entries stay in (head, tail) order
    LKG_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, g->col, t_tail, iota, t_perm, (int)nnz, 0, bits, stream));
    gather_i32_kernel<<<blocks, 256, 0, stream>>>(rows, t_perm, nnz, t_head);
    LKG_LAUNCH_CHECK("gather_i32_kernel");
    return LKG_OK;
}

extern "C" int lkg_spmm_coo(const int32_t* seg, const int32_t* src, const int32_t* perm, const float* vals, int64_t nnz,
                            const float* x, int64_t ldx, int32_t d, float* out, int64_t ldo, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (nnz == 0) return LKG_OK;
    LKG_REQUIRE(seg && src && vals && x && out, "null argument");
    LKG_REQUIRE(d > 0 && d % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && aligned16(x) && aligned16(out),
                "spmm rows must be whole 16-byte vectors (d %d)", d);
    SpmmParams p{seg, src, perm, vals, nnz, x, ldx, out, ldo, d / 4, 0};
    const int nvec = d / 4;
    if (nvec <= 4) { p.chunk = 32; return launch_spmm<4, 1>(p, stream); }
    if (nvec <= 8) { p.chunk = 32; return launch_spmm<8, 1>(p, stream); }
    if (nvec <= 16) { p.chunk = 64; return launch_spmm<16, 1>(p, stream); }
    p.chunk = 128;
    if (nvec <= 32) return launch_spmm<32, 1>(p, stream);
    if (nvec <= 64) return launch_spmm<32, 2>(p, stream);
    if (nvec <= 96) return launch_spmm<32, 3>(p, stream);
    if (nvec <= 128) return launch_spmm<32, 4>(p, stream);
    LKG_FAIL(LKG_ERR_UNSUPPORTED, "spmm: d %d > 512", d);
}

extern "C" int lkg_layer_bwd_rows(int64_t n, int32_t c, int32_t has_o2, const float* y, int64_t ld_y, const float* o,
                                  int64_t ld_o, const float* mask, const float* dy_in, int64_t ld_dy,
                                  const float* dyn, int64_t ld_dyn, const float* ln_weight, float* d_o, int64_t ld_do,
                                  float* dgamma_dbeta, float* amax, float* amax2, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) return LKG_OK;
    LKG_REQUIRE(y && o && ln_weight && d_o && dgamma_dbeta && c > 0, "null argument");
    if (c > 64) LKG_FAIL(LKG_ERR_UNSUPPORTED, "layer backward: d_out %d > 64", c);
    LayerBwdParams p{n, c, has_o2, y, ld_y, o, ld_o, mask, dy_in, ld_dy, dyn, ld_dyn, ln_weight, d_o, ld_do, dgamma_dbeta,
                     amax, amax2};
    const bool vec = c % 4 == 0 && rows16(y, ld_y) && rows16(o, ld_o) && rows16(mask, c) && rows16(dy_in, ld_dy) &&
                     rows16(dyn, ld_dyn) && rows16(d_o, ld_do);
    const int lpr = vec ? (c <= 32 ? 8 : 16) : 32;
    const int64_t units = (n + 32 / lpr - 1) / (32 / lpr);
    const int grid = (int)std::min<int64_t>((units + 7) / 8, (int64_t)sm_count() * 8);
    auto* kernel = vec ? (c <= 32 ? layer_bwd_rows_kernel<GroupQuads<8, 1>> : layer_bwd_rows_kernel<GroupQuads<16, 1>>)
                       : (c <= 32 ? layer_bwd_rows_kernel<WarpChannels<1>> : layer_bwd_rows_kernel<WarpChannels<2>>);
    kernel<<<grid, 256, 0, stream>>>(p);
    LKG_LAUNCH_CHECK("layer_bwd_rows_kernel");
    return LKG_OK;
}

extern "C" int lkg_bi_bwd_rows(int64_t n, int32_t d, int32_t c, const float* d_o2, int64_t ld_do, const float* p2,
                               const float* x, int64_t ld_x, const float* side, int64_t ld_side, float* w_out,
                               int64_t ld_w, float* dx, int64_t ld_dx, int32_t accumulate, float* xs_out, int64_t ld_xs,
                               float* xs_amax, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) return LKG_OK;
    LKG_REQUIRE(d_o2 && p2 && x && side && w_out && dx && d > 0 && c > 0, "null argument");
    if (c > 64) LKG_FAIL(LKG_ERR_UNSUPPORTED, "bi backward: d_out %d > 64", c);
    if (d <= 64 && d % 4 == 0 && c % 4 == 0 && c <= (d <= 32 ? 32 : 64) && rows16(d_o2, ld_do) && rows16(x, ld_x) &&
        rows16(side, ld_side) && rows16(w_out, ld_w) && rows16(dx, ld_dx) && rows16(xs_out, ld_xs)) {
        const int lpr = d <= 32 ? 8 : 16;
        BiBwdParams p{n, d, c, d_o2, ld_do, p2, x, ld_x, side, ld_side, w_out, ld_w, dx, ld_dx, xs_out, ld_xs, accumulate, 0,
                      xs_out ? xs_amax : nullptr};
        const size_t smem = (size_t)c * 4 * lpr * sizeof(float);
        const int64_t units = (n + 32 / lpr - 1) / (32 / lpr);
        const int grid = (int)std::min<int64_t>((units + 7) / 8, (int64_t)sm_count() * 8);
        if (lpr == 8) bi_bwd_rows_vec_kernel<8><<<grid, 256, smem, stream>>>(p);
        else bi_bwd_rows_vec_kernel<16><<<grid, 256, smem, stream>>>(p);
        LKG_LAUNCH_CHECK("bi_bwd_rows_vec_kernel");
        return LKG_OK;
    }
    const int cq = (c + 3) / 4;
    int ps = 4 * cq;
    if ((ps / 4) % 2 == 0) ps += 4;                           // 4 * odd
    const size_t smem = ((size_t)d * ps + 8 * 64) * sizeof(float);
    if (smem > 227 * 1024) LKG_FAIL(LKG_ERR_UNSUPPORTED, "bi backward: d_in %d x d_out %d does not fit shared memory", d, c);
    BiBwdParams p{n, d, c, d_o2, ld_do, p2, x, ld_x, side, ld_side, w_out, ld_w, dx, ld_dx, xs_out, ld_xs, accumulate, ps,
                  xs_out ? xs_amax : nullptr};
    const int per_sm = smem > 100 * 1024 ? 1 : (smem > 48 * 1024 ? 2 : 4);
    const int grid = (int)std::min<int64_t>((n + 7) / 8, (int64_t)sm_count() * per_sm);
#define LKG_BI_CASE(Q)                                                                                              \
    if (cq <= Q) {                                                                                                   \
        LKG_CUDA(cudaFuncSetAttribute(bi_bwd_rows_kernel<Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        bi_bwd_rows_kernel<Q><<<grid, 256, smem, stream>>>(p);                                                       \
        LKG_LAUNCH_CHECK("bi_bwd_rows_kernel");                                                                      \
        return LKG_OK;                                                                                               \
    }
    LKG_BI_CASE(4) LKG_BI_CASE(8) LKG_BI_CASE(16)
#undef LKG_BI_CASE
    LKG_FAIL(LKG_ERR_UNSUPPORTED, "bi backward: d_out %d", c);
}

extern "C" int lkg_gate_bwd(const float* dh, int64_t ld_dh, const float* gz, int64_t ld_gz, const float* ent,
                            int64_t ld_ent, int64_t n, int32_t dim, float* d_pre, int64_t ld_pre, float* d_ent,
                            int64_t ld_de, float* pre_amax, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) return LKG_OK;
    LKG_REQUIRE(dh && gz && ent && d_pre && d_ent && dim > 0, "null argument");
    LKG_REQUIRE(ld_gz % 2 == 0 && ld_pre % 2 == 0 && (reinterpret_cast<uintptr_t>(gz) & 7u) == 0 &&
                    (reinterpret_cast<uintptr_t>(d_pre) & 7u) == 0, "gate backward: (g, z) pairs must be 8-byte aligned");
    const bool vec = dim % 4 == 0 && rows16(dh, ld_dh) && rows16(gz, ld_gz) && rows16(ent, ld_ent) &&
                     rows16(d_pre, ld_pre) && rows16(d_ent, ld_de);
    const int64_t units = n * (vec ? dim / 4 : dim);
    const int grid = (int)std::min<int64_t>((units + 255) / 256, (int64_t)sm_count() * 8);
    const bool wide = units >= ((int64_t)1 << 30);
    auto* kernel = vec ? (wide ? gate_bwd_kernel<QuadSlot, uint64_t> : gate_bwd_kernel<QuadSlot, uint32_t>)
                       : (wide ? gate_bwd_kernel<ScalarSlot, uint64_t> : gate_bwd_kernel<ScalarSlot, uint32_t>);
    kernel<<<grid, 256, 0, stream>>>(dh, ld_dh, gz, ld_gz, ent, ld_ent, n, dim, d_pre, ld_pre, d_ent, ld_de, pre_amax);
    LKG_LAUNCH_CHECK("gate_bwd_kernel");
    return LKG_OK;
}

extern "C" int lkg_leaky_bwd(const float* grad, int64_t ld_g, const float* out, int64_t ld_out, int64_t n, int32_t c,
                             float* d_pre, int64_t ld_d, float* amax, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) return LKG_OK;
    LKG_REQUIRE(grad && out && d_pre && c > 0, "null argument");
    const bool vec = c % 4 == 0 && rows16(grad, ld_g) && rows16(out, ld_out) && rows16(d_pre, ld_d);
    const int64_t units = n * (vec ? c / 4 : c);
    const int grid = (int)std::min<int64_t>((units + 511) / 512, (int64_t)sm_count() * 8);
    const bool wide = units >= ((int64_t)1 << 30);
    auto* kernel = vec ? (wide ? leaky_bwd_kernel<QuadSlot, uint64_t> : leaky_bwd_kernel<QuadSlot, uint32_t>)
                       : (wide ? leaky_bwd_kernel<ScalarSlot, uint64_t> : leaky_bwd_kernel<ScalarSlot, uint32_t>);
    kernel<<<std::max(grid, 1), 256, 0, stream>>>(grad, ld_g, out, ld_out, n, c, d_pre, ld_d, amax);
    LKG_LAUNCH_CHECK("leaky_bwd_kernel");
    return LKG_OK;
}
