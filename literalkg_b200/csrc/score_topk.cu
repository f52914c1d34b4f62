// All-entity link-prediction scoring with a fused top-k epilogue (BASELINE.json north star (d); extension of
// calc_score, model.py:473-486 -- the reference has no top-k, SURVEY.md fact 7; its oracle is torch.topk applied to
// calc_score's output).  The B_h x N_t score matrix is never materialised.
//
//   lkg_score_index      fp32 embedding rows -> scaled fp16 "hi" plane + row norms + max norm (one pass)
//   lkg_score_topk       1. threshold: thr_h = theta_h - E_h, theta_h = k-th best EXACT score of the head among a
//                           sample of the tails (so the true k-th best is >= theta_h), E_h = rigorous bound of the
//                           single-product fp16 error, c * |h| * max_t |t|;
//                        2. filter GEMM (tcgen05, ONE fp16 product per k-step): every (head, tail) whose approximate
//                           score reaches thr_h is appended to the head's candidate list -- the true top-k is a
//                           subset by construction;
//                        3. finalize: candidates re-scored exactly (fp32 products summed in fp64, rounded once to
//                           fp32), sorted by (score desc, column asc), first k written out.  A head whose list
//                           overflowed falls back to an exact scan of all tails on the device (slow, correct).
//
// sm_100a design of the filter GEMM
//   * persistent CTA per SM; the A operand (two 128-row head blocks x K <= 256, <= 128 KB) is loaded by TMA once and
//     stays resident in shared memory; tail tiles (128 rows x 64-wide K chunks, 16 KB) stream through a 5-stage
//     mbarrier ring -- per tile one B fill feeds two MMAs, which halves the L2->SM traffic per flop (a 128 x 256
//     tile with both operands streamed needs ~175 GB/s per SM, more than L2 can deliver to 148 SMs);
//   * CTAs that share a tail tile (different head blocks) have consecutive ids, so a tile is read from HBM once
//     and hit in L2 by the other head blocks;
//   * accumulators: 2 buffers x 2 head blocks x 128 TMEM columns (all 512), epilogue of tile i overlaps MMAs of i+1;
//   * epilogue: 4 warps, thread = head row, tcgen05.ld 32 columns at a time, max-reduce, ONE compare against the
//     row's threshold (pre-multiplied by the operand scales).  Candidates go to a list private to this (head row,
//     CTA stream): exactly one thread of one CTA writes it, so the counter lives in a register and there is no
//     atomic.  They are staged in shared memory, 16 per row, and flushed to the global list when the stage fills
//     up: a global store (let alone an atomicAdd round trip) in front of the releasing mbarrier.arrive that hands
//     the accumulator back made the epilogue wait for the store to land on most tiles (measured 3.6 ms vs 1.1 ms).
#include "tc.cuh"

namespace lkg {
namespace {

using namespace tc;

constexpr int kBN = 128;                 // tails per tile
constexpr int kStages = 5;
constexpr int kThreads = 192;            // warps 0-3 epilogue, warp 4 TMA producer, warp 5 MMA issuer
constexpr int kMaxChunks = 4;            // K <= 256
constexpr uint32_t kChunkBytes = kBM * kBK * 2;     // 16 KB: 128 rows x 64 fp16 (A block chunk and B stage alike)
constexpr int kStageCand = 16;                      // candidates staged in shared memory per (thread, head block)
constexpr float kErrCoef = 1.15f / 1024.f;          // |s~ - s| <= kErrCoef |h| |t|: two fp16 roundings (2 * 2^-11),
                                                    // fp32 accumulation over K <= 256 (2^-16), theta's own 2^-21
constexpr int kFinalThreads = 256;

struct FilterParams {
    CUtensorMap a_map;       // heads hi plane [n_heads, K] fp16
    CUtensorMap b_map;       // tails hi plane [n_tails, K] fp16
    int n_heads, n_tails, n_chunks, n_pairs, n_tiles;
    const float* thr;        // [n_heads] threshold in accumulator (scaled) units
    int* cnt;                // [n_heads, n_streams] candidates seen by each CTA stream
    int* cand;               // [n_heads, n_streams, cap_s] candidate columns (positions in the tail list)
    int cap_s;               // slots per (head, stream) sublist
    // sampling mode (tilemax != NULL): visit tiles 0, tile_stride, 2 tile_stride, ... (n_tiles of them) and store
    // every head's largest approximate score of each visited tile instead of filtering
    float* tilemax;          // [n_heads, n_tiles]
    int tile_stride;
};

__global__ void __launch_bounds__(kThreads, 1) score_filter_kernel(const __grid_constant__ FilterParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;                                           // [2 blocks][n_chunks] x 16 KB
    uint8_t* smem_b = smem + 2 * kMaxChunks * kChunkBytes;            // [kStages] x 16 KB
    int* smem_cand = reinterpret_cast<int*>(smem_b + kStages * kChunkBytes);        // [2][kStageCand][128]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_cand + 2 * kStageCand * 128);
    uint64_t* full = bars;                    // [kStages]
    uint64_t* empty = bars + kStages;         // [kStages]
    uint64_t* acc_full = bars + 2 * kStages;  // [2]
    uint64_t* acc_empty = acc_full + 2;       // [2]
    uint64_t* a_full = acc_empty + 2;         // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pair = blockIdx.x % p.n_pairs;
    const int stream = blockIdx.x / p.n_pairs, n_streams = gridDim.x / p.n_pairs;
    const int row_base = pair * 2 * kBM;
    const int n_blk = row_base + kBM < p.n_heads ? 2 : 1;             // a pair whose second block is empty skips it

    if (warp == 4 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&p.a_map) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&p.b_map) : "memory");
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&acc_full[a], 1);
            mbar_init(&acc_empty[a], 128);
        }
        mbar_init(a_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4) {
        // ===== TMA producer =====
        if (lane == 0) {
            mbar_expect_tx(a_full, (uint32_t)(n_blk * p.n_chunks) * kChunkBytes);
            for (int b = 0; b < n_blk; ++b)
                for (int kc = 0; kc < p.n_chunks; ++kc)
                    tma_load_2d(&p.a_map, a_full, smem_a + (b * kMaxChunks + kc) * kChunkBytes, kc * kBK,
                                row_base + b * kBM);
            uint32_t stage = 0, phase = 0;
            for (int tile = stream; tile < p.n_tiles; tile += n_streams) {
                for (int kc = 0; kc < p.n_chunks; ++kc) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], kChunkBytes);
                    tma_load_2d(&p.b_map, &full[stage], smem_b + stage * kChunkBytes, kc * kBK,
                                tile * p.tile_stride * kBN);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 5) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t idesc = umma_idesc(kBN);
            mbar_wait(a_full, 0);
            tc_fence_after();
            uint32_t stage = 0, phase = 0;
            int it = 0;
            for (int tile = stream; tile < p.n_tiles; tile += n_streams, ++it) {
                const int buf = it & 1;
                mbar_wait(&acc_empty[buf], ((it >> 1) & 1) ^ 1);
                tc_fence_after();
                for (int kc = 0; kc < p.n_chunks; ++kc) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t b_addr = smem_u32(smem_b + stage * kChunkBytes);
                    for (int b = 0; b < n_blk; ++b) {
                        const uint32_t a_addr = smem_u32(smem_a + (b * kMaxChunks + kc) * kChunkBytes);
                        const uint32_t tmem_d = tmem_base + buf * 2 * kBN + b * kBN;
#pragma unroll
                        for (int k = 0; k < kBK / 16; ++k)
                            tc_mma_f16(tmem_d, umma_desc(a_addr + k * 32), umma_desc(b_addr + k * 32), idesc,
                                       (kc | k) != 0);
                    }
                    tc_commit(&empty[stage]);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                tc_commit(&acc_full[buf]);
            }
        }
    } else {
        // ===== epilogue warps 0-3: TMEM lane = head row of the block =====
        // The candidate path is rare per thread but hit by some lane of the warp on most tiles, so it is kept small
        // (a bit mask + a compact loop, no unrolled copies): a 32-way unrolled version made the kernel 600 KB of
        // SASS and every entry into it an instruction-cache miss (3.6 ms instead of 1.1 ms).
        int row[2], seen[2] = {0, 0}, staged[2] = {0, 0};
        float thr[2];
        int* my_cand[2];
        int* my_stage = smem_cand + threadIdx.x;        // slot i of block b: my_stage[(b * kStageCand + i) * 128]
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            row[b] = row_base + b * kBM + warp * 32 + lane;
            thr[b] = (row[b] < p.n_heads && !p.tilemax) ? __ldg(p.thr + row[b]) : INFINITY;
            my_cand[b] = p.cand + ((int64_t)row[b] * n_streams + stream) * p.cap_s;
        }
        int it = 0;
        for (int tile = stream; tile < p.n_tiles; tile += n_streams, ++it) {
            const int buf = it & 1;
            mbar_wait(&acc_full[buf], (it >> 1) & 1);
            tc_fence_after();
            const int tile_col0 = tile * p.tile_stride * kBN;
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                if (b >= n_blk) break;
                const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + buf * 2 * kBN + b * kBN;
                float tmax = -INFINITY;
#pragma unroll 1
                for (int c0 = 0; c0 < kBN; c0 += 32) {
                    uint32_t r[32];
                    tc_ld32_nowait(taddr + c0, r);
                    tc_ld_wait();
                    const int col0 = tile_col0 + c0;
                    const int valid = p.n_tails - col0;                  // columns of this group inside the tail list
                    float m = __uint_as_float(r[0]);
#pragma unroll
                    for (int j = 1; j < 32; ++j) m = fmaxf(m, __uint_as_float(r[j]));
                    if (p.tilemax) {
                        if (valid < 32) {                                // last, partial tile: TMA zero-filled the rest
                            m = -INFINITY;
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < valid) m = fmaxf(m, __uint_as_float(r[j]));
                        }
                        tmax = fmaxf(tmax, m);
                    } else if (m >= thr[b]) {
                        uint32_t mask = 0;
#pragma unroll
                        for (int j = 0; j < 32; ++j) mask |= (__uint_as_float(r[j]) >= thr[b] ? 1u : 0u) << j;
                        if (valid < 32) mask &= valid <= 0 ? 0u : (1u << valid) - 1u;
#pragma unroll 1
                        while (mask) {
                            const int j = __ffs(mask) - 1;
                            mask &= mask - 1;
                            my_stage[(b * kStageCand + staged[b]) * 128] = col0 + j;
                            if (++staged[b] == kStageCand) {             // stage full: flush to the global list
#pragma unroll 1
                                for (int i = 0; i < kStageCand; ++i)
                                    if (seen[b] + i < p.cap_s) my_cand[b][seen[b] + i] = my_stage[(b * kStageCand + i) * 128];
                                seen[b] += kStageCand;
                                staged[b] = 0;
                            }
                        }
                    }
                }
                if (p.tilemax && row[b] < p.n_heads) p.tilemax[(int64_t)row[b] * p.n_tiles + tile] = tmax;
            }
            tc_fence_before();
            mbar_arrive(&acc_empty[buf]);
        }
        if (!p.tilemax) {
#pragma unroll
            for (int b = 0; b < 2; ++b) {
#pragma unroll 1
                for (int i = 0; i < staged[b]; ++i)
                    if (seen[b] + i < p.cap_s) my_cand[b][seen[b] + i] = my_stage[(b * kStageCand + i) * 128];
                seen[b] += staged[b];
                if (row[b] < p.n_heads) p.cnt[(int64_t)row[b] * n_streams + stream] = seen[b];
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    }
}

constexpr uint32_t kFilterSmem = (2 * kMaxChunks + kStages) * kChunkBytes + 2 * kStageCand * 128 * 4 /*candidates*/ +
                                 1024 /*align*/ + 256 /*barriers*/;
static_assert(kFilterSmem <= 227 * 1024, "filter kernel shared memory");

int make_map_2d(CUtensorMap* map, const void* base, int64_t rows, int k, int64_t ld) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) LKG_FAIL(LKG_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    LKG_REQUIRE(aligned16(base) && (ld * 2) % 16 == 0, "hi planes must be 16-byte aligned (base, row stride)");
    cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)kBM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) LKG_FAIL(LKG_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return LKG_OK;
}

// ---- index: fp32 rows -> scaled fp16 hi plane + norms ------------------------------------------------------------
__global__ void score_index_kernel(const float* __restrict__ emb, int64_t ld, const int64_t* __restrict__ rows,
                                   int64_t m, int dim, const float* __restrict__ rec, __half* __restrict__ hi,
                                   int64_t ld_hi, float* __restrict__ norms, float* __restrict__ max_norm) {
    const float scale = __ldg(rec + 1);
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int groups = (int)(ld_hi >> 3);
    float wmax = 0.f;
    for (int64_t r = warp; r < m; r += nwarps) {
        const float* src = emb + (rows ? rows[r] : r) * ld;
        float ss = 0.f;
        for (int gq = lane; gq < groups; gq += 32) {
            const int c0 = 8 * gq;
            float x[8];
            if (c0 + 8 <= dim && (ld & 3) == 0) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(src + c0));
                const float4 b = __ldg(reinterpret_cast<const float4*>(src + c0) + 1);
                x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) x[j] = c0 + j < dim ? __ldg(src + c0 + j) : 0.f;
            }
            __align__(16) __half h[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float v = x[j] * scale;
                h[j] = __float2half_rn(v);
                ss = fmaf(v, v, ss);
            }
            *reinterpret_cast<uint4*>(hi + r * ld_hi + c0) = *reinterpret_cast<const uint4*>(h);
        }
        const float nrm = sqrtf(warp_sum(ss)) * 1.000001f;     // scaled units, rounded up
        if (lane == 0) norms[r] = nrm;
        wmax = fmaxf(wmax, nrm);
    }
    if (lane == 0 && wmax > 0.f) atomicMax(reinterpret_cast<uint32_t*>(max_norm), __float_as_uint(wmax));
}

// E (accumulator units): bound of |single-product fp16 score - exact score| for one head against any tail
__device__ __forceinline__ float score_err(float nh, float nt, int dim) {
    return kErrCoef * nh * nt + 4.8e-7f /*2^-21*/ * (nh + nt) * sqrtf((float)dim) + 1.f;
}

// thr = theta * scale^2 - E with theta a lower bound of the head's k-th best EXACT score (caller supplied)
__global__ void score_threshold_kernel(const float* __restrict__ theta, int64_t theta_stride, int n_heads,
                                       const float* __restrict__ head_norms, const float* __restrict__ tail_max_norm,
                                       const float* __restrict__ rec, int dim, float* __restrict__ thr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_heads) return;
    const float s2 = rec[1] * rec[1];
    const float err = score_err(head_norms[i], *tail_max_norm, dim);
    const float th = theta ? theta[(int64_t)i * theta_stride] : -INFINITY;
    // theta == -inf (no bound known): every tail is a candidate
    thr[i] = th == -INFINITY ? -INFINITY : th * s2 - err - fabsf(th * s2) * 1e-6f;
}

// ---- keys and their sort -----------------------------------------------------------------------------------------
// enc: order-preserving 32-bit code of a float (-0 < +0); the selection kernels sort 64-bit keys (enc(s) << 32) | ~p,
// so a descending sort gives "larger score first, ties -> lower position", and key 0 sorts last.
__device__ __forceinline__ uint32_t enc(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// Sorts keys[0, n) descending in place (shared memory, the whole block): 0 keys pad the list to the next power of two
// (keys must have room for them), then a bitonic network.
__device__ void sort_keys_desc(unsigned long long* keys, int n) {
    int p2 = 1;
    while (p2 < n) p2 <<= 1;
    for (int i = n + threadIdx.x; i < p2; i += blockDim.x) keys[i] = 0ull;
    __syncthreads();
    for (int size = 2; size <= p2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < p2; i += blockDim.x) {
                const int j = i ^ stride;
                if (j > i) {
                    const bool desc = (i & size) == 0;
                    const unsigned long long a = keys[i], b = keys[j];
                    if ((a < b) == desc) {
                        keys[i] = b;
                        keys[j] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
}

// thr = (k-th largest tile maximum of the sampled tiles) - 2E.  The tile maxima are k distinct tails whose
// APPROXIMATE scores reach m_k, so their exact scores reach m_k - E, so the exact k-th best is >= m_k - E and every
// member of the true top-k has an approximate score >= m_k - 2E.  One CTA per head, the maxima sorted as enc() keys.
__global__ void __launch_bounds__(256) score_sample_threshold_kernel(const float* __restrict__ tilemax, int n_st, int k,
                                                                     const float* __restrict__ head_norms,
                                                                     const float* __restrict__ tail_max_norm, int dim,
                                                                     float* __restrict__ thr) {
    extern __shared__ unsigned long long sv[];
    const int head = blockIdx.x;
    for (int i = threadIdx.x; i < n_st; i += blockDim.x) sv[i] = enc(tilemax[(int64_t)head * n_st + i]);
    sort_keys_desc(sv, n_st);
    if (threadIdx.x == 0) {
        const float mk = k <= n_st ? dec((uint32_t)sv[k - 1]) : -INFINITY;
        thr[head] = mk == -INFINITY ? -INFINITY : mk - 2.f * score_err(head_norms[head], *tail_max_norm, dim) - fabsf(mk) * 1e-6f;
    }
}

// Score kinds: the dot product emb[h] . emb[j], or the negated squared distance -|q - p_j|^2 of the relation-aware
// triple score (TransR / TransE), and the dense instance of the filter that reads a score matrix.
constexpr int kDot = 0, kL2 = 1, kScores = 2;
constexpr int kL2MaxDim = 508;           // distance rows: dim % 4 == 0, the augmented width dim + 4 <= 512
// Query row staged by the rank kernels (zero padded): the distance's augmented width, the dot score's GEMM K.
template <int Kind> constexpr int row_floats() { return Kind == kL2 ? kL2MaxDim + 4 : kMaxChunks * kBK; }

// Exact score of one (query, candidate) pair, larger = better: s = a . b (kDot) or s = -|a - b|^2 (kL2).  Products
// and differences of fp32 values are exact in fp64; they are summed in fp64 with one fma per element and rounded once
// to fp32 (the distance is then negated, which is exact, so "s_j > s_t" is "d_j < d_t" and one comparison and one tie
// rule serve both kinds).  Eight lanes share a candidate row (lane q of the group takes float4 q, q + 8, ...), so a
// warp scores four candidates at once with all its row loads in flight together.  NV float4 per lane: 8 covers widths
// up to 256, 16 up to 512; float4 v >= dim / 4 is skipped, so for dim <= 256 both instances load the same values and
// sum them in the same order.  `a` (the query row) may live in shared or global memory: every caller of a kind sees
// the same values in the same order, so rank prepare, finalize and the filter, or the top-k threshold and finalize,
// return the same bits for the same pair.
template <int Kind, int NV>
__device__ __forceinline__ float exact_score(const float* a, const float* __restrict__ b, int dim, int q, bool live) {
    double acc = 0.0;
    const int nv = dim >> 2;                                   // dim % 4 == 0 is checked on the host side
    float4 t[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int v = q + 8 * i;
        t[i] = (live && v < nv) ? __ldg(reinterpret_cast<const float4*>(b) + v) : make_float4(0, 0, 0, 0);
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int v = q + 8 * i;
        if (v < nv) {
            const float4 h = *reinterpret_cast<const float4*>(a + 4 * v);
            if constexpr (Kind == kL2) {
                double d = (double)h.x - (double)t[i].x;
                acc = fma(d, d, acc);
                d = (double)h.y - (double)t[i].y;
                acc = fma(d, d, acc);
                d = (double)h.z - (double)t[i].z;
                acc = fma(d, d, acc);
                d = (double)h.w - (double)t[i].w;
                acc = fma(d, d, acc);
            } else {
                acc = fma((double)h.x, (double)t[i].x, acc);
                acc = fma((double)h.y, (double)t[i].y, acc);
                acc = fma((double)h.z, (double)t[i].z, acc);
                acc = fma((double)h.w, (double)t[i].w, acc);
            }
        }
    }
    acc += __shfl_xor_sync(kFull, acc, 4);
    acc += __shfl_xor_sync(kFull, acc, 2);
    acc += __shfl_xor_sync(kFull, acc, 1);
    return Kind == kL2 ? -(float)acc : (float)acc;
}

// The rank kernels' instance: the float4 count of their staged row.
template <int Kind>
__device__ __forceinline__ float rank_score(const float* a, const float* __restrict__ b, int dim, int q, bool live) {
    return exact_score<Kind, row_floats<Kind>() / 32>(a, b, dim, q, live);
}

// fp64 sums over the float4s v = lane, lane + L, ... of a row, reduced over L lanes: |a|^2 and, with a centre c
// (nullable), a . c and sum |a_k c_k|.  The band margins take the norms of the query operand from here.
struct RowSums {
    double aa, ac, aca;
};
template <int L>
__device__ __forceinline__ RowSums row_sums(const float* __restrict__ a, const float* __restrict__ c, int dim,
                                            int lane) {
    RowSums r{0.0, 0.0, 0.0};
    for (int v = lane; v < (dim >> 2); v += L) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(a) + v);
        r.aa = fma((double)x.x, (double)x.x, r.aa);
        r.aa = fma((double)x.y, (double)x.y, r.aa);
        r.aa = fma((double)x.z, (double)x.z, r.aa);
        r.aa = fma((double)x.w, (double)x.w, r.aa);
        if (c) {
            const float4 y = __ldg(reinterpret_cast<const float4*>(c) + v);
            r.ac = fma((double)x.x, (double)y.x, r.ac);
            r.ac = fma((double)x.y, (double)y.y, r.ac);
            r.ac = fma((double)x.z, (double)y.z, r.ac);
            r.ac = fma((double)x.w, (double)y.w, r.ac);
            r.aca += fabs((double)x.x * y.x) + fabs((double)x.y * y.y) + fabs((double)x.z * y.z) +
                     fabs((double)x.w * y.w);
        }
    }
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) {
        r.aa += __shfl_xor_sync(kFull, r.aa, o);
        if (c) {
            r.ac += __shfl_xor_sync(kFull, r.ac, o);
            r.aca += __shfl_xor_sync(kFull, r.aca, o);
        }
    }
    return r;
}

// Stages a query row in shared memory, zero padded to N floats (the exact scorer reads whole float4s of it).
template <int N>
__device__ __forceinline__ void stage_row(float* s_row, const float* __restrict__ row, int dim) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) s_row[i] = i < dim ? __ldg(row + i) : 0.f;
}

// Exact scan of positions [0, n) keeping the best `half` keys (keys holds 2 half): each chunk of `half` positions is
// keyed after the kept keys, sorted with them and cut back to `half`.  score(p, q, live) is the exact score of
// position p (all 8 lanes of a group call it: the scorer shuffles), key(s, p) its key.  -> the number of kept keys.
template <class Score, class Key>
__device__ int scan_best(unsigned long long* keys, int n, int half, Score score, Key key) {
    __shared__ int s_kept;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int grp = lane >> 3, q = lane & 7;
    if (threadIdx.x == 0) s_kept = 0;
    __syncthreads();
    for (int base = 0; base < n; base += half) {
        const int chunk = min(half, n - base);
        const int kept = s_kept;
        for (int c0 = 4 * warp; c0 < chunk; c0 += 4 * nwarps) {
            const int c = c0 + grp;
            const bool live = c < chunk;
            const int p = live ? base + c : 0;
            const float s = score(p, q, live);
            if (live && q == 0) keys[kept + c] = key(s, p);
        }
        __syncthreads();
        sort_keys_desc(keys, kept + chunk);
        if (threadIdx.x == 0) s_kept = min(kept + chunk, half);
        __syncthreads();
    }
    return s_kept;
}

// Writes the first k of n sorted keys as (score, position), padded with -1 and the worst score; kL2 writes d = -s.
template <int Kind>
__device__ __forceinline__ void write_first_k(const unsigned long long* keys, int n, int k, float* val, int64_t* pos) {
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const unsigned long long key = i < n ? keys[i] : 0ull;
        const float s = dec((uint32_t)(key >> 32));
        val[i] = key ? (Kind == kL2 ? -s : s) : (Kind == kL2 ? INFINITY : -INFINITY);
        pos[i] = key ? (int64_t)(~(uint32_t)(key & 0xffffffffu)) : -1;
    }
}

// Block-wide count of the columns c in [0, n) that beat the target (score t, position tp) under the tie rule of the
// ranks: s > t, or s == t and p < tp -- compared as enc() keys for kScores (-0 < +0 there).  Four columns per warp, 8
// lanes each: score(c, q, &p) is called by all lanes of column c's group (c >= n included: the exact scorer shuffles)
// and sets p, the column's candidate position, or p < 0 when the column does not count.  -> the total, in thread 0.
template <int Kind, class Score>
__device__ int64_t count_beating(int n, float t, int64_t tp, Score score) {
    __shared__ int s_cnt[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int grp = lane >> 3, q = lane & 7;
    int cnt = 0;
    for (int c0 = 4 * warp; c0 < n; c0 += 4 * nwarps) {
        int p = -1;
        const float s = score(c0 + grp, q, p);
        const bool beats = Kind == kScores ? enc(s) > enc(t) || (enc(s) == enc(t) && p < tp)
                                           : s > t || (s == t && p < tp);
        if (p >= 0 && q == 0 && beats) ++cnt;
    }
    cnt = (int)warp_sum((float)cnt);                 // < 2^24 per warp
    if (lane == 0) s_cnt[warp] = cnt;
    __syncthreads();
    int64_t tot = 0;
    if (threadIdx.x == 0)
        for (int w = 0; w < nwarps; ++w) tot += s_cnt[w];
    return tot;
}

struct FinalParams {
    const float* emb;           // tails' matrix
    int64_t ld_emb;
    const float* head_emb;      // heads' matrix (may be the same)
    int64_t ld_head_emb;
    const int64_t* head_rows;   // nullable: head i = row head_row_base + i
    int64_t head_row_base;
    const int64_t* tail_rows;   // nullable: tail j = row j
    int n_heads, n_tails, dim, k, cap;
    int n_streams, cap_s;       // candidate sublists per head and their capacity (n_streams * cap_s <= cap)
    const int* cnt;
    const int* cand;
    float* top_val;
    int64_t* top_col;
};

// One CTA per head.  keys: (ordered score << 32) | ~column, so a descending sort gives "larger score first, ties ->
// lower column".
__global__ void __launch_bounds__(kFinalThreads) score_finalize_kernel(FinalParams p) {
    extern __shared__ unsigned long long keys[];
    const int head = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = kFinalThreads / 32;
    const int grp = lane >> 3, q = lane & 7;                    // 4 candidates per warp, 8 lanes each
    __shared__ __align__(16) float s_head[kMaxChunks * kBK];
    stage_row<kMaxChunks * kBK>(s_head, p.head_emb + (p.head_rows ? p.head_rows[head] : p.head_row_base + head) *
                                                         p.ld_head_emb, p.dim);
    // gather the head's sublists (one per CTA stream of the filter kernel) into one column list
    int* cols = reinterpret_cast<int*>(keys + p.cap);
    __shared__ int s_off[161], s_n, s_over;
    for (int sidx = threadIdx.x; sidx < p.n_streams; sidx += blockDim.x)
        s_off[sidx] = p.cnt[(int64_t)head * p.n_streams + sidx];
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0, over = 0;
        for (int sidx = 0; sidx < p.n_streams; ++sidx) {
            const int c = s_off[sidx];
            over |= c > p.cap_s;
            s_off[sidx] = tot;
            tot += min(c, p.cap_s);
        }
        s_off[p.n_streams] = tot;
        s_n = tot;
        s_over = over;
    }
    __syncthreads();
    auto score = [&](int col, int q, bool live) {
        return exact_score<kDot, 8>(s_head, p.emb + (p.tail_rows ? p.tail_rows[col] : col) * p.ld_emb, p.dim, q, live);
    };
    auto key = [](float s, int col) { return ((unsigned long long)enc(s) << 32) | (uint32_t)(~(uint32_t)col); };
    int n;
    if (s_over == 0) {
        n = s_n;
        for (int sidx = warp; sidx < p.n_streams; sidx += nwarps) {
            const int o = s_off[sidx], c = s_off[sidx + 1] - o;
            const int* src = p.cand + ((int64_t)head * p.n_streams + sidx) * p.cap_s;
            for (int i = lane; i < c; i += 32) cols[o + i] = src[i];
        }
        __syncthreads();
        for (int c0 = 4 * warp; c0 < n; c0 += 4 * nwarps) {
            const int c = c0 + grp;
            const bool live = c < n;
            const int col = live ? cols[c] : 0;
            const float s = score(col, q, live);
            if (live && q == 0) keys[c] = key(s, col);
        }
        sort_keys_desc(keys, n);
    } else {
        // Overflow fallback (the candidate band held more than `cap` tails, e.g. a plateau of near-identical
        // scores): exact scan of every tail (cap / 2 >= k is checked on the host side).
        n = scan_best(keys, p.n_tails, p.cap / 2, score, key);
    }
    write_first_k<kDot>(keys, n, p.k, p.top_val + (int64_t)head * p.k, p.top_col + (int64_t)head * p.k);
}

// ---- rank of a given tail per head (north star (d): "top-k and rank epilogue") -----------------------------------
// rank_i = #{ j : s_ij > s_it  or  (s_ij == s_it and j < t_i) } with s the EXACT scores (fp32 products summed in fp64,
// one rounding -- the values the fused top-k returns) and t_i the position of head i's target in the tail list.
//   1. lkg_rank_prepare   tau_i = exact score of (head i, target i); band tau_i -/+ E_i with E_i a bound of the
//                         3-product fp16 hi/lo GEMM's error for K <= 256: representation (operands kept to 2^-22, the
//                         lo * lo product dropped) 3 * 2^-22 |h||t| = 0.7e-6, fp32 accumulation of 48 MMAs at <= 2^-23
//                         of the running magnitude each = 5.7e-6; kRankErr = 1e-5 leaves a factor 1.5 on top;
//   2. lkg_score_rank     (gemm_tc.cu) the score GEMM with a counting epilogue: columns certainly above tau are counted,
//                         the ones inside the band are listed; no score leaves the SM;
//   3. lkg_rank_finalize  the listed columns re-scored exactly and compared with tau under the tie rule.
constexpr float kRankErr = 1.0e-5f;

// The same bound as a function of the GEMM's K (the engine runs whole 64-wide chunks: 3 MMAs per 16 columns of them),
// relative to |a| |b| of the two operand rows: per MMA 2^-23 of the running magnitude, 3 * 2^-22 for the hi/lo
// representation of both operands and the dropped lo * lo product, times 1.5.  DESIGN.md §6 has the derivation.
__host__ __device__ constexpr double rank_err(int k) {
    return 1.5 * (3.0 * ((k + kBK - 1) / kBK) * (kBK / 16) * 0x1p-23 + 3.0 * 0x1p-22);
}
static_assert(rank_err(kMaxChunks * kBK) <= kRankErr, "kRankErr must cover the dot rank GEMM at K = 256");

// ---- distance rank (the triple score, TransR / TransE) -----------------------------------------------------------
// d_j = |q - p_j|^2 is turned into the counting GEMM's form by centring on c (the candidates' mean row) and one
// augmented column: with u = q - c, w_j = p_j - c and nu_j = -|w_j|^2 / 2,
//     d_j = |u|^2 - 2 (u . w_j + nu_j),
// so "closer" is "larger u~ . v~_j" with u~ = [u, alpha, 0..] and v~_j = [w_j, nu_j / alpha, 0..].  alpha is a power of
// two near max_j |w_j| (exact division): it keeps |u~| and |v~_j| of the order of the rows' own norms, so the GEMM's
// error band scales like the distances do whatever the embeddings' magnitude.
// stats (float[2] per candidate table): {W = max_j |w_j|, V = max_j |v~_j|}, both rounded up.
__device__ __forceinline__ float l2_alpha(float w) {
    if (!(w > 0.f && w < 3.0e38f)) return 1.f;
    int ex;
    frexpf(w, &ex);                                     // w in [2^(ex-1), 2^ex)
    ex = ex - 1 > 60 ? 60 : (ex - 1 < -60 ? -60 : ex - 1);
    return ldexpf(1.f, ex);
}

// One warp per row.  pass 0: the norms of the centred rows only (stats[0] = W); pass 1: candidates [w, nu / alpha, 0..]
// and stats[1] = V; pass 2: queries [u, alpha, 0..].  The row norm is accumulated in fp64 from the ROUNDED fp32 x - c
// (the values the GEMM and the bound see) and rounded once.
__global__ void l2_rank_rows_kernel(const float* __restrict__ src, int64_t ld, const int64_t* __restrict__ rows,
                                    int64_t m, int dim, const float* __restrict__ center, int pass,
                                    float* __restrict__ stats, float* __restrict__ out, int64_t ld_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int nv = dim >> 2;
    const float alpha = pass == 0 ? 1.f : l2_alpha(__ldg(stats));
    float wmax = 0.f;
    for (int64_t r = warp; r < m; r += nwarps) {
        const float4* x4 = reinterpret_cast<const float4*>(src + (rows ? rows[r] : r) * ld);
        float4* o4 = reinterpret_cast<float4*>(out + r * ld_out);
        double nn = 0.0;
        for (int v = lane; v < nv; v += 32) {
            const float4 x = __ldg(x4 + v), c = __ldg(reinterpret_cast<const float4*>(center) + v);
            const float4 u = make_float4(x.x - c.x, x.y - c.y, x.z - c.z, x.w - c.w);
            nn = fma((double)u.x, (double)u.x, nn);
            nn = fma((double)u.y, (double)u.y, nn);
            nn = fma((double)u.z, (double)u.z, nn);
            nn = fma((double)u.w, (double)u.w, nn);
            if (pass != 0) o4[v] = u;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nn += __shfl_xor_sync(kFull, nn, o);
        if (pass == 0) {
            wmax = fmaxf(wmax, __double2float_ru(__dsqrt_ru(nn)));
        } else if (lane == 0) {
            float aug = alpha;
            if (pass == 1) {
                aug = (float)(-0.5 * nn) / alpha;
                wmax = fmaxf(wmax, __double2float_ru(__dsqrt_ru(nn + (double)aug * aug)));
            }
            o4[nv] = make_float4(aug, 0.f, 0.f, 0.f);
        }
    }
    wmax = warp_max(wmax);
    if (pass != 2 && lane == 0 && wmax > 0.f)
        atomicMax(reinterpret_cast<uint32_t*>(stats + (pass == 0 ? 0 : 1)), __float_as_uint(wmax));
}

// center (nullable, [dim]): the GEMM's tails are t_j - center (a common shift moves every score of a head by the same
// h . center, so the ranking is unchanged while the error bound shrinks from |h| max|t| to |h| max|t - center| -- the
// embeddings of a trained or freshly initialised model are tightly clustered around their mean, and a band relative
// to |t| would hold tens of thousands of tails); the thresholds are then taken around tau - h . center.
// out[r, :] = src[rows ? rows[r] : r, :] - center  (the shifted tails of the rank GEMM)
__global__ void shift_rows_kernel(const float* __restrict__ src, int64_t ld, const int64_t* __restrict__ rows, int64_t m,
                                  int k, const float* __restrict__ center, float* __restrict__ out, int64_t ldo) {
    const int64_t total = m * k;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / k;
        const int c = (int)(i - r * k);
        out[r * ldo + c] = src[(rows ? rows[r] : r) * ld + c] - __ldg(center + c);
    }
}

// M of the distance band: with the GEMM value g_j of a candidate, g_j > sigma + M implies d_j < t and g_j < sigma - M
// implies d_j > t, for a target distance t and sigma = (|u|^2 - t) / 2 (derivation in rank_prepare_kernel and DESIGN.md
// §6 "Bound").  uu = |u|^2 and alpha: the query operand u~ = [u, alpha]; stats: the candidate operand's {W, V}; inv_q,
// inv_c: the inverse scales (record slot 2) of the query's and the candidates' planes.  The rank prepare kernel and the
// top-k threshold kernel both take their band from here.
__device__ __forceinline__ double l2_band_margin(double uu, double alpha, double t, int dim, const float* stats,
                                                 float inv_q, float inv_c) {
    const int k = dim + 4;
    const double w = stats[0], vmax = stats[1];
    const double nu = __dsqrt_ru(uu) * (1.0 + 0x1p-40), nua = __dsqrt_ru(uu + alpha * alpha) * (1.0 + 0x1p-40);
    const double e = rank_err(k) * nua * vmax + 0x1p-24 * sqrt((double)k) * 1.001 * (vmax * inv_q + nua * inv_c);
    const double r = 0x1p-21 * (nu + w) * (nu + w);
    const double sigma = 0.5 * (uu - t);
    return e + 0.5 * r + 0x1p-21 * t + (uu + fabs(sigma)) * 0x1p-40 + 1e-30;
}

// What the distance instance of rank_prepare_kernel reads besides the dot instance's arguments (which it reads as:
// emb = the candidates' projected rows p_j, head_emb = the query rows q, tail_max_norm = the stats of the candidate
// operand, rec = the scale record of its planes).
struct L2Prep {
    const float* aug;        // [n_heads, ld_aug] the query operand u~ = [q - c, alpha, 0..]
    int64_t ld_aug;
    const float* rec_q;      // scale record of its planes
};

template <int Kind>
__global__ void rank_prepare_kernel(const float* __restrict__ emb, int64_t ld, const int64_t* __restrict__ tail_rows,
                                    const float* __restrict__ head_emb, int64_t ld_h,
                                    const int64_t* __restrict__ head_rows, const int64_t* __restrict__ target_pos,
                                    int n_heads, int dim, const float* __restrict__ tail_max_norm,
                                    const float* __restrict__ rec, const float* __restrict__ center,
                                    float* __restrict__ tau, float* __restrict__ thr, const L2Prep l2) {
    // 8 lanes per query (the exact scorer's layout), 4 queries per warp.  The target's score s_t comes from the scorer
    // finalize and the filter re-score with, on the same rows in the same order, so the target never beats itself.
    const int gq = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    const int q = threadIdx.x & 7;
    const bool live = gq < n_heads;
    const int head = live ? gq : 0;
    const float* hrow = head_emb + (head_rows ? head_rows[head] : head) * ld_h;
    const int64_t tp = target_pos[head];
    const float s = rank_score<Kind>(hrow, emb + (tail_rows ? tail_rows[tp] : tp) * ld, dim, q, live);
    if constexpr (Kind == kL2) {
        // tau = d_t = -s.  With D_j the exact distance on the fp32 rows q, p_j, the GEMM value g_j and
        // S~_j = u . w_j + nu_j on the rounded fp32 operands (DESIGN.md §6):
        //   |g_j - S~_j| <= E = rank_err(K) |u~| V + 2^-24 sqrt(K) (V / s_q + |u~| / s_c)  (the second term: fp16
        //                       subnormals of the lo planes, 1 / s the record's inverse scales),
        //   |D_j - (|u|^2 - 2 S~_j)| <= R = 2^-21 (|u| + W)^2  (rounding of q - c, p_j - c and nu_j),
        // so g_j > sigma + M implies D_j < d_t (1 - 2^-22), hence d_j = fl(D_j) < d_t, and g_j < sigma - M implies
        // d_j > d_t, with sigma = (|u|^2 - d_t) / 2 and M = E + R / 2 + 2^-21 d_t + the fp64 rounding of sigma.
        const float t = -s;
        const float* arow = l2.aug + (int64_t)head * l2.ld_aug;
        const double uu = row_sums<8>(arow, nullptr, dim, q).aa;
        if (live && q == 0) {
            const double sigma = 0.5 * (uu - (double)t);
            const double mrg = l2_band_margin(uu, arow[dim], t, dim, tail_max_norm, __ldg(l2.rec_q + 2), __ldg(rec + 2));
            tau[head] = t;
            thr[2 * head] = __double2float_rd(sigma - mrg);
            thr[2 * head + 1] = __double2float_ru(sigma + mrg);
        }
    } else {
        const RowSums h = row_sums<8>(hrow, center, dim, q);         // |h|^2 and h . c
        if (live && q == 0) {
            const float ts = (float)((double)s - h.ac);              // the target score in the GEMM's (shifted) frame
            // bound of the GEMM's error (norms of the tails: scaled units) + the roundings of s_t and ts
            const float e = kRankErr * (float)sqrt(h.aa) * (*tail_max_norm) * rec[2] * 1.0001f +
                            (fabsf(s) + fabsf(ts) + (float)fabs(h.ac)) * 2e-7f + 1e-30f;
            tau[head] = s;
            thr[2 * head] = ts - e;
            thr[2 * head + 1] = ts + e;
        }
    }
}

// Kind == kL2: emb = the candidates' projected rows p_j (tail_rows NULL), head_emb = the query rows q, tau = d_t; the
// comparison runs on s = -d against -tau, so the tie rule and the counting are the dot instance's.
template <int Kind>
__global__ void __launch_bounds__(256) rank_finalize_kernel(const float* __restrict__ emb, int64_t ld,
                                                            const int64_t* __restrict__ tail_rows,
                                                            const float* __restrict__ head_emb, int64_t ld_h,
                                                            const int64_t* __restrict__ head_rows,
                                                            const int64_t* __restrict__ target_pos,
                                                            const float* __restrict__ tau, const int* __restrict__ above,
                                                            const int* __restrict__ band_cnt, const int* __restrict__ band,
                                                            int cap, int n_tails, int dim, int64_t* __restrict__ ranks) {
    __shared__ __align__(16) float s_head[row_floats<Kind>()];
    const int head = blockIdx.x;
    stage_row<row_floats<Kind>()>(s_head, head_emb + (head_rows ? head_rows[head] : head) * ld_h, dim);
    __syncthreads();
    const float t = Kind == kL2 ? -tau[head] : tau[head];
    const int n_band = band_cnt[head];
    const bool overflow = n_band > cap;            // the band held more columns than the list: exact scan of every tail
    const int n = overflow ? n_tails : n_band;
    const int64_t better = count_beating<Kind>(n, t, target_pos[head], [&](int c, int q, int& p) {
        const bool live = c < n;
        const int col = live ? (overflow ? c : band[(int64_t)head * cap + c]) : 0;
        const float s = rank_score<Kind>(s_head, emb + (tail_rows ? tail_rows[col] : col) * ld, dim, q, live);
        p = live ? col : -1;
        return s;
    });
    if (threadIdx.x == 0) ranks[head] = better + (overflow ? 0 : above[head]);
}

// ---- filtered rank: subtract the known true tails that beat the target ------------------------------------------
// Filter run of a query: the tails t' of the known triples (h, r, t') -- a binary search of r in the head's att row,
// which is sorted by (relation, tail) -- or, without a relation (r < 0), the head's agg row of unique (h, t') pairs.
// Both runs are sorted by tail; the att run keeps duplicate triples, so callers skip a tail equal to its predecessor.
__device__ __forceinline__ void filter_run(const lkg_graph& g, int64_t h, int64_t r, const int32_t** tails, int* lo,
                                           int* hi) {
    if (r < 0) {
        *tails = g.col;
        *lo = g.rowptr[h];
        *hi = g.rowptr[h + 1];
        return;
    }
    int a = g.att_rowptr[h], b = g.att_rowptr[h + 1];
    int l = a, u = b;                                  // first index with rel >= r
    while (l < u) {
        const int m = (l + u) >> 1;
        if (g.att_rel[m] < r) l = m + 1; else u = m;
    }
    a = l;
    u = b;                                             // first index with rel > r
    while (l < u) {
        const int m = (l + u) >> 1;
        if (g.att_rel[m] <= r) l = m + 1; else u = m;
    }
    *tails = g.att_tail;
    *lo = a;
    *hi = l;
}

// One CTA per query, the run split over the warps like rank_finalize_kernel's band (a hub head can have thousands of
// known tails).  A filter tail f at candidate position p != t is subtracted when it beats the target under the rule
// the raw rank was counted with, on the same scores:
//   kExact  (fused path, after lkg_rank_finalize): s_f = rank_score of the same head row staged the same way, compared
//           with the same tau by the same float comparison.  finalize counts a column either because the GEMM put it
//           above tau + E -- and then its exact score is above tau, the band bound being rigorous -- or because its
//           exact score beats tau; either way the bit-identical re-score here reaches the same verdict;
//   kL2     (distance path, after lkg_rank_finalize_l2): the same argument with s = rank_score = -d of the query row (row qi
//           of qrows, staged like finalize stages it) and f's row in the candidate table (src row p), against -tau;
//   kScores (dense path, after lkg_topk_rows): s_f and s_t are read from the score matrix and compared as the
//           order-preserving keys lkg_topk_rows compares (-0 < +0 there).
template <int Kind>
__global__ void __launch_bounds__(256) rank_filter_kernel(const lkg_graph g, const int64_t* __restrict__ heads,
                                                          const int64_t* __restrict__ rels,
                                                          const int32_t* __restrict__ cand_map,
                                                          const int64_t* __restrict__ target_pos,
                                                          const float* __restrict__ src, int64_t ld, int dim,
                                                          const float* __restrict__ tau, int64_t* __restrict__ ranks,
                                                          const float* __restrict__ qrows, int64_t ld_q) {
    constexpr bool kExact = Kind != kScores;
    __shared__ __align__(16) float s_head[row_floats<Kind>()];
    const int qi = blockIdx.x;
    const int64_t h = heads[qi];
    const int64_t tp = target_pos[qi];
    if (kExact) {
        stage_row<row_floats<Kind>()>(s_head, Kind == kL2 ? qrows + (int64_t)qi * ld_q : src + h * ld, dim);
        __syncthreads();
    }
    const int32_t* run;
    int lo, hi;
    filter_run(g, h, rels ? rels[qi] : -1, &run, &lo, &hi);
    const float* srow = src + (int64_t)qi * ld;                      // dense: this query's row of the score matrix
    const float t = Kind == kL2 ? -tau[qi] : (kExact ? tau[qi] : srow[tp]);
    const int n = hi - lo;
    const int64_t sub = count_beating<Kind>(n, t, tp, [&](int c, int q, int& p) {
        bool live = c < n;
        int f = 0;
        if (live) {
            f = run[lo + c];
            p = cand_map ? cand_map[f] : f;
            live = p >= 0 && p != tp && (c == 0 || run[lo + c - 1] != f);
        }
        float s = 0.f;
        if constexpr (kExact) s = rank_score<Kind>(s_head, src + (int64_t)(Kind == kL2 ? p : f) * ld, dim, q, live);
        else if (live) s = srow[p];
        if (!live) p = -1;
        return s;
    });
    if (threadIdx.x == 0) ranks[qi] -= sub;
}

// ---- filtered top-k: the triple score (distance) and the dot score ------------------------------------------------
// Per query (q_i, excluded set X_i) the k candidates j not in X_i with the best exact score, ties -> lower position:
// kL2 the smallest d_j = |q_i - p_j|^2, kDot the largest s_j = h_i . t_j, both by exact_score<Kind, 16>.  The counting
// GEMM serves as a candidate filter (DESIGN.md §6):
//   1. lkg_topk_threshold_*  theta_i = the exact k-th best score among S strided samples not in X_i (so at least k
//                            admissible candidates score at least as well: the true k-th best is no worse than
//                            theta_i), and thr_i = {lo, +inf}: kL2 lo = sigma - M with sigma = (|u|^2 - theta_i) / 2
//                            and M = l2_band_margin, kDot lo = theta_i - h . c - M with M = dot_band_margin;
//   2. lkg_score_rank        lists every column with g_j >= lo (above stays 0): g_j < lo implies that j scores worse
//                            than theta_i, so every top-k member is listed;
//   3. lkg_topk_finalize_*   the listed columns re-scored exactly, X_i dropped, sorted, first k written; a query
//                            whose list overflowed is re-scanned exactly.
constexpr int kTopkThreads = 256;
constexpr int kThetaChunk = 1024;        // samples scored per round of the threshold kernel
constexpr int kThetaBuf = 2048;          // kept distances: after a round <= k + kThetaChunk <= 2048 (k <= 1024)
constexpr int kTopkMaxK = 1024;
constexpr int kTopkMaxCap = 16384;
constexpr int kTopkRow = 512;            // staged query row: the distance's augmented width, the dot score's dim
static_assert(row_floats<kL2>() == kTopkRow, "the distance instances stage their rows as before");

// M of the dot band: with the GEMM value g_j = h . w_j (w_j = fl(t_j - c), the centred candidate operand) of a
// candidate, g_j < theta - hc - M implies s_j = fl(h . t_j) < theta (derivation in DESIGN.md §6, "Filtered top-k
// under the dot score").  hh = |h|^2, hc = h . c and hca = sum |h_k c_k|, all three summed in fp64; max_w = max_j |w_j|
// as lkg_score_index records it (scaled units, fp32 sums); inv_q, inv_c: the inverse scales (record slot 2) of the
// query's and the candidates' planes.  W = max_w inv_c (1 + 2^-15) bounds max_j |w_j| in real units (the recorded norm
// is off by less than 2^-19 relative: <= 64 fp32 additions of positive squares, a square root, the factor 1.000001).
// Terms: the 3-product GEMM's error E at K = dim; the rounding of the centred rows, |h . (w_j - (t_j - c))| <=
// 2^-24 |h| W; the fp64 sum of h . c over <= 512 products, <= 2^-43 hca; half an ulp of theta, <= 2^-24 |theta|
// (2^-149 for a subnormal); and the fp64 roundings of theta - hc - M.
__device__ __forceinline__ double dot_band_margin(double hh, double hc, double hca, double theta, int dim, float max_w,
                                                  float inv_q, float inv_c) {
    const double w = (double)max_w * inv_c * (1.0 + 0x1p-15);
    const double nh = __dsqrt_ru(hh) * (1.0 + 0x1p-40);
    const double e = rank_err(dim) * nh * w + 0x1p-24 * sqrt((double)dim) * 1.001 * (w * inv_q + nh * inv_c);
    const double r = 0x1p-24 * nh * w * (1.0 + 0x1p-20);
    return e + r + 0x1p-43 * hca + 0x1p-24 * fabs(theta) + 0x1p-149 + (fabs(theta) + fabs(hc)) * 0x1p-40 + 1e-30;
}

// What the dot instances of the top-k kernels read besides the distance instances' arguments (which they read as:
// cand = the embedding rows of the candidates, query = the embedding rows of the anchors, stats = max_j |w_j| of the
// centred candidate operand in its planes' scaled units, aug unused).
struct TopkDot {
    const int64_t* cand_rows;    // nullable: candidate position p -> row of cand
    const int64_t* query_rows;   // nullable: query i -> row of query
    const float* center;         // [dim] c, the centre the candidate operand was shifted by
};

// The excluded set of a query: the entities of the (anchors[i], rels[i]) run of a known plan (g.att_rowptr NULL: none;
// rels NULL: of any relation), looked up by the entity id of a candidate position (cand_ids NULL: position = id).
struct TopkExclude {
    lkg_graph g;
    const int64_t* anchors;
    const int64_t* rels;
    const int64_t* cand_ids;
};

struct KnownRun {
    const int32_t* ent;      // sorted by entity id; duplicate triples repeat an id, which a lower bound passes over
    int lo, hi;
    __device__ bool has(int64_t e) const {
        int l = lo, u = hi;
        while (l < u) {
            const int m = (l + u) >> 1;
            if (ent[m] < e) l = m + 1; else u = m;
        }
        return l < hi && ent[l] == e;
    }
};

__device__ __forceinline__ KnownRun known_run(const TopkExclude& x, int qi) {
    KnownRun run{nullptr, 0, 0};
    if (x.g.att_rowptr) filter_run(x.g, x.anchors[qi], x.rels ? x.rels[qi] : -1, &run.ent, &run.lo, &run.hi);
    return run;
}

__device__ __forceinline__ bool is_excluded(const KnownRun& run, const TopkExclude& x, int p) {
    return run.hi > run.lo && run.has(x.cand_ids ? x.cand_ids[p] : (int64_t)p);
}

// The exact score of candidate position p under the top-k kernels' instance of the scorer: s = h . t_p on the
// uncentred rows, or s = -d_p (larger is better for both).
template <int Kind>
__device__ __forceinline__ float topk_score(const float* s_q, const float* cand, int64_t ld, const TopkDot& dot, int p,
                                            int dim, int q, bool live) {
    const int64_t row = Kind == kDot && dot.cand_rows ? dot.cand_rows[p] : (int64_t)p;
    return exact_score<Kind, kTopkRow / 32>(s_q, cand + row * ld, dim, q, live);
}

template <int Kind>
__device__ __forceinline__ const float* topk_query_row(const float* query, int64_t ld_q, const TopkDot& dot, int qi) {
    return query + (Kind == kDot && dot.query_rows ? dot.query_rows[qi] : (int64_t)qi) * ld_q;
}

// One CTA per query.  Samples i = 0 .. n_sample - 1 at positions floor(i n_cand / n_sample), kThetaChunk per round;
// a sample enters the buffer only when it scores better than the current k-th best (theta so far), and the buffer is
// sorted and cut to k when the next round might not fit.  Exact selection: theta is a real admissible score.
template <int Kind>
__global__ void __launch_bounds__(kTopkThreads) topk_threshold_kernel(
    const float* __restrict__ cand, int64_t ld, int n_cand, const float* __restrict__ query, int64_t ld_q,
    const float* __restrict__ aug, int64_t ld_aug, int dim, int k, int n_sample, const float* __restrict__ stats,
    const float* __restrict__ rec_q, const float* __restrict__ rec_c, const TopkExclude x, float* __restrict__ thr,
    float* __restrict__ theta, const TopkDot dot) {
    __shared__ __align__(16) float s_q[kTopkRow];
    __shared__ unsigned long long keys[kThetaBuf];       // enc(s) << 32: a descending sort puts the best first
    __shared__ int s_cnt;
    __shared__ float s_theta;                            // the k-th best score s so far (kL2: s = -d)
    __shared__ RowSums s_rs;
    const int qi = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int grp = lane >> 3, q = lane & 7;
    const float* qrow = topk_query_row<Kind>(query, ld_q, dot, qi);
    stage_row<kTopkRow>(s_q, qrow, dim);
    const float* arow = aug + (int64_t)qi * ld_aug;
    if (warp == 0) {
        // kL2: |u|^2 of the query operand; kDot: |h|^2, h . c and sum |h_k c_k| of the anchor row
        const RowSums rs = Kind == kDot ? row_sums<32>(qrow, dot.center, dim, lane) : row_sums<32>(arow, nullptr, dim, lane);
        if (lane == 0) {
            s_rs = rs;
            s_cnt = 0;
            s_theta = -INFINITY;
        }
    }
    const KnownRun run = known_run(x, qi);
    __syncthreads();
    for (int base = 0; base < n_sample; base += kThetaChunk) {
        const int chunk = min(kThetaChunk, n_sample - base);
        const float bound = s_theta;
        for (int c0 = 4 * warp; c0 < chunk; c0 += 4 * nwarps) {   // uniform per warp: the exact scores shuffle
            const int c = c0 + grp;
            const bool live = c < chunk;
            const int p = live ? (int)((int64_t)(base + c) * n_cand / n_sample) : 0;
            const float s = topk_score<Kind>(s_q, cand, ld, dot, p, dim, q, live);
            if (live && q == 0 && s > bound && !is_excluded(run, x, p))
                keys[atomicAdd(&s_cnt, 1)] = (unsigned long long)enc(s) << 32;
        }
        __syncthreads();
        const int cnt = s_cnt;
        __syncthreads();                                 // every thread has read cnt before the next round adds to it
        if (cnt > kThetaBuf - kThetaChunk || base + kThetaChunk >= n_sample) {
            sort_keys_desc(keys, cnt);
            if (threadIdx.x == 0) {
                if (cnt >= k) s_theta = dec((uint32_t)(keys[k - 1] >> 32));
                s_cnt = min(cnt, k);
            }
            __syncthreads();
        }
    }
    if (threadIdx.x == 0) {
        const float th = Kind == kL2 ? -s_theta : s_theta;          // theta: the k-th best s, or d for kL2
        float lo = -INFINITY;                            // fewer than k admissible samples: every column is listed
        if (s_theta > -INFINITY) {
            if constexpr (Kind == kDot) {
                const double hc = s_rs.ac;
                lo = __double2float_rd(((double)th - hc) - dot_band_margin(s_rs.aa, hc, s_rs.aca, th, dim, __ldg(stats),
                                                                           __ldg(rec_q + 2), __ldg(rec_c + 2)));
            } else {
                const double uu = s_rs.aa, sigma = 0.5 * (uu - (double)th);
                lo = __double2float_rd(sigma - l2_band_margin(uu, arow[dim], th, dim, stats, __ldg(rec_q + 2),
                                                              __ldg(rec_c + 2)));
            }
        }
        thr[2 * qi] = lo;
        thr[2 * qi + 1] = INFINITY;
        if (theta) theta[qi] = th;
    }
}

// One CTA per query.  keys [next_pow2(cap)]: (enc(s) << 32) | ~position; an excluded or missing entry is key 0, which
// sorts last and is never written out.
template <int Kind>
__global__ void __launch_bounds__(kTopkThreads) topk_finalize_kernel(
    const float* __restrict__ cand, int64_t ld, int n_cand, const float* __restrict__ query, int64_t ld_q, int dim,
    const int* __restrict__ band_cnt, const int* __restrict__ band, int cap, int k, const TopkExclude x,
    float* __restrict__ dist, int64_t* __restrict__ pos, const TopkDot dot) {
    extern __shared__ unsigned long long keys[];
    __shared__ __align__(16) float s_q[kTopkRow];
    const int qi = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int grp = lane >> 3, q = lane & 7;
    stage_row<kTopkRow>(s_q, topk_query_row<Kind>(query, ld_q, dot, qi), dim);
    const KnownRun run = known_run(x, qi);
    __syncthreads();
    auto score = [&](int p, int q, bool live) { return topk_score<Kind>(s_q, cand, ld, dot, p, dim, q, live); };
    auto key = [&](float s, int p) -> unsigned long long {
        return is_excluded(run, x, p) ? 0ull : ((unsigned long long)enc(s) << 32) | (uint32_t)(~(uint32_t)p);
    };
    const int n_band = band_cnt[qi];
    int n;
    if (n_band <= cap) {
        n = n_band;
        const int* list = band + (int64_t)qi * cap;
        for (int c0 = 4 * warp; c0 < n; c0 += 4 * nwarps) {
            const int c = c0 + grp;
            const bool live = c < n;
            const int p = live ? list[c] : 0;
            const float s = score(p, q, live);
            if (live && q == 0) keys[c] = key(s, p);
        }
        sort_keys_desc(keys, n);
    } else {
        // Overflow (more than cap columns listed, e.g. a weak theta or a plateau of equal scores): exact scan of
        // every candidate, as score_finalize_kernel does (cap / 2 >= k is checked).
        n = scan_best(keys, n_cand, cap / 2, score, key);
    }
    write_first_k<Kind>(keys, n, k, dist + (int64_t)qi * k, pos + (int64_t)qi * k);
}

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

}  // namespace
}  // namespace lkg

using namespace lkg;

extern "C" int lkg_score_index(const float* emb, int64_t ld, const int64_t* rows, int64_t m, int32_t dim,
                               const float* rec, uint16_t* hi, int64_t ld_hi, float* norms, float* max_norm,
                               void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    LKG_REQUIRE(emb && rec && hi && norms && max_norm && m >= 0 && dim > 0, "null / bad argument");
    LKG_REQUIRE(ld_hi % 8 == 0 && ld_hi >= dim && aligned16(hi) && aligned16(emb), "hi plane rows must be 16-byte aligned");
    LKG_CUDA(cudaMemsetAsync(max_norm, 0, sizeof(float), stream));
    if (m == 0) return LKG_OK;
    int64_t blocks = (m * 32 + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    score_index_kernel<<<(int)(blocks > cap ? cap : blocks), 256, 0, stream>>>(emb, ld, rows, m, dim, rec, (__half*)hi,
                                                                              ld_hi, norms, max_norm);
    LKG_LAUNCH_CHECK("score_index_kernel");
    return LKG_OK;
}

extern "C" int lkg_shift_rows(const float* src, int64_t ld, const int64_t* rows, int64_t m, int32_t k, const float* center,
                              float* out, int64_t ld_out, void* stream_) {
    LKG_REQUIRE(src && center && out && m >= 0 && k > 0 && ld_out >= k, "bad shift arguments");
    if (m == 0) return LKG_OK;
    int64_t blocks = (m * k + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    shift_rows_kernel<<<(unsigned)(blocks > cap ? cap : blocks), 256, 0, (cudaStream_t)stream_>>>(src, ld, rows, m, k, center,
                                                                                            out, ld_out);
    LKG_LAUNCH_CHECK("shift_rows_kernel");
    return LKG_OK;
}

// The rows the dot rank kernels score with exact_score<kDot, 8>: float4 loads of widths up to the GEMM's K.
static int check_rank_rows(const float* emb, int64_t ld_emb, const float* head_emb, int64_t ld_head_emb, int32_t dim) {
    LKG_REQUIRE(dim >= 4 && dim % 4 == 0 && dim <= kMaxChunks * kBK && ld_emb % 4 == 0 && ld_head_emb % 4 == 0 &&
                    aligned16(emb) && aligned16(head_emb),
                "the rank path supports dim %% 4 == 0, dim <= %d, 16-byte aligned rows", kMaxChunks * kBK);
    return LKG_OK;
}

extern "C" int lkg_rank_prepare(const float* emb, int64_t ld_emb, const int64_t* tail_rows, const float* head_emb,
                                int64_t ld_head_emb, const int64_t* head_rows, const int64_t* target_pos, int64_t n_heads,
                                int32_t dim, const float* tail_max_norm, const float* rec, const float* center,
                                float* tau, float* thr, void* stream_) {
    LKG_REQUIRE(emb && head_emb && target_pos && tail_max_norm && rec && tau && thr && n_heads >= 0 &&
                    n_heads < (1ll << 31) && dim > 0,
                "bad rank arguments");
    if (int rc = check_rank_rows(emb, ld_emb, head_emb, ld_head_emb, dim)) return rc;
    if (n_heads == 0) return LKG_OK;
    const int64_t blocks = (n_heads * 8 + 255) / 256;
    rank_prepare_kernel<kDot><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(emb, ld_emb, tail_rows, head_emb,
                                                                                   ld_head_emb, head_rows, target_pos,
                                                                                   (int)n_heads, dim, tail_max_norm, rec,
                                                                                   center, tau, thr, L2Prep{});
    LKG_LAUNCH_CHECK("rank_prepare_kernel<dot>");
    return LKG_OK;
}

extern "C" int lkg_rank_finalize(const float* emb, int64_t ld_emb, const int64_t* tail_rows, const float* head_emb,
                                 int64_t ld_head_emb, const int64_t* head_rows, const int64_t* target_pos,
                                 const float* tau, const int32_t* above, const int32_t* band_cnt, const int32_t* band,
                                 int32_t band_cap, int64_t n_heads, int64_t n_tails, int32_t dim, int64_t* ranks,
                                 void* stream_) {
    LKG_REQUIRE(emb && head_emb && target_pos && tau && above && band_cnt && band && ranks && band_cap > 0 &&
                    n_tails < (1ll << 31),
                "bad rank arguments");
    if (int rc = check_rank_rows(emb, ld_emb, head_emb, ld_head_emb, dim)) return rc;
    if (n_heads == 0) return LKG_OK;
    rank_finalize_kernel<kDot><<<(unsigned)n_heads, 256, 0, (cudaStream_t)stream_>>>(emb, ld_emb, tail_rows, head_emb, ld_head_emb,
                                                                               head_rows, target_pos, tau, above, band_cnt,
                                                                               band, band_cap, (int)n_tails, dim, ranks);
    LKG_LAUNCH_CHECK("rank_finalize_kernel<dot>");
    return LKG_OK;
}

static int check_filter_args(const lkg_graph* known, const int64_t* heads, const int64_t* target_pos, int64_t n_queries,
                             int64_t* ranks) {
    LKG_REQUIRE(known && known->att_rowptr && known->att_tail && known->att_rel && known->rowptr && known->col,
                "the known plan needs its att and agg arrays");
    LKG_REQUIRE(heads && target_pos && ranks && n_queries >= 0 && n_queries < (1ll << 31), "bad filter arguments");
    return LKG_OK;
}

extern "C" int lkg_rank_filter(const lkg_graph* known, const int64_t* heads, const int64_t* rels,
                               const int32_t* cand_map, const int64_t* target_pos, int64_t n_queries, const float* emb,
                               int64_t ld_emb, int32_t dim, const float* tau, int64_t* ranks, void* stream_) {
    if (int rc = check_filter_args(known, heads, target_pos, n_queries, ranks)) return rc;
    LKG_REQUIRE(emb && tau, "bad filter arguments");
    if (int rc = check_rank_rows(emb, ld_emb, emb, ld_emb, dim)) return rc;
    if (n_queries == 0) return LKG_OK;
    rank_filter_kernel<kDot><<<(unsigned)n_queries, 256, 0, (cudaStream_t)stream_>>>(*known, heads, rels, cand_map,
                                                                                    target_pos, emb, ld_emb, dim, tau,
                                                                                    ranks, nullptr, 0);
    LKG_LAUNCH_CHECK("rank_filter_kernel<exact>");
    return LKG_OK;
}

extern "C" int lkg_rank_filter_scores(const lkg_graph* known, const int64_t* heads, const int64_t* rels,
                                      const int32_t* cand_map, const int64_t* target_pos, int64_t n_queries,
                                      const float* scores, int64_t ld_scores, int64_t n_cols, int64_t* ranks,
                                      void* stream_) {
    if (int rc = check_filter_args(known, heads, target_pos, n_queries, ranks)) return rc;
    LKG_REQUIRE(scores && n_cols >= 1 && ld_scores >= n_cols, "bad score matrix");
    LKG_REQUIRE(cand_map || n_cols == known->n_entities,
                "without a candidate map the score matrix needs one column per entity of the known plan");
    if (n_queries == 0) return LKG_OK;
    rank_filter_kernel<kScores><<<(unsigned)n_queries, 256, 0, (cudaStream_t)stream_>>>(*known, heads, rels, cand_map,
                                                                                     target_pos, scores, ld_scores, 0,
                                                                                     nullptr, ranks, nullptr, 0);
    LKG_LAUNCH_CHECK("rank_filter_kernel<scores>");
    return LKG_OK;
}

// ---- distance rank (triple score) --------------------------------------------------------------------------------
// The rows of the distance paths (kL2: dim <= 508, the augmented width dim + 4 <= 512) and of the dot top-k (kDot:
// dim <= 512): float4 loads by the exact scorer.
template <int Kind>
static int check_rows(const char* what, const float* p, int64_t ld, int32_t dim) {
    constexpr int max_dim = Kind == kL2 ? kL2MaxDim : kTopkRow;
    LKG_REQUIRE(p, "%s is null", what);
    LKG_REQUIRE(dim >= 4 && dim % 4 == 0 && dim <= max_dim, "the %s path supports dim %% 4 == 0, 4 <= dim <= %d%s, got %d",
                Kind == kL2 ? "distance rank" : "dot top-k", max_dim,
                Kind == kL2 ? " (augmented width dim + 4 <= 512)" : "", dim);
    LKG_REQUIRE(ld >= dim && ld % 4 == 0 && aligned16(p), "%s rows must be 16-byte aligned (ld %% 4 == 0, ld >= dim)",
                what);
    return LKG_OK;
}

extern "C" int lkg_l2_rank_rows(const float* src, int64_t ld, const int64_t* rows, int64_t m, int32_t dim,
                                const float* center, int32_t mode, float* stats, float* out, int64_t ld_out,
                                void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (int rc = check_rows<kL2>("src", src, ld, dim)) return rc;
    LKG_REQUIRE(center && aligned16(center), "center must be a 16-byte aligned [dim] vector");
    LKG_REQUIRE(stats && out && m >= 0, "bad operand arguments (stats, out, m)");
    LKG_REQUIRE(ld_out >= dim + 4 && ld_out % 4 == 0 && aligned16(out),
                "out rows need dim + 4 columns and 16-byte alignment (ld_out %% 4 == 0)");
    LKG_REQUIRE(mode == LKG_L2_QUERY || mode == LKG_L2_CANDIDATE, "mode must be LKG_L2_QUERY or LKG_L2_CANDIDATE");
    if (mode == LKG_L2_CANDIDATE) LKG_CUDA(cudaMemsetAsync(stats, 0, 2 * sizeof(float), stream));
    if (m == 0) return LKG_OK;
    const int64_t blocks = (m * 32 + 255) / 256, cap = (int64_t)sm_count() * 16;
    const unsigned grid = (unsigned)(blocks > cap ? cap : blocks);
    for (int pass = mode == LKG_L2_CANDIDATE ? 0 : 2; pass < (mode == LKG_L2_CANDIDATE ? 2 : 3); ++pass) {
        l2_rank_rows_kernel<<<grid, 256, 0, stream>>>(src, ld, rows, m, dim, center, pass, stats, out, ld_out);
        LKG_LAUNCH_CHECK("l2_rank_rows_kernel");
    }
    return LKG_OK;
}

extern "C" int lkg_rank_prepare_l2(const float* cand, int64_t ld_cand, const float* query, int64_t ld_query,
                                   const float* query_aug, int64_t ld_aug, const int64_t* target_pos, int64_t n_queries,
                                   int32_t dim, const float* stats, const float* rec_query, const float* rec_cand,
                                   float* tau, float* thr, void* stream_) {
    if (int rc = check_rows<kL2>("cand", cand, ld_cand, dim)) return rc;
    if (int rc = check_rows<kL2>("query", query, ld_query, dim)) return rc;
    LKG_REQUIRE(query_aug && ld_aug >= dim + 4 && ld_aug % 4 == 0 && aligned16(query_aug),
                "query_aug rows need dim + 4 columns and 16-byte alignment");
    LKG_REQUIRE(target_pos && stats && rec_query && rec_cand && tau && thr && n_queries >= 0 && n_queries < (1ll << 31),
                "bad rank arguments");
    if (n_queries == 0) return LKG_OK;
    const L2Prep l2{query_aug, ld_aug, rec_query};
    rank_prepare_kernel<kL2><<<(unsigned)((n_queries * 8 + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(
        cand, ld_cand, nullptr, query, ld_query, nullptr, target_pos, (int)n_queries, dim, stats, rec_cand, nullptr, tau,
        thr, l2);
    LKG_LAUNCH_CHECK("rank_prepare_kernel<l2>");
    return LKG_OK;
}

extern "C" int lkg_rank_finalize_l2(const float* cand, int64_t ld_cand, const float* query, int64_t ld_query,
                                    const int64_t* target_pos, const float* tau, const int32_t* above,
                                    const int32_t* band_cnt, const int32_t* band, int32_t band_cap, int64_t n_queries,
                                    int64_t n_cand, int32_t dim, int64_t* ranks, void* stream_) {
    if (int rc = check_rows<kL2>("cand", cand, ld_cand, dim)) return rc;
    if (int rc = check_rows<kL2>("query", query, ld_query, dim)) return rc;
    LKG_REQUIRE(target_pos && tau && above && band_cnt && band && ranks && band_cap > 0 && n_queries >= 0 &&
                    n_queries < (1ll << 31) && n_cand >= 0 && n_cand < (1ll << 31),
                "bad rank arguments");
    if (n_queries == 0) return LKG_OK;
    rank_finalize_kernel<kL2><<<(unsigned)n_queries, 256, 0, (cudaStream_t)stream_>>>(
        cand, ld_cand, nullptr, query, ld_query, nullptr, target_pos, tau, above, band_cnt, band, band_cap, (int)n_cand,
        dim, ranks);
    LKG_LAUNCH_CHECK("rank_finalize_kernel<l2>");
    return LKG_OK;
}

extern "C" int lkg_rank_filter_l2(const lkg_graph* known, const int64_t* anchors, const int64_t* rels,
                                  const int32_t* cand_map, const int64_t* target_pos, int64_t n_queries,
                                  const float* cand, int64_t ld_cand, const float* query, int64_t ld_query, int32_t dim,
                                  const float* tau, int64_t* ranks, void* stream_) {
    if (int rc = check_filter_args(known, anchors, target_pos, n_queries, ranks)) return rc;
    if (int rc = check_rows<kL2>("cand", cand, ld_cand, dim)) return rc;
    if (int rc = check_rows<kL2>("query", query, ld_query, dim)) return rc;
    LKG_REQUIRE(tau, "bad filter arguments");
    if (n_queries == 0) return LKG_OK;
    rank_filter_kernel<kL2><<<(unsigned)n_queries, 256, 0, (cudaStream_t)stream_>>>(*known, anchors, rels, cand_map,
                                                                                   target_pos, cand, ld_cand, dim, tau,
                                                                                   ranks, query, ld_query);
    LKG_LAUNCH_CHECK("rank_filter_kernel<l2>");
    return LKG_OK;
}

extern "C" int lkg_score_topk_workspace_bytes(int64_t n_heads, int32_t cap, int32_t sample_tiles, size_t* bytes) {
    LKG_REQUIRE(bytes && n_heads >= 0 && cap >= 2 && (cap & (cap - 1)) == 0, "cap must be a power of two");
    LKG_REQUIRE(sample_tiles >= 0 && sample_tiles <= 4096, "sample_tiles must be in [0, 4096]");
    // counters [n_heads, <= 160 streams], thresholds, candidate sublists (n_streams * cap_s <= cap), tile maxima
    *bytes = align_up((size_t)n_heads * 160 * 4) + align_up((size_t)n_heads * 4) + align_up((size_t)n_heads * cap * 4) +
             align_up((size_t)n_heads * sample_tiles * 4);
    return LKG_OK;
}

extern "C" int lkg_score_topk(const uint16_t* heads_hi, int64_t ld_heads_hi, const float* head_norms, int64_t n_heads,
                              const uint16_t* tails_hi, int64_t ld_tails_hi, const float* tail_max_norm,
                              int64_t n_tails, int32_t dim, const float* rec, const float* theta,
                              int64_t theta_stride, int32_t sample_tiles, const float* emb, int64_t ld_emb,
                              const float* head_emb, int64_t ld_head_emb, const int64_t* head_rows,
                              const int64_t* tail_rows, int32_t k, int32_t cap,
                              float* top_values, int64_t* top_cols, void* workspace, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    LKG_REQUIRE(n_heads >= 0 && n_tails >= 1 && n_tails < (1ll << 31) - kBN, "bad shape");
    LKG_REQUIRE(dim >= 4 && dim % 4 == 0 && dim <= kMaxChunks * kBK,
                "the fused scoring path supports dim %% 4 == 0, dim <= %d (got %d)", kMaxChunks * kBK, dim);
    LKG_REQUIRE(ld_emb % 4 == 0 && aligned16(emb) && (!head_emb || (ld_head_emb % 4 == 0 && aligned16(head_emb))),
                "embedding rows must be 16-byte aligned");
    LKG_REQUIRE(k >= 1 && cap >= 2 * k && (cap & (cap - 1)) == 0 && cap <= 16384,
                "cap must be a power of two in [2k, 16384]");
    if (n_heads == 0) return LKG_OK;
    LKG_REQUIRE(heads_hi && head_norms && tails_hi && tail_max_norm && rec && emb && top_values && top_cols && workspace,
                "null argument");
    char* ws = static_cast<char*>(workspace);
    int* cnt = reinterpret_cast<int*>(ws);
    float* thr = reinterpret_cast<float*>(ws + align_up((size_t)n_heads * 160 * 4));
    int* cand = reinterpret_cast<int*>(ws + align_up((size_t)n_heads * 160 * 4) + align_up((size_t)n_heads * 4));
    float* tilemax = reinterpret_cast<float*>(ws + align_up((size_t)n_heads * 160 * 4) + align_up((size_t)n_heads * 4) +
                                              align_up((size_t)n_heads * cap * 4));
    if (theta || sample_tiles <= 0) {
        score_threshold_kernel<<<(int)((n_heads + 255) / 256), 256, 0, stream>>>(theta, theta_stride, (int)n_heads,
                                                                                head_norms, tail_max_norm, rec, dim, thr);
        LKG_LAUNCH_CHECK("score_threshold_kernel");
    }
    const int n_tiles_all = (int)((n_tails + kBN - 1) / kBN);
    int n_st = 0, st_stride = 1;
    if (!theta && sample_tiles > 0) {
        LKG_REQUIRE(sample_tiles <= 4096, "sample_tiles must be <= 4096");
        st_stride = n_tiles_all / sample_tiles > 0 ? n_tiles_all / sample_tiles : 1;
        n_st = (n_tiles_all + st_stride - 1) / st_stride;
        if (n_st > sample_tiles) n_st = sample_tiles;
    }

    const int sms = sm_count() < 160 ? sm_count() : 160;
    const int max_pairs = sms;                      // heads per launch <= 256 * SMs
    auto kern = score_filter_kernel;
    LKG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFilterSmem));
    const size_t fsmem = (size_t)cap * (sizeof(unsigned long long) + sizeof(int));
    LKG_CUDA(cudaFuncSetAttribute(score_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
    for (int64_t h0 = 0; h0 < n_heads; h0 += (int64_t)max_pairs * 2 * kBM) {
        const int nh = (int)((n_heads - h0) < (int64_t)max_pairs * 2 * kBM ? (n_heads - h0) : (int64_t)max_pairs * 2 * kBM);
        FilterParams p{};
        if (int rc = make_map_2d(&p.a_map, heads_hi + h0 * ld_heads_hi, nh, dim, ld_heads_hi)) return rc;
        if (int rc = make_map_2d(&p.b_map, tails_hi, n_tails, dim, ld_tails_hi)) return rc;
        p.n_heads = nh;
        p.n_tails = (int)n_tails;
        p.n_chunks = (dim + kBK - 1) / kBK;
        p.n_pairs = (nh + 2 * kBM - 1) / (2 * kBM);
        p.thr = thr + h0;
        // pass 0 (optional): tile maxima over the sampled tiles -> thresholds; pass 1: filter over all tiles
        int streams = 1;
        for (int pass = (n_st > 0 ? 0 : 1); pass < 2; ++pass) {
            p.n_tiles = pass == 0 ? n_st : n_tiles_all;
            p.tile_stride = pass == 0 ? st_stride : 1;
            p.tilemax = pass == 0 ? tilemax + h0 * n_st : nullptr;
            streams = sms / p.n_pairs;
            if (streams > p.n_tiles) streams = p.n_tiles;
            p.cnt = cnt + h0 * 160;
            p.cand = cand + h0 * cap;
            p.cap_s = cap / streams;
            kern<<<p.n_pairs * streams, kThreads, kFilterSmem, stream>>>(p);
            LKG_LAUNCH_CHECK("score_filter_kernel");
            if (pass == 0) {
                int p2 = 1;
                while (p2 < n_st) p2 <<= 1;
                score_sample_threshold_kernel<<<(unsigned)nh, 256, p2 * sizeof(unsigned long long), stream>>>(
                    p.tilemax, n_st, k, head_norms + h0, tail_max_norm, dim, thr + h0);
                LKG_LAUNCH_CHECK("score_sample_threshold_kernel");
            }
        }

        FinalParams f{};
        f.emb = emb;
        f.ld_emb = ld_emb;
        f.head_emb = head_emb ? head_emb : emb;
        f.ld_head_emb = head_emb ? ld_head_emb : ld_emb;
        f.head_rows = head_rows ? head_rows + h0 : nullptr;
        f.head_row_base = head_rows ? 0 : h0;
        f.tail_rows = tail_rows;
        f.n_heads = nh;
        f.n_tails = (int)n_tails;
        f.dim = dim;
        f.k = k;
        f.cap = cap;
        f.n_streams = streams;
        f.cap_s = cap / streams;
        f.cnt = cnt + h0 * 160;
        f.cand = cand + h0 * cap;
        f.top_val = top_values + h0 * k;
        f.top_col = top_cols + h0 * k;
        score_finalize_kernel<<<(unsigned)nh, kFinalThreads, fsmem, stream>>>(f);
        LKG_LAUNCH_CHECK("score_finalize_kernel");
    }
    return LKG_OK;
}

// ---- relation-aware top-k under the distance ----------------------------------------------------------------------
static int topk_exclude(const lkg_graph* known, const int64_t* anchors, const int64_t* rels, const int64_t* cand_ids,
                        TopkExclude* x) {
    *x = TopkExclude{};
    if (!known) return LKG_OK;
    LKG_REQUIRE(known->att_rowptr && known->att_tail && known->att_rel && known->rowptr && known->col,
                "the known plan needs its att and agg arrays");
    LKG_REQUIRE(anchors, "the anchors are required with a known plan");
    x->g = *known;
    x->anchors = anchors;
    x->rels = rels;
    x->cand_ids = cand_ids;
    return LKG_OK;
}

// The checks and the launch the two kinds of the top-k threshold share (the rows and the kind's own operands are
// checked by the caller).
template <int Kind>
static int launch_topk_threshold(const float* cand, int64_t ld_cand, int64_t n_cand, const float* query,
                                 int64_t ld_query, const float* aug, int64_t ld_aug, int64_t n_queries, int32_t dim,
                                 const float* stats, const float* rec_query, const float* rec_cand, int32_t k,
                                 int32_t n_sample, const lkg_graph* known, const int64_t* anchors, const int64_t* rels,
                                 const int64_t* cand_ids, float* thr, float* theta, const TopkDot& dot,
                                 cudaStream_t stream) {
    LKG_REQUIRE(n_queries >= 0 && n_queries < (1ll << 31) && n_cand >= 1 && n_cand < (1ll << 31),
                "bad top-k shape (n_queries, n_cand)");
    LKG_REQUIRE(k >= 1 && k <= kTopkMaxK, "k must be in [1, %d], got %d", kTopkMaxK, k);
    LKG_REQUIRE(n_sample >= 1 && n_sample <= n_cand, "n_sample must be in [1, n_cand], got %d", n_sample);
    TopkExclude x;
    if (int rc = topk_exclude(known, anchors, rels, cand_ids, &x)) return rc;
    if (n_queries == 0) return LKG_OK;
    topk_threshold_kernel<Kind><<<(unsigned)n_queries, kTopkThreads, 0, stream>>>(
        cand, ld_cand, (int)n_cand, query, ld_query, aug, ld_aug, dim, k, n_sample, stats, rec_query, rec_cand, x, thr,
        theta, dot);
    LKG_LAUNCH_CHECK(Kind == kL2 ? "topk_threshold_kernel<l2>" : "topk_threshold_kernel<dot>");
    return LKG_OK;
}

// The same for the top-k finalize: shape, k, cap, the excluded set and the sort buffer (next_pow2(cap) keys).
template <int Kind>
static int launch_topk_finalize(const float* cand, int64_t ld_cand, int64_t n_cand, const float* query,
                                int64_t ld_query, int64_t n_queries, int32_t dim, const int32_t* band_cnt,
                                const int32_t* band, int32_t cap, int32_t k, const lkg_graph* known,
                                const int64_t* anchors, const int64_t* rels, const int64_t* cand_ids, float* val,
                                int64_t* pos, const TopkDot& dot, cudaStream_t stream) {
    LKG_REQUIRE(n_queries >= 0 && n_queries < (1ll << 31) && n_cand >= 1 && n_cand < (1ll << 31),
                "bad top-k shape (n_queries, n_cand)");
    LKG_REQUIRE(k >= 1 && k <= kTopkMaxK, "k must be in [1, %d], got %d", kTopkMaxK, k);
    LKG_REQUIRE(cap >= 2 * k && cap <= kTopkMaxCap, "cap must be in [2k, %d], got %d (k = %d)", kTopkMaxCap, cap, k);
    TopkExclude x;
    if (int rc = topk_exclude(known, anchors, rels, cand_ids, &x)) return rc;
    if (n_queries == 0) return LKG_OK;
    int p2 = 1;
    while (p2 < cap) p2 <<= 1;
    const int smem = p2 * (int)sizeof(unsigned long long);
    LKG_CUDA(cudaFuncSetAttribute(topk_finalize_kernel<Kind>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    topk_finalize_kernel<Kind><<<(unsigned)n_queries, kTopkThreads, smem, stream>>>(
        cand, ld_cand, (int)n_cand, query, ld_query, dim, band_cnt, band, cap, k, x, val, pos, dot);
    LKG_LAUNCH_CHECK(Kind == kL2 ? "topk_finalize_kernel<l2>" : "topk_finalize_kernel<dot>");
    return LKG_OK;
}

extern "C" int lkg_topk_threshold_l2(const float* cand, int64_t ld_cand, int64_t n_cand, const float* query,
                                     int64_t ld_query, const float* query_aug, int64_t ld_aug, int64_t n_queries,
                                     int32_t dim, const float* stats, const float* rec_query, const float* rec_cand,
                                     int32_t k, int32_t n_sample, const lkg_graph* known, const int64_t* anchors,
                                     const int64_t* rels, const int64_t* cand_ids, float* thr, float* theta,
                                     void* stream_) {
    if (int rc = check_rows<kL2>("cand", cand, ld_cand, dim)) return rc;
    if (int rc = check_rows<kL2>("query", query, ld_query, dim)) return rc;
    LKG_REQUIRE(query_aug && ld_aug >= dim + 4 && ld_aug % 4 == 0 && aligned16(query_aug),
                "query_aug rows need dim + 4 columns and 16-byte alignment");
    LKG_REQUIRE(stats && rec_query && rec_cand && thr, "bad top-k arguments (stats, rec_query, rec_cand, thr)");
    return launch_topk_threshold<kL2>(cand, ld_cand, n_cand, query, ld_query, query_aug, ld_aug, n_queries, dim, stats,
                                      rec_query, rec_cand, k, n_sample, known, anchors, rels, cand_ids, thr, theta,
                                      TopkDot{}, (cudaStream_t)stream_);
}

extern "C" int lkg_topk_finalize_l2(const float* cand, int64_t ld_cand, int64_t n_cand, const float* query,
                                    int64_t ld_query, int64_t n_queries, int32_t dim, const int32_t* band_cnt,
                                    const int32_t* band, int32_t cap, int32_t k, const lkg_graph* known,
                                    const int64_t* anchors, const int64_t* rels, const int64_t* cand_ids, float* dist,
                                    int64_t* pos, void* stream_) {
    if (int rc = check_rows<kL2>("cand", cand, ld_cand, dim)) return rc;
    if (int rc = check_rows<kL2>("query", query, ld_query, dim)) return rc;
    LKG_REQUIRE(band_cnt && band && dist && pos, "bad top-k arguments (band_cnt, band, dist, pos)");
    return launch_topk_finalize<kL2>(cand, ld_cand, n_cand, query, ld_query, n_queries, dim, band_cnt, band, cap, k,
                                     known, anchors, rels, cand_ids, dist, pos, TopkDot{}, (cudaStream_t)stream_);
}

// ---- filtered top-k under the dot score -----------------------------------------------------------------------------
extern "C" int lkg_topk_threshold_dot(const float* cand, int64_t ld_cand, const int64_t* cand_rows, int64_t n_cand,
                                      const float* query, int64_t ld_query, const int64_t* query_rows,
                                      int64_t n_queries, int32_t dim, const float* center, const float* cand_max_norm,
                                      const float* rec_query, const float* rec_cand, int32_t k, int32_t n_sample,
                                      const lkg_graph* known, const int64_t* anchors, const int64_t* rels,
                                      const int64_t* cand_ids, float* thr, float* theta, void* stream_) {
    if (int rc = check_rows<kDot>("cand", cand, ld_cand, dim)) return rc;
    if (int rc = check_rows<kDot>("query", query, ld_query, dim)) return rc;
    LKG_REQUIRE(center && aligned16(center), "center must be a 16-byte aligned [dim] vector");
    LKG_REQUIRE(cand_max_norm && rec_query && rec_cand && thr,
                "bad top-k arguments (cand_max_norm, rec_query, rec_cand, thr)");
    return launch_topk_threshold<kDot>(cand, ld_cand, n_cand, query, ld_query, nullptr, 0, n_queries, dim,
                                       cand_max_norm, rec_query, rec_cand, k, n_sample, known, anchors, rels, cand_ids,
                                       thr, theta, TopkDot{cand_rows, query_rows, center}, (cudaStream_t)stream_);
}

extern "C" int lkg_topk_finalize_dot(const float* cand, int64_t ld_cand, const int64_t* cand_rows, int64_t n_cand,
                                     const float* query, int64_t ld_query, const int64_t* query_rows,
                                     int64_t n_queries, int32_t dim, const int32_t* band_cnt, const int32_t* band,
                                     int32_t cap, int32_t k, const lkg_graph* known, const int64_t* anchors,
                                     const int64_t* rels, const int64_t* cand_ids, float* score, int64_t* pos,
                                     void* stream_) {
    if (int rc = check_rows<kDot>("cand", cand, ld_cand, dim)) return rc;
    if (int rc = check_rows<kDot>("query", query, ld_query, dim)) return rc;
    LKG_REQUIRE(band_cnt && band && score && pos, "bad top-k arguments (band_cnt, band, score, pos)");
    return launch_topk_finalize<kDot>(cand, ld_cand, n_cand, query, ld_query, n_queries, dim, band_cnt, band, cap, k,
                                      known, anchors, rels, cand_ids, score, pos, TopkDot{cand_rows, query_rows, nullptr},
                                      (cudaStream_t)stream_);
}
