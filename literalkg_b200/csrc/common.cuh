// Shared helpers for liblkg (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/lkg.h"

namespace lkg {

void set_error(const char* fmt, ...);

#define LKG_FAIL(code, ...)              \
    do {                                 \
        ::lkg::set_error(__VA_ARGS__);   \
        return (code);                   \
    } while (0)

#define LKG_REQUIRE(cond, ...)                               \
    do {                                                     \
        if (!(cond)) LKG_FAIL(LKG_ERR_INVALID, __VA_ARGS__); \
    } while (0)

#define LKG_CUDA(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            LKG_FAIL(LKG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),   \
                     __FILE__, __LINE__);                                                     \
    } while (0)

#define LKG_LAUNCH_CHECK(name)                                                                \
    do {                                                                                      \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess)                                                                \
            LKG_FAIL(LKG_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(_e)); \
    } while (0)

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

inline int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// streaming 128-bit load through the read-only path, no L1 allocation (gathered rows are used once)
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}

// ---- per-warp ring of gathered rows: one cp.async.bulk (TMA unit, 1-D) per row, completion on an mbarrier ----
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ring_bar_init(uint64_t* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(bar)));
}
__device__ __forceinline__ void ring_issue(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
// two copies behind one barrier: ring_expect(total bytes) once, then ring_copy for each piece
__device__ __forceinline__ void ring_expect(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ring_copy(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void ring_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(smem_addr(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

__device__ __forceinline__ float leaky(float x) { return x > 0.f ? x : 0.01f * x; }

// ---- fp16 hi/lo operands of the tensor-core paths: s x = hi + lo, hi = fp16(s x), lo = fp16(s x - hi), s = 2^e ----
// e that parks amax * 2^e in [2^11, 2^12), clamped to [-lim, lim] (0 for a zero or non-finite amax)
__device__ __forceinline__ int plane_exp(float amax, int lim = 120) {
    int e = 0;
    if (amax > 0.f && amax < 3.0e38f) {
        int ex;
        frexpf(amax, &ex);                 // amax = f * 2^ex, f in [0.5, 1)
        e = 12 - ex;
        e = e > lim ? lim : (e < -lim ? -lim : e);
    }
    return e;
}
__device__ __forceinline__ float pow2(int e) { return __int_as_float((127 + e) << 23); }   // 2^e, |e| <= 126
// x is already multiplied by the operand's power-of-two scale
__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}

// tanh with ~2e-7 absolute error: odd polynomial near zero, (1-e)/(1+e) with e = exp(-2|x|) elsewhere
__device__ __forceinline__ float tanh_acc(float x) {
    const float ax = fabsf(x);
    const float x2 = x * x;
    float p = fmaf(x2, 2.1869488e-2f, -5.3968254e-2f);   // 62/2835, -17/315
    p = fmaf(x2, p, 1.3333334e-1f);                       // 2/15
    p = fmaf(x2, p, -3.3333334e-1f);                      // -1/3
    p = fmaf(x2 * x, p, x);
    const float e = exp2f(-2.8853900817779268f * ax);     // exp(-2|x|)
    const float q = copysignf(__fdividef(1.f - e, 1.f + e), x);
    return ax < 0.25f ? p : q;
}

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.f / (1.f + __expf(-x)); }

// ---- lane layouts of a row, shared by the aggregation layer's forward and backward ----------------------------------
// A lane layout says which channels of a row a lane holds -- N slots, slot i = channels [ch(i), ch(i) + width of Slot)
// -- and how the lanes of a row reduce.  Its Slot type says how a slot's values enter the lane's partial sums and how
// they are loaded and stored.  The order of every sum is part of the output bits, so each path keeps its own.
struct ScalarSlot {                         // one channel: sequential partial sums, squares by fma
    using V = float;
    static __device__ float& at(float& v, int) { return v; }
    static __device__ float at(const float& v, int) { return v; }
    static __device__ float add(float s, float v) { return s + v; }
    static __device__ float add_dev2(float s, float d) { return fmaf(d, d, s); }
    static __device__ float add_sq(float s, float v) { return fmaf(v, v, s); }
    static __device__ float ld(const float* q) { return __ldg(q); }
    static __device__ void st(float* q, float v) { *q = v; }
    static __device__ void st_planes(__half* q, int64_t plane_stride, float v) {
        __half h, l;
        split_f16(v, h, l);
        q[0] = h;
        q[plane_stride] = l;
    }
};
struct QuadSlot {                           // four channels: pairwise sums in the slot, 16-byte (planes: 8-byte) moves
    using V = float4;
    static __device__ float& at(float4& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }
    static __device__ float at(const float4& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }
    static __device__ float add(float s, float4 v) { return s + ((v.x + v.y) + (v.z + v.w)); }
    // squares in pairs, one product fused into the other's add; the variance and the norm pair them the opposite way
    // round, as this kernel always has (written out so that no contraction choice of the compiler can move the bits)
    static __device__ float add_dev2(float s, float4 d) {
        return s + (fmaf(d.x, d.x, d.y * d.y) + fmaf(d.z, d.z, d.w * d.w));
    }
    static __device__ float add_sq(float s, float4 v) {
        return s + (fmaf(v.y, v.y, v.x * v.x) + fmaf(v.w, v.w, v.z * v.z));
    }
    static __device__ float4 ld(const float* q) { return __ldg(reinterpret_cast<const float4*>(q)); }
    static __device__ void st(float* q, float4 v) { *reinterpret_cast<float4*>(q) = v; }
    static __device__ void st_planes(__half* q, int64_t plane_stride, float4 v) {
        __align__(8) __half h[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) split_f16(at(v, k), h[k], l[k]);
        *reinterpret_cast<uint2*>(q) = *reinterpret_cast<const uint2*>(h);
        *reinterpret_cast<uint2*>(q + plane_stride) = *reinterpret_cast<const uint2*>(l);
    }
};
template <int NC>
struct WarpChannels {                       // generic and stream per-row paths: channel lane + 32 i, the whole warp
    using Slot = ScalarSlot;
    static constexpr int N = NC;
    int lane;
    __device__ int ch(int i) const { return lane + 32 * i; }
    static __device__ float reduce(float s) { return warp_sum(s); }
};
template <int LPR, int CPL>
struct GroupQuads {                         // narrow kernel: channels 4 (gl + LPR i) + [0, 4), the LPR lanes of a group
    using Slot = QuadSlot;
    static constexpr int N = CPL;
    int gl;
    __device__ int ch(int i) const { return 4 * (gl + LPR * i); }
    static __device__ float reduce(float s) {
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
        return s;
    }
};

}  // namespace lkg
