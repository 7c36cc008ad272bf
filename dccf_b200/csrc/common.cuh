// common.cuh — shared device helpers for the DCCF sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/dccf_b200.h"

namespace dccf {

constexpr int D = DCCF_DIM;  // 64

// ------------------------------------------------------------------------------------------
// error plumbing for the C-ABI
// ------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define DCCF_CHECK_ARG(cond, ...)              \
    do {                                       \
        if (!(cond)) {                         \
            dccf::set_error(__VA_ARGS__);      \
            return DCCF_ERR_ARG;               \
        }                                      \
    } while (0)

#define DCCF_CHECK_LAUNCH(name)                                                        \
    do {                                                                               \
        cudaError_t e__ = cudaGetLastError();                                          \
        if (e__ != cudaSuccess) {                                                      \
            dccf::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));   \
            return DCCF_ERR_CUDA;                                                      \
        }                                                                              \
    } while (0)

// cudaFuncSetAttribute is PER DEVICE: one-time kernel configuration (shared-memory opt-in) is remembered per call site
// and device, so a process that drives several GPUs configures each of them (one process per GPU is the normal mode).
//     static PerDeviceOnce once;  if (once.need()) { ...configure...; once.mark(); }
struct PerDeviceOnce {
    bool done[64] = {};
    int cur = 0;
    bool need() {
        int d = 0;
        cudaGetDevice(&d);
        cur = d & 63;
        return !done[cur];
    }
    void mark() { done[cur] = true; }
};

// ------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based generator (Salmon et al., SC'11).  Counter layout of this
// library (identical in the fused kernels and in the materialisers):
//   key = (seed_lo, seed_hi)
//   ctr = (quad, row, offset_lo, offset_hi | domain << 30)
// where `quad` indexes 4 consecutive columns of `row`, offset is the per-call counter and
// domain 0 = feature noise, 1 = dropout.
// ------------------------------------------------------------------------------------------
constexpr uint32_t PHILOX_M0 = 0xD2511F53u;
constexpr uint32_t PHILOX_M1 = 0xCD9E8D57u;
constexpr uint32_t PHILOX_W0 = 0x9E3779B9u;
constexpr uint32_t PHILOX_W1 = 0xBB67AE85u;

constexpr uint32_t DOMAIN_NOISE = 0u;
constexpr uint32_t DOMAIN_DROPOUT = 1u;

struct RngKey {
    uint32_t k0, k1;  // seed
    uint32_t c2, c3;  // offset words (domain folded into c3)
};

__host__ __device__ __forceinline__ RngKey make_rng_key(uint64_t seed, uint64_t offset, uint32_t domain) {
    RngKey k;
    k.k0 = (uint32_t)seed;
    k.k1 = (uint32_t)(seed >> 32);
    k.c2 = (uint32_t)offset;
    k.c3 = ((uint32_t)(offset >> 32) & 0x3FFFFFFFu) | (domain << 30);
    return k;
}

// Rounds: 10, as curand's Philox4_32_10 behind the reference's normal_().
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        // one 32x32->64 multiply (IMAD.WIDE.U32) per product instead of a high and a low multiply
        uint32_t hi0, lo0, hi1, lo1;
        asm("{\n\t.reg .b64 t;\n\tmul.wide.u32 t, %2, %3;\n\tmov.b64 {%0, %1}, t;\n\t}" : "=r"(lo0), "=r"(hi0) : "r"(PHILOX_M0), "r"(c0));
        asm("{\n\t.reg .b64 t;\n\tmul.wide.u32 t, %2, %3;\n\tmov.b64 {%0, %1}, t;\n\t}" : "=r"(lo1), "=r"(hi1) : "r"(PHILOX_M1), "r"(c2));
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += PHILOX_W0;
        k1 += PHILOX_W1;
    }
    return make_uint4(c0, c1, c2, c3);
}

// host-side description of a mode-2 stream; resolved to an RngKey inside the kernel so that the
// per-call counter may live in device memory (CUDA-graph replay)
struct RngSpec {
    uint64_t seed;
    uint64_t offset;
    const uint64_t* offset_dev;
};
__device__ __forceinline__ RngKey resolve_rng_key(const RngSpec& s, uint32_t domain) {
    const uint64_t off = (s.offset_dev != nullptr) ? __ldg(s.offset_dev) : s.offset;
    return make_rng_key(s.seed, off, domain);
}

// Box-Muller on two 32-bit words -> two normals of standard deviation `std` (std folded into the radius).
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float std, float& n0, float& n1) {
    // u in (0,1]: (a + 0.5) * 2^-32  (rounds to 1.0f at the very top, never 0), so -2 ln u >= 0
    const float u = fmaf((float)a, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
    // theta in [-pi, pi)
    const float theta = (float)(int32_t)b * 1.4629180792671596e-9f;  // pi * 2^-31
    // u and t are never subnormal (u >= 2^-33; t = 0 or >= 1e-7), so the flush-to-zero forms give the same bits as
    // the default ones and skip their subnormal pre/post-scaling (3 extra instructions per MUFU.LG2 / MUFU.SQRT)
    float lg;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u));
    const float t = __fmul_rn(-1.3862943611198906f, lg);            // -2 ln u = -2 ln2 log2 u
    float rad;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(t));
    rad = __fmul_rn(rad, std);
    float s, c;
    __sincosf(theta, &s, &c);
    n0 = __fmul_rn(rad, c);
    n1 = __fmul_rn(rad, s);
}

// eps for columns 4*quad .. 4*quad+3 of `row`: N(0, std^2).  Every kernel and the materialiser go through this
// one function (explicit round-to-nearest multiplies, no contraction), so they agree bit for bit.
__device__ __forceinline__ float4 noise_quad(const RngKey& key, uint32_t row, uint32_t quad, float std) {
    const uint4 x = philox4x32_10(quad, row, key.c2, key.c3, key.k0, key.k1);
    float n0, n1, n2, n3;
    box_muller(x.x, x.y, std, n0, n1);
    box_muller(x.z, x.w, std, n2, n3);
    return make_float4(n0, n1, n2, n3);
}

// dropout multipliers for columns 4*quad..4*quad+3 of `row`: keep with prob 1-p, scaled 1/(1-p).
__device__ __forceinline__ float4 dropout_quad(const RngKey& key, uint32_t row, uint32_t quad,
                                               float keep_prob, float scale) {
    const uint4 x = philox4x32_10(quad, row, key.c2, key.c3, key.k0, key.k1);
    const float s = 2.3283064365386963e-10f;  // 2^-32
    float4 m;
    m.x = ((float)x.x * s < keep_prob) ? scale : 0.0f;
    m.y = ((float)x.y * s < keep_prob) ? scale : 0.0f;
    m.z = ((float)x.z * s < keep_prob) ? scale : 0.0f;
    m.w = ((float)x.w * s < keep_prob) ? scale : 0.0f;
    return m;
}

// ------------------------------------------------------------------------------------------
// debug timeline: when a buffer is installed (dccf_debug_timeline), thread 0 of every CTA of an instrumented
// kernel records the earliest start / latest end of its kernel in nanoseconds of %globaltimer:
// slot s -> {min start, max end}.  A null pointer (the default) costs one uniform load per CTA.
// ------------------------------------------------------------------------------------------
// (__constant__, not __device__: the pointer is read by thread 0 of EVERY CTA before the CTA's first barrier and again
// before it exits — as a global-memory word it cost a dependent L2 / DRAM round trip at both ends of every kernel of the
// step (ncu: 4-7 % of the stall samples of the training kernels); the constant cache serves it in a few cycles)
static __constant__ unsigned long long* g_timeline = nullptr;
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void tl_begin(int slot) {
    if (threadIdx.x == 0 && g_timeline != nullptr) atomicMin(g_timeline + 2 * slot, global_ns());
}
__device__ __forceinline__ void tl_end(int slot) {
    if (threadIdx.x == 0 && g_timeline != nullptr) atomicMax(g_timeline + 2 * slot + 1, global_ns());
}

// ------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

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

// clamp an id into [0, n) and raise the error flag if it was outside
__device__ __forceinline__ int32_t checked_id(int64_t id, int32_t n, int32_t* err_flag) {
    if (id < 0 || id >= (int64_t)n) {
        if (err_flag) atomicExch(err_flag, 1);
        return 0;
    }
    return (int32_t)id;
}

// item occupying slot z of pair p: slot 0 = the true item, 1..S = sampled confounders
// (src/models/DCCF.py:74)
__device__ __forceinline__ int64_t slot_item(const int64_t* __restrict__ X, const int64_t* __restrict__ sample_item,
                                             int64_t p, int z, int S) {
    return (z == 0) ? X[2 * p + 1] : sample_item[p * S + (z - 1)];
}

}  // namespace dccf
