// Shared helpers for libipdm_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cstring>

#include "../../include/ipdm_b200.h"

namespace ipdm {

// ---- error plumbing: no exceptions cross the C ABI (include/ipdm_b200.h) ----
void set_error(const char* fmt, ...);
const char* last_error();

#define IPDM_CHECK_CUDA(expr)                                                                    \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            ::ipdm::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return IPDM_ERR_CUDA;                                                                \
        }                                                                                        \
    } while (0)

#define IPDM_REQUIRE(cond, ...)                                                                  \
    do {                                                                                         \
        if (!(cond)) {                                                                           \
            ::ipdm::set_error(__VA_ARGS__);                                                      \
            return IPDM_ERR_ARG;                                                                 \
        }                                                                                        \
    } while (0)

#define IPDM_CHECK(expr)                                                                         \
    do {                                                                                         \
        int _rc = (expr);                                                                        \
        if (_rc != IPDM_OK) return _rc;                                                          \
    } while (0)

#define IPDM_CHECK_LAUNCH() IPDM_CHECK_CUDA(cudaGetLastError())

constexpr int kNumSMs = 148;

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// kernel launch counter (bench.py reports it as gpu_launches)
extern unsigned long long g_launch_count;
inline void count_launch(int n = 1) { g_launch_count += (unsigned long long)n; }

// per-kernel-family profiler (off by default): CUDA events around every launch, summed by family.
// cudaFuncSetAttribute applies to the CURRENT device: a launcher remembers per device whether it has configured its kernels
// (one process per GPU is the normal deployment, but a host that drives several devices must not inherit the first one's state).
struct DeviceOnce {
    bool done[64] = {};
    bool need() {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return true;
        if (done[d]) return false;
        done[d] = true;
        return true;
    }
};

enum ProfKind { PROF_CONV_TC = 0, PROF_ATTENTION, PROF_CONV_DIRECT, PROF_GROUPNORM, PROF_UPSAMPLE, PROF_FBP_FILTER,
                PROF_FBP_BACKPROJECT, PROF_SAMPLER, PROF_CONV_HALO_PERS, PROF_KINDS };
extern bool g_prof_on;
void prof_begin(int kind, cudaStream_t st);
void prof_end(int kind, cudaStream_t st, double work, double bytes);
struct ProfScope {
    int kind; cudaStream_t st; double work, bytes;       // bytes: algorithmic HBM bytes of a FLOP-counted launch (ipdm_profile_roofline), else 0
    ProfScope(int k, cudaStream_t s, double w, double b = 0) : kind(k), st(s), work(w), bytes(b) { if (g_prof_on) prof_begin(kind, st); }
    ~ProfScope() { if (g_prof_on) prof_end(kind, st, work, bytes); }
};

// ---- device helpers ----
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- Philox4x32-10 + Box-Muller: 4 N(0,1) draws per 128-bit counter (c0..c3) under the 64-bit key (k0, k1) ----
// Shared by the sampler (sampler.cu: key = seed ^ device-resident epoch) and the low-dose noise (project.cu: key = seed).
__device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
}
__device__ __forceinline__ float4 philox_normal4_keyed(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) { philox_round(c0, c1, c2, c3, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const float s = 2.3283064365386963e-10f;                  // 2^-32
    const float u0 = fmaf((float)c0, s, 0.5f * s), u1 = (float)c1 * s, u2 = fmaf((float)c2, s, 0.5f * s), u3 = (float)c3 * s;
    const float r0 = sqrtf(-2.0f * __logf(u0)), r1 = sqrtf(-2.0f * __logf(u2));
    float s0, co0, s1, co1;
    __sincosf(6.283185307179586f * u1, &s0, &co0);
    __sincosf(6.283185307179586f * u3, &s1, &co1);
    return make_float4(r0 * co0, r0 * s0, r1 * co1, r1 * s1);
}

__device__ __forceinline__ float4 ld_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(float4* p, const float4& v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}


// Round to the nearest TF32 value (10-bit mantissa).  The tensor core only reads the upper 19 bits of an
// fp32 operand, i.e. it TRUNCATES; truncation shrinks every product coherently (measured: 4.3e-4 rel-L2 on a
// K=1152 conv), whereas pre-rounded operands leave only zero-mean noise.  Operand producers call this.
// 2^x in one MUFU instruction (exp2f adds a range fix-up of three more per call); arguments here are <= 0, underflow flushes to 0
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// x * sigmoid(x) with two MUFU operations (ex2, rcp) and no range fix-up: ex2 overflows to +inf for x < -88 (x * rcp(inf) = -0, the limit)
// and flushes to 0 for x > 88 (x / 1 = x); every GroupNorm + SiLU in the library (apply pass, direct conv, fused operand path) uses this one
__device__ __forceinline__ float silu(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + ex2_approx(-1.4426950408889634f * x)));
    return x * r;
}

__device__ __forceinline__ float tanh_approx(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

__device__ __forceinline__ float tf32_rn(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// Same rounding for a value that only the tensor core will read (kind::tf32 ignores the low 13 bits): the add alone, no mask.
// Finite inputs only (activations); +-inf would turn into NaN.
__device__ __forceinline__ float tf32_rn_hw(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }
inline float tf32_rn_host(float x) {
    uint32_t b; memcpy(&b, &x, 4);
    if ((b & 0x7F800000u) == 0x7F800000u) return x;
    b += 0x00000FFFu + ((b >> 13) & 1u);
    b &= 0xFFFFE000u;
    float y; memcpy(&y, &b, 4); return y;
}

}  // namespace ipdm
