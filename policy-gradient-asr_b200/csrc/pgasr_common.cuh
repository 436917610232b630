// Shared device/host helpers for libpgasr_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "pgasr.h"

namespace pgasr {

extern thread_local int g_last_cuda_error;
extern thread_local unsigned long long g_launches;   // kernels launched by this thread (bench.py's gpu_launches)

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return PGASR_ERR_CUDA;
}

#define PGASR_CUDA_TRY(expr)                                   \
    do {                                                       \
        cudaError_t _e = (expr);                               \
        if (_e != cudaSuccess) return ::pgasr::cuda_fail(_e);  \
    } while (0)

#define PGASR_LAUNCH_CHECK()                \
    do {                                    \
        ++::pgasr::g_launches;              \
        PGASR_CUDA_TRY(cudaGetLastError()); \
    } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Optional phase timing (build with -DPGASR_TIMING; tools/phase_timing.py): clock64 stamps of CTA ticket 0.
#ifdef PGASR_TIMING
static __device__ long long g_dbg[64];   // one copy per translation unit; fused_spl8.cu's is the one read back
#define PGASR_STAMP(cond, slot) do { if (cond) ::pgasr::g_dbg[slot] = clock64(); } while (0)
#define PGASR_ACCUM(cond, slot, v) do { if (cond) ::pgasr::g_dbg[slot] += (v); } while (0)
#else
#define PGASR_STAMP(cond, slot) do { } while (0)
#define PGASR_ACCUM(cond, slot, v) do { } while (0)
#endif

constexpr int kMaxV = 64;         // classes the fused step and the host pipeline take (fast paths: V <= 32)
constexpr int kMaxWideV = 256;    // classes the sampler, the step (chain of stand-alone kernels above kMaxV) and the
                                  // beam search take: the uint8 sample format's limit
constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---------------------------------------------------------------------------------------------
// Sampler contract (DESIGN.md "sampler spec"): every operation is one fp32 operation rounded to
// nearest even; __f*_rn intrinsics are never contracted into FMAs by nvcc.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float exp_spec(float x0) {
    // branch free (an early return made every call its own basic block: neighbouring calls could not interleave):
    // the polynomial runs on max(x, -87), the spec's "x < -87 -> +0" (and NaN -> +0) is a select at the end
    const float x = fmaxf(x0, -87.0f);
    float t = __fmul_rn(x, 1.44269504088896341f);
    float n = rintf(t);
    float r = __fsub_rn(x, __fmul_rn(n, 0.693359375f));
    r = __fsub_rn(r, __fmul_rn(n, -2.12194440e-4f));
    float p = 1.9875691500e-4f;
    p = __fadd_rn(__fmul_rn(p, r), 1.3981999507e-3f);
    p = __fadd_rn(__fmul_rn(p, r), 8.3334519073e-3f);
    p = __fadd_rn(__fmul_rn(p, r), 4.1665795894e-2f);
    p = __fadd_rn(__fmul_rn(p, r), 1.6666665459e-1f);
    p = __fadd_rn(__fmul_rn(p, r), 5.0000001201e-1f);
    float r2 = __fmul_rn(r, r);
    float y = __fmul_rn(p, r2);
    y = __fadd_rn(y, r);
    y = __fadd_rn(y, 1.0f);
    int ni = (int)n;
    float scale = __int_as_float((ni + 127) << 23);
    // (a multiplication by 1 or 0, not a select: the compiler turns "cond ? value : 0" back into a branch around the
    // whole polynomial; y * scale is finite and >= 0, so the product is exact: the value itself or +0)
    return __fmul_rn(__fmul_rn(y, scale), x0 >= -87.0f ? 1.0f : 0.0f);
}

// Philox4x32-10 (Salmon et al. 2011).  Counter (t, b, k/4, 'PGAS'), key = seed.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ float u32_to_uniform(uint32_t x) {
    return __fmul_rn((float)(x >> 8), 5.9604644775390625e-08f);   // top 24 bits, exact
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

}  // namespace pgasr
