// K1: fused softmax + inverse-CDF categorical sampler (SURVEY.md 8a row a6; no upstream code).
// One CTA per utterance, one thread per frame.  The class is picked by the bit-exact contract in
// DESIGN.md "sampler spec" (same operations as oracle/pgasr_oracle.c:orc_softmax_sample).
#include "fused_args.cuh"

namespace pgasr {

constexpr int kSamplerThreads = 256;
constexpr int kSamplerMaxK = 64;

template <int VP>
__global__ void __launch_bounds__(kSamplerThreads)
softmax_sample_kernel(const float* __restrict__ logits, const int32_t* __restrict__ in_len,
                      const float* __restrict__ uniforms, uint64_t seed, int T, int V, int K,
                      uint8_t* __restrict__ samples, float* __restrict__ logp,
                      float* __restrict__ probs) {
    __shared__ double warp_acc[kSamplerThreads / kWarp][kSamplerMaxK];   // log p ~ -1000: partial sums in fp64
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int Tb = in_len ? in_len[b] : T;
    Tb = min(max(Tb, 0), T);
    for (int i = threadIdx.x; i < (kSamplerThreads / kWarp) * kSamplerMaxK; i += blockDim.x)
        (&warp_acc[0][0])[i] = 0.0;
    __syncthreads();

    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    // every warp walks the same number of iterations so the shuffles below stay converged
    for (int t0 = 0; t0 < T; t0 += blockDim.x) {
        const int t = t0 + threadIdx.x;
        const bool live = t < Tb;
        const float* z = logits + ((size_t)b * T + (live ? t : 0)) * V;
        float cdf[VP];
        float m = -INFINITY, S = 0.0f, logS = 0.0f;
        if (live) {
            float zr[VP];
#pragma unroll
            for (int v = 0; v < VP; ++v) zr[v] = v < V ? __ldg(z + v) : -INFINITY;
#pragma unroll
            for (int v = 0; v < VP; ++v) m = fmaxf(m, zr[v]);
            float c = 0.0f;
#pragma unroll
            for (int v = 0; v < VP; ++v) {
                if (v < V) {
                    float e = exp_spec(__fsub_rn(zr[v], m));
                    c = __fadd_rn(c, e);
                    zr[v] = e;
                }
                cdf[v] = c;
            }
            S = c;
            logS = logf(S);
            if (probs) {
                float inv = 1.0f / S;
                float* pr = probs + ((size_t)b * T + t) * V;
#pragma unroll
                for (int v = 0; v < VP; ++v)
                    if (v < V) pr[v] = zr[v] * inv;
            }
        } else if (t < T && probs) {
            float* pr = probs + ((size_t)b * T + t) * V;
            for (int v = 0; v < V; ++v) pr[v] = 0.0f;
        }
        uint4 rnd = make_uint4(0, 0, 0, 0);
        for (int k = 0; k < K; ++k) {
            float term = 0.0f;
            if (live) {
                float u;
                if (uniforms) {
                    u = __ldg(uniforms + ((size_t)b * K + k) * T + t);
                } else {
                    if ((k & 3) == 0)
                        rnd = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)b, (uint32_t)(k >> 2),
                                                       0x50474153u), key);
                    uint32_t x = (k & 3) == 0 ? rnd.x : (k & 3) == 1 ? rnd.y : (k & 3) == 2 ? rnd.z : rnd.w;
                    u = u32_to_uniform(x);
                }
                const float tau = __fmul_rn(u, S);
                int cnt = 0;
#pragma unroll
                for (int v = 0; v < VP; ++v) cnt += (v < V && cdf[v] <= tau) ? 1 : 0;
                const int pi = min(cnt, V - 1);
                samples[((size_t)b * K + k) * T + t] = (uint8_t)pi;
                term = (__ldg(z + pi) - m) - logS;
            } else if (t < T) {
                samples[((size_t)b * K + k) * T + t] = 0;
            }
            term = warp_sum(term);
            if (lane == 0) warp_acc[warp][k] += (double)term;
        }
    }
    __syncthreads();
    if (threadIdx.x < K) {
        double s = 0.0;
        for (int w = 0; w < kSamplerThreads / kWarp; ++w) s += warp_acc[w][threadIdx.x];
        logp[(size_t)b * K + threadIdx.x] = (float)s;
    }
}

// Exploration variant (DESIGN.md "exploration spec"): the kernel above reading every logit as z' = fl32(z theta), so
// the draws, logp and probs are those of softmax(theta z).  A copy, so that the default kernel stays the kernel it was:
// a shared __forceinline__ body moved its register count (91 -> 89), and a bool template parameter with a theta
// argument renames its symbol and grows its parameter block (968 -> 972 bytes), as the word modes avoided for
// FusedArgs.  Keep the two bodies in step.
template <int VP>
__global__ void __launch_bounds__(kSamplerThreads)
softmax_sample_theta_kernel(const float* __restrict__ logits, const int32_t* __restrict__ in_len,
                            const float* __restrict__ uniforms, uint64_t seed, int T, int V, int K, float theta,
                            uint8_t* __restrict__ samples, float* __restrict__ logp, float* __restrict__ probs) {
    __shared__ double warp_acc[kSamplerThreads / kWarp][kSamplerMaxK];   // log p ~ -1000: partial sums in fp64
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int Tb = in_len ? in_len[b] : T;
    Tb = min(max(Tb, 0), T);
    for (int i = threadIdx.x; i < (kSamplerThreads / kWarp) * kSamplerMaxK; i += blockDim.x)
        (&warp_acc[0][0])[i] = 0.0;
    __syncthreads();

    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    // every warp walks the same number of iterations so the shuffles below stay converged
    for (int t0 = 0; t0 < T; t0 += blockDim.x) {
        const int t = t0 + threadIdx.x;
        const bool live = t < Tb;
        const float* z = logits + ((size_t)b * T + (live ? t : 0)) * V;
        float cdf[VP];
        float m = -INFINITY, S = 0.0f, logS = 0.0f;
        if (live) {
            float zr[VP];
#pragma unroll
            for (int v = 0; v < VP; ++v) zr[v] = v < V ? __fmul_rn(__ldg(z + v), theta) : -INFINITY;
#pragma unroll
            for (int v = 0; v < VP; ++v) m = fmaxf(m, zr[v]);
            float c = 0.0f;
#pragma unroll
            for (int v = 0; v < VP; ++v) {
                if (v < V) {
                    float e = exp_spec(__fsub_rn(zr[v], m));
                    c = __fadd_rn(c, e);
                    zr[v] = e;
                }
                cdf[v] = c;
            }
            S = c;
            logS = logf(S);
            if (probs) {
                float inv = 1.0f / S;
                float* pr = probs + ((size_t)b * T + t) * V;
#pragma unroll
                for (int v = 0; v < VP; ++v)
                    if (v < V) pr[v] = zr[v] * inv;
            }
        } else if (t < T && probs) {
            float* pr = probs + ((size_t)b * T + t) * V;
            for (int v = 0; v < V; ++v) pr[v] = 0.0f;
        }
        uint4 rnd = make_uint4(0, 0, 0, 0);
        for (int k = 0; k < K; ++k) {
            float term = 0.0f;
            if (live) {
                float u;
                if (uniforms) {
                    u = __ldg(uniforms + ((size_t)b * K + k) * T + t);
                } else {
                    if ((k & 3) == 0)
                        rnd = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)b, (uint32_t)(k >> 2),
                                                       0x50474153u), key);
                    uint32_t x = (k & 3) == 0 ? rnd.x : (k & 3) == 1 ? rnd.y : (k & 3) == 2 ? rnd.z : rnd.w;
                    u = u32_to_uniform(x);
                }
                const float tau = __fmul_rn(u, S);
                int cnt = 0;
#pragma unroll
                for (int v = 0; v < VP; ++v) cnt += (v < V && cdf[v] <= tau) ? 1 : 0;
                const int pi = min(cnt, V - 1);
                samples[((size_t)b * K + k) * T + t] = (uint8_t)pi;
                term = (__fmul_rn(__ldg(z + pi), theta) - m) - logS;
            } else if (t < T) {
                samples[((size_t)b * K + k) * T + t] = 0;
            }
            term = warp_sum(term);
            if (lane == 0) warp_acc[warp][k] += (double)term;
        }
    }
    __syncthreads();
    if (threadIdx.x < K) {
        double s = 0.0;
        for (int w = 0; w < kSamplerThreads / kWarp; ++w) s += warp_acc[w][threadIdx.x];
        logp[(size_t)b * K + threadIdx.x] = (float)s;
    }
}

// Wide alphabets (kMaxV < V <= kMaxWideV): the same contract, with the frame's row in shared memory instead of
// registers (a 256-class row and its CDF would spill).  One CTA per utterance walks tiles of kWideFrames frames:
//   1. one warp per row: coalesced loads of the row (4 rows in flight), m = max (exact in any order), the e_v in
//      shared memory (row stride V | 1, odd, so the column walk of step 2 is conflict free);
//   2. one thread per frame: the sequential CDF chain of the spec, in place over the e_v;
//   3. one thread per (frame, group of 4 draws): one Philox call and 4 binary searches over the CDF; the warp sums the
//      log-probability terms of its 32 frames and adds them to a per-(draw, frame block) fp64 slot that only it
//      writes, so logp is summed in one fixed order whatever the schedule;
//   4. probs (when asked for): one warp per row, e_v recomputed from the logits (the chain overwrote them).
constexpr int kWideFrames = 128;
constexpr int kWideBlocks = kWideFrames / kWarp;                 // 32-frame blocks of a tile
constexpr int kWideRows = 4;                                     // rows one warp loads at once in step 1
constexpr int kWideCols = kMaxWideV / kWarp;                     // classes per lane of a row

__host__ __device__ inline int wide_row_stride(int V) { return V | 1; }
static size_t wide_smem_bytes(int V) { return (size_t)kWideFrames * wide_row_stride(V) * sizeof(float); }

template <bool kTheta>
__global__ void __launch_bounds__(kSamplerThreads)
softmax_sample_wide_kernel(const float* __restrict__ logits, const int32_t* __restrict__ in_len,
                           const float* __restrict__ uniforms, uint64_t seed, int T, int V, int K, float theta,
                           uint8_t* __restrict__ samples, float* __restrict__ logp, float* __restrict__ probs) {
    extern __shared__ float cdf_s[];                             // [kWideFrames][RS]: e_v, then cdf[v]
    __shared__ float m_s[kWideFrames], S_s[kWideFrames], logS_s[kWideFrames];
    __shared__ double acc[kSamplerMaxK][kWideBlocks];
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int kWarps = kSamplerThreads / kWarp;
    const int RS = wide_row_stride(V);
    int Tb = in_len ? in_len[b] : T;
    Tb = min(max(Tb, 0), T);
    for (int i = threadIdx.x; i < kSamplerMaxK * kWideBlocks; i += blockDim.x) (&acc[0][0])[i] = 0.0;
    const float* zb = logits + (size_t)b * T * V;
    auto zval = [&](const float* p) { return kTheta ? __fmul_rn(__ldg(p), theta) : __ldg(p); };
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const int G = (K + 3) >> 2;                                  // groups of 4 draws (one Philox call each)

    for (int t0 = 0; t0 < T; t0 += kWideFrames) {
        const int nlive = min(max(Tb - t0, 0), kWideFrames);    // live frames of this tile
        // ---- 1. max and e_v, one warp per row ----------------------------------------------------------
        for (int r0 = warp * kWideRows; r0 < nlive; r0 += kWarps * kWideRows) {
            float z[kWideRows][kWideCols];
#pragma unroll
            for (int i = 0; i < kWideRows; ++i)
#pragma unroll
                for (int j = 0; j < kWideCols; ++j) {
                    const int v = lane + j * kWarp;
                    z[i][j] = (r0 + i < nlive && v < V) ? zval(zb + (size_t)(t0 + r0 + i) * V + v) : -INFINITY;
                }
#pragma unroll
            for (int i = 0; i < kWideRows; ++i) {
                if (r0 + i >= nlive) break;                      // (warp uniform)
                float m = -INFINITY;
#pragma unroll
                for (int j = 0; j < kWideCols; ++j) m = fmaxf(m, z[i][j]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFull, m, o));
                float* row = cdf_s + (size_t)(r0 + i) * RS;
#pragma unroll
                for (int j = 0; j < kWideCols; ++j) {
                    const int v = lane + j * kWarp;
                    if (v < V) row[v] = exp_spec(__fsub_rn(z[i][j], m));
                }
                if (lane == 0) m_s[r0 + i] = m;
            }
        }
        __syncthreads();
        // ---- 2. the sequential CDF chain, one thread per frame -----------------------------------------------
        if (threadIdx.x < nlive) {
            float* row = cdf_s + (size_t)threadIdx.x * RS;
            float c = 0.0f;
#pragma unroll 8
            for (int v = 0; v < V; ++v) {
                c = __fadd_rn(c, row[v]);
                row[v] = c;
            }
            S_s[threadIdx.x] = c;
            logS_s[threadIdx.x] = logf(c);
        }
        __syncthreads();
        // ---- 3. draws: item = (frame f, group g); a warp's 32 items share g and one 32-frame block ----------
        for (int it = threadIdx.x; it < kWideFrames * G; it += blockDim.x) {
            const int f = it % kWideFrames, g = it / kWideFrames;
            const int t = t0 + f;
            const bool live = f < nlive;
            const float* row = cdf_s + (size_t)f * RS;
            const float S = live ? S_s[f] : 0.0f, m = live ? m_s[f] : 0.0f, logS = live ? logS_s[f] : 0.0f;
            uint4 rnd = make_uint4(0, 0, 0, 0);
            if (live && !uniforms)
                rnd = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)b, (uint32_t)g, 0x50474153u), key);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = 4 * g + j;
                if (k >= K) break;                               // (warp uniform)
                float term = 0.0f;
                if (live) {
                    const float u = uniforms ? __ldg(uniforms + ((size_t)b * K + k) * T + t)
                                             : u32_to_uniform(j == 0 ? rnd.x : j == 1 ? rnd.y : j == 2 ? rnd.z : rnd.w);
                    const float tau = __fmul_rn(u, S);
                    // #{v : cdf[v] <= tau} by binary search: every e_v is finite and >= 0 (exp_spec maps NaN and
                    // x < -87 to +0), and adding a value >= 0 under round-to-nearest never decreases a sum, so the
                    // CDF is non-decreasing and the v with cdf[v] <= tau are exactly a prefix [0, cnt): cnt is the
                    // upper-bound index, the same count the register kernels take with V compares.
                    int cnt = 0;
#pragma unroll
                    for (int s = kMaxWideV; s > 0; s >>= 1)
                        if (cnt + s <= V && row[cnt + s - 1] <= tau) cnt += s;
                    const int pi = min(cnt, V - 1);
                    samples[((size_t)b * K + k) * T + t] = (uint8_t)pi;
                    term = (zval(zb + (size_t)t * V + pi) - m) - logS;
                } else if (t < T) {
                    samples[((size_t)b * K + k) * T + t] = 0;
                }
                term = warp_sum(term);
                if (lane == 0) acc[k][f / kWarp] += (double)term;
            }
        }
        // ---- 4. probs = e_v * (1 / S), one warp per row; rows after in_len are zero ---------------------------
        if (probs) {
            const int nrows = min(T - t0, kWideFrames);
            for (int r = warp; r < nrows; r += kWarps) {
                float* pr = probs + ((size_t)b * T + t0 + r) * V;
                if (r >= nlive) {
                    for (int v = lane; v < V; v += kWarp) pr[v] = 0.0f;
                    continue;
                }
                const float m = m_s[r], inv = 1.0f / S_s[r];
                const float* z = zb + (size_t)(t0 + r) * V;
                for (int v = lane; v < V; v += kWarp) pr[v] = exp_spec(__fsub_rn(zval(z + v), m)) * inv;
            }
        }
        __syncthreads();                                         // the next tile overwrites the rows
    }
    if (threadIdx.x < K) {
        double s = 0.0;
        for (int i = 0; i < kWideBlocks; ++i) s += acc[threadIdx.x][i];
        logp[(size_t)b * K + threadIdx.x] = (float)s;
    }
}

template <bool kTheta>
static int launch_sample_wide(const float* logits, const int32_t* in_len, const float* uniforms, uint64_t seed, int B,
                              int T, int V, int K, float theta, uint8_t* samples, float* logp, float* probs,
                              cudaStream_t st) {
    const size_t smem = wide_smem_bytes(V);
    if (smem > 48 * 1024)
        PGASR_CUDA_TRY(cudaFuncSetAttribute(softmax_sample_wide_kernel<kTheta>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    softmax_sample_wide_kernel<kTheta><<<B, kSamplerThreads, smem, st>>>(logits, in_len, uniforms, seed, T, V, K, theta,
                                                                         samples, logp, probs);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

// the chain path's sampler of the exploration variant (the public pgasr_softmax_sample keeps theta = 1)
int softmax_sample_theta(const float* logits, const int32_t* in_len, const float* uniforms, uint64_t seed, int B, int T,
                         int V, int K, float theta, uint8_t* samples, float* logp, float* probs, cudaStream_t st) {
    if (!logits || !samples || !logp || B < 0 || T <= 0 || V <= 0 || K <= 0) return PGASR_ERR_INVALID_ARG;
    if (V > kMaxWideV || K > kSamplerMaxK) return PGASR_ERR_UNSUPPORTED;
    if (B == 0) return PGASR_OK;
    if (V > kMaxV)
        return launch_sample_wide<true>(logits, in_len, uniforms, seed, B, T, V, K, theta, samples, logp, probs, st);
    if (V <= 32)
        softmax_sample_theta_kernel<32><<<B, kSamplerThreads, 0, st>>>(logits, in_len, uniforms, seed, T, V, K, theta,
                                                                      samples, logp, probs);
    else
        softmax_sample_theta_kernel<64><<<B, kSamplerThreads, 0, st>>>(logits, in_len, uniforms, seed, T, V, K, theta,
                                                                      samples, logp, probs);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

}  // namespace pgasr

extern "C" int pgasr_softmax_sample(const float* logits, const int32_t* in_len, const float* uniforms,
                                    uint64_t seed, int B, int T, int V, int K, uint8_t* samples,
                                    float* logp, float* probs, void* stream) {
    using namespace pgasr;
    if (!logits || !samples || !logp || B < 0 || T <= 0 || V <= 0 || K <= 0) return PGASR_ERR_INVALID_ARG;
    if (V > kMaxWideV || K > kSamplerMaxK) return PGASR_ERR_UNSUPPORTED;
    if (B == 0) return PGASR_OK;
    if (V > kMaxV)
        return launch_sample_wide<false>(logits, in_len, uniforms, seed, B, T, V, K, 1.0f, samples, logp, probs,
                                         as_stream(stream));
    if (V <= 32)
        softmax_sample_kernel<32><<<B, kSamplerThreads, 0, as_stream(stream)>>>(
            logits, in_len, uniforms, seed, T, V, K, samples, logp, probs);
    else
        softmax_sample_kernel<64><<<B, kSamplerThreads, 0, as_stream(stream)>>>(
            logits, in_len, uniforms, seed, T, V, K, samples, logp, probs);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}
