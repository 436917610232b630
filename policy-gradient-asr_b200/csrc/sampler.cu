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


// the chain path's sampler of the exploration variant (the public pgasr_softmax_sample keeps theta = 1)
int softmax_sample_theta(const float* logits, const int32_t* in_len, const float* uniforms, uint64_t seed, int B, int T,
                         int V, int K, float theta, uint8_t* samples, float* logp, float* probs, cudaStream_t st) {
    if (!logits || !samples || !logp || B < 0 || T <= 0 || V <= 0 || K <= 0) return PGASR_ERR_INVALID_ARG;
    if (V > kMaxV || K > kSamplerMaxK) return PGASR_ERR_UNSUPPORTED;
    if (B == 0) return PGASR_OK;
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
    if (V > kMaxV || K > kSamplerMaxK) return PGASR_ERR_UNSUPPORTED;
    if (B == 0) return PGASR_OK;
    if (V <= 32)
        softmax_sample_kernel<32><<<B, kSamplerThreads, 0, as_stream(stream)>>>(
            logits, in_len, uniforms, seed, T, V, K, samples, logp, probs);
    else
        softmax_sample_kernel<64><<<B, kSamplerThreads, 0, as_stream(stream)>>>(
            logits, in_len, uniforms, seed, T, V, K, samples, logp, probs);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}
