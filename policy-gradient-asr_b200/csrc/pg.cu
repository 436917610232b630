// K4: rewards, baseline, advantages and the REINFORCE gradient scatter (SURVEY.md 8a row a7; no upstream
// code -- the reward follows metrics.py:24-25 (ED, or ED / len(reference))), and the customNLLLoss slot
// (row a5, upstream loss.py:13-17).
#include "fused_args.cuh"

namespace pgasr {

// one warp per utterance; K <= 64 handled as two lanes-strided passes
__global__ void pg_advantages_kernel(const int32_t* __restrict__ dist, const int32_t* __restrict__ tgt_len,
                                     const float* __restrict__ logp, int B, int K, int Lmax,
                                     int reward_mode, int baseline_mode, float baseline_value,
                                     float* __restrict__ rewards, float* __restrict__ adv,
                                     float* __restrict__ loss_terms) {
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= B) return;
    const int m = tgt_len ? tgt_len[b] : Lmax;
    // rewards are fp32 by contract; baseline, advantage and the loss term in fp64 (A times log p ~ -1000 cancels heavily)
    double sumR = 0.0;
    for (int k = lane; k < K; k += 32) {
        float R = -(float)dist[(size_t)b * K + k];
        if (reward_mode == PGASR_REWARD_NEG_CER) R = __fdiv_rn(R, (float)m);
        rewards[(size_t)b * K + k] = R;
        sumR += (double)R;
    }
    sumR = warp_sum(sumR);
    double term = 0.0;
    for (int k = lane; k < K; k += 32) {
        const float R = rewards[(size_t)b * K + k];
        double base = 0.0;
        if (baseline_mode == PGASR_BASELINE_MEAN) base = sumR / (double)K;
        else if (baseline_mode == PGASR_BASELINE_LOO) base = K > 1 ? (sumR - (double)R) / (double)(K - 1) : 0.0;
        else if (baseline_mode == PGASR_BASELINE_VALUE) base = (double)baseline_value;
        const double Ad = (double)R - base;
        adv[(size_t)b * K + k] = (float)Ad;
        term += -Ad * (double)logp[(size_t)b * K + k];
    }
    term = warp_sum(term);
    if (lane == 0 && loss_terms) loss_terms[b] = (float)term;
}

// one thread per logit: dlogits[b,t,v] (+)= scale * (p * sumA - sum_k A_k [pi_k == v])
__global__ void pg_grad_kernel(const uint8_t* __restrict__ samples, const float* __restrict__ adv,
                               const float* __restrict__ probs, const int32_t* __restrict__ in_len,
                               int B, int T, int V, int K, float scale, int accumulate,
                               float* __restrict__ dlogits) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)B * T * V;
    if (idx >= total) return;
    const int v = (int)(idx % V);
    const size_t bt = idx / V;
    const int t = (int)(bt % T);
    const int b = (int)(bt / T);
    const int Tb = in_len ? min(max(in_len[b], 0), T) : T;
    float g = 0.0f;
    if (t < Tb) {
        float sumA = 0.0f, hit = 0.0f;
        for (int k = 0; k < K; ++k) {
            const float A = __ldg(adv + (size_t)b * K + k);
            sumA += A;
            if (samples[((size_t)b * K + k) * T + t] == v) hit += A;
        }
        g = -hit;
        if (probs) g += probs[idx] * sumA;
        g *= scale;
    }
    dlogits[idx] = accumulate ? dlogits[idx] + g : g;
}

// Exploration variant (DESIGN.md "exploration spec"), one CTA per utterance, one thread per frame: the frame's row of
// p' = softmax(theta z) from the logits, then dlogits[b,t,v] (+)= theta (scale (p' sum_k A_k [dense] - sum_k A_k
// [pi_kt = v]) + (beta / B) p' (log p' + H_t)); H_b = sum_t H_t in a fixed order goes to the entropy output and, times
// beta K / w_pg, out of the utterance's loss term (written by pg_advantages_kernel before this kernel runs).
constexpr int kPgxThreads = 256;
__global__ void __launch_bounds__(kPgxThreads)
pg_grad_explore_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ samples,
                       const float* __restrict__ adv, const int32_t* __restrict__ in_len, int T, int V, int K,
                       float scale, int dense, int accumulate, const ExploreArgs x, float* __restrict__ loss_terms,
                       float* __restrict__ dlogits) {
    __shared__ double ent_w[kPgxThreads / kWarp];
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int Tb = in_len ? min(max(in_len[b], 0), T) : T;
    const float* A = adv + (size_t)b * K;
    float sumA = 0.0f;
    for (int k = 0; k < K; ++k) sumA += __ldg(A + k);
    const bool ent = x.ent_c != 0.0f || x.entropy != nullptr;
    const float th = x.theta, c = __fmul_rn(scale, th), ec = __fmul_rn(x.ent_c, th);
    double hsum = 0.0;
    for (int t = threadIdx.x; t < T; t += kPgxThreads) {
        float* out = dlogits + ((size_t)b * T + t) * V;
        if (t >= Tb) {
            if (!accumulate)
                for (int v = 0; v < V; ++v) out[v] = 0.0f;
            continue;
        }
        const float* z = logits + ((size_t)b * T + t) * V;
        float m = -INFINITY, S = 0.0f;
        for (int v = 0; v < V; ++v) m = fmaxf(m, __fmul_rn(__ldg(z + v), th));
        for (int v = 0; v < V; ++v) S += __expf(__fmul_rn(__ldg(z + v), th) - m);
        const float lz = m + logf(S);
        float H = 0.0f;
        if (ent) {
            for (int v = 0; v < V; ++v) {
                const float lp = __fmul_rn(__ldg(z + v), th) - lz;      // log p' = z' - m' - ln S, never log(p')
                H -= ent_plogp(__expf(lp), lp);
            }
            hsum += (double)H;
        }
        for (int v = 0; v < V; ++v) {
            const float lp = __fmul_rn(__ldg(z + v), th) - lz, p = __expf(lp);
            float hit = 0.0f;
            for (int k = 0; k < K; ++k)
                if (samples[((size_t)b * K + k) * T + t] == v) hit += __ldg(A + k);
            float g = c * ((dense ? p * sumA : 0.0f) - hit);
            if (ent) g += ent_grad(p, ec * (lp + H));
            out[v] = accumulate ? out[v] + g : g;
        }
    }
    hsum = warp_sum(hsum);
    if (lane == 0) ent_w[warp] = hsum;
    __syncthreads();
    if (threadIdx.x == 0 && ent) {
        double Hb = 0.0;
        for (int w = 0; w < kPgxThreads / kWarp; ++w) Hb += ent_w[w];
        if (x.entropy) x.entropy[b] = (float)Hb;
        if (x.ent_lt != 0.0f && loss_terms) loss_terms[b] = (float)((double)loss_terms[b] - (double)x.ent_lt * Hb);
    }
}

int pg_grad_explore(const float* logits, const uint8_t* samples, const float* adv, const int32_t* in_len, int B, int T,
                    int V, int K, float scale, bool dense, int accumulate, const ExploreArgs& x, float* loss_terms,
                    float* dlogits, cudaStream_t st) {
    if (!logits || !samples || !adv || !dlogits || B < 0 || T <= 0 || V <= 0 || K <= 0) return PGASR_ERR_INVALID_ARG;
    if (B == 0) return PGASR_OK;
    pg_grad_explore_kernel<<<B, kPgxThreads, 0, st>>>(logits, samples, adv, in_len, T, V, K, scale, dense ? 1 : 0,
                                                      accumulate, x, loss_terms, dlogits);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

// customNLLLoss.forward (loss.py:13-17): one CTA, deterministic order.  step i: mean over the
// non-ignored batch entries of -inp[i,b,target[b,i]]; the steps are summed.
__global__ void nll_sum_forward_kernel(const float* __restrict__ inp, const int64_t* __restrict__ target,
                                       int L, int B, int V, int ignore_index, float* __restrict__ loss) {
    __shared__ float part[32];
    float acc = 0.0f;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int i = warp; i < L; i += nw) {
        float s = 0.0f, cnt = 0.0f;
        for (int b = lane; b < B; b += 32) {
            const long long c = target[(size_t)b * L + i];
            if (c == (long long)ignore_index) continue;
            // a class id outside [0,V) that is not the ignore value: torch raises there; here the loss turns NaN
            // (loud, and no out-of-bounds read)
            s += (c >= 0 && c < V) ? -inp[((size_t)i * B + b) * V + c] : __int_as_float(0x7fc00000);
            cnt += 1.0f;
        }
        s = warp_sum(s);
        cnt = warp_sum(cnt);
        acc += s / cnt;                                // 0/0 = NaN, as torch's mean over nothing
    }
    if (lane == 0) part[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.0f;
        for (int w = 0; w < nw; ++w) tot += part[w];
        loss[0] = tot;
    }
}

__global__ void nll_sum_backward_kernel(const int64_t* __restrict__ target, const float* __restrict__ grad_out,
                                        int L, int B, int V, int ignore_index, float* __restrict__ grad_inp) {
    // one warp per step i: count the live entries, then write the whole [B,V] slab of the step
    const int i = blockIdx.x;
    const int lane = threadIdx.x & 31;
    __shared__ float s_cnt;
    if (threadIdx.x < 32) {
        float cnt = 0.0f;
        for (int b = lane; b < B; b += 32) {
            const long long c = target[(size_t)b * L + i];
            if (c != (long long)ignore_index) cnt += 1.0f;
        }
        cnt = warp_sum(cnt);
        if (lane == 0) s_cnt = cnt;
    }
    __syncthreads();
    const float w = -grad_out[0] / s_cnt;
    for (int e = threadIdx.x; e < B * V; e += blockDim.x) {
        const int b = e / V, v = e - b * V;
        const long long c = target[(size_t)b * L + i];
        const bool live = c != (long long)ignore_index;
        grad_inp[((size_t)i * B + b) * V + v] = (live && v == c) ? w : 0.0f;
    }
}

}  // namespace pgasr

extern "C" int pgasr_pg_advantages(const int32_t* dist, const int32_t* tgt_len, const float* logp, int B,
                                   int K, int Lmax, int reward_mode, int baseline_mode, float baseline_value,
                                   float* rewards, float* adv, float* loss_terms, void* stream) {
    using namespace pgasr;
    if (!dist || !logp || !rewards || !adv || B < 0 || K <= 0) return PGASR_ERR_INVALID_ARG;
    if (reward_mode < 0 || reward_mode > 1 || baseline_mode < 0 || baseline_mode > 3) return PGASR_ERR_INVALID_ARG;
    if (B == 0) return PGASR_OK;
    const int wpb = 4;
    pg_advantages_kernel<<<(B + wpb - 1) / wpb, wpb * 32, 0, as_stream(stream)>>>(
        dist, tgt_len, logp, B, K, Lmax, reward_mode, baseline_mode, baseline_value, rewards, adv, loss_terms);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

extern "C" int pgasr_pg_grad(const uint8_t* samples, const float* adv, const float* probs,
                             const int32_t* in_len, int B, int T, int V, int K, float scale, int accumulate,
                             float* dlogits, void* stream) {
    using namespace pgasr;
    if (!samples || !adv || !dlogits || B < 0 || T <= 0 || V <= 0 || K <= 0) return PGASR_ERR_INVALID_ARG;
    if (B == 0) return PGASR_OK;
    const size_t total = (size_t)B * T * V;
    const int threads = 256;
    pg_grad_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, as_stream(stream)>>>(
        samples, adv, probs, in_len, B, T, V, K, scale, accumulate, dlogits);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

extern "C" int pgasr_nll_sum_forward(const float* inp, const int64_t* target, int L, int B, int V,
                                     int ignore_index, float* loss, void* stream) {
    using namespace pgasr;
    if (!inp || !target || !loss || L <= 0 || B <= 0 || V <= 0) return PGASR_ERR_INVALID_ARG;
    nll_sum_forward_kernel<<<1, 256, 0, as_stream(stream)>>>(inp, target, L, B, V, ignore_index, loss);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

extern "C" int pgasr_nll_sum_backward(const int64_t* target, const float* grad_out, int L, int B, int V,
                                      int ignore_index, float* grad_inp, void* stream) {
    using namespace pgasr;
    if (!target || !grad_out || !grad_inp || L <= 0 || B <= 0 || V <= 0) return PGASR_ERR_INVALID_ARG;
    nll_sum_backward_kernel<<<L, 256, 0, as_stream(stream)>>>(target, grad_out, L, B, V, ignore_index, grad_inp);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}
