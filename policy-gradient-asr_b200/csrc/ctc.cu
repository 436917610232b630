// K5: CTC alpha-beta loss and gradient (SURVEY.md 8a row a8; no upstream code; spec = DESIGN.md "CTC spec").
//
// Design (B200): one CTA per utterance.  Warp 0 runs the alpha recurrence forward in time, warp 1 runs beta
// backward, at the same time, and they meet in the middle: each stores the half of its lattice the other one
// needs (pre-emission sums, fp64, [frame][j][lane] so every store/load is a coalesced 256 B line), one
// __syncthreads, then each warp finishes its pass and emits the gradient rows of the frames it now owns.
// The serial depth is T frame steps instead of 2T, and only the 1-2 halo values cross lanes per frame
// (warp shuffles; every lane owns SPL consecutive label states in registers).
//
// Arithmetic: the lattice is kept in LINEAR space in fp64 with exact power-of-two rescaling (the exponent is
// read off the warp maximum with one redux.sync every 4 frames).  Measured on B200 (tools/pipe_probe.cu): the
// fp64 pipe sustains 17.3 T fma/s against 4.6 T ex2/s on the MUFU pipe, latency 8.5 vs ~40 cycles, and a
// log-space recurrence needs 3 ex2 + 1 lg2 per state per frame and loses ~1e-4 relative in fp32 at
// |log alpha| ~ 1e3.  The frame loop is branch free: illegal two-state transitions are a multiply by 0.0,
// label states beyond the transcript read a zero slot of the probability row.
//
// Gradient: occupancies gamma_t(s) = alpha_t(s) beta'_t(s) / P.  P is measured once, at the first frame of a
// warp's second half (Z0 = sum_s alpha beta'); later frames reuse it through the recorded power-of-two exponents,
// so no per-frame reduction over states is needed.  gamma is converted to 2^-30 fixed point by one fma with the
// 2^52+2^51 magic constant, the blank column is summed with one integer redux.sync, label columns with integer
// shared-memory atomics (exact, order independent => deterministic).
#include "ctc_core.cuh"
#include "fused_args.cuh"

namespace pgasr {

constexpr int kCtcThreads = 128;  // warp 0: alpha, warp 1: beta, all four: softmax rows

// One utterance; kChunk frames per staged batch of each walking warp (kCtcChunk, or kCtcChunkWide for rows too wide
// for it).  The two kernels below are this body with either depth.
template <int SPL, bool kAccum, int kChunk>
__device__ __forceinline__ void
ctc_utterance(const float* __restrict__ logits, const float* __restrict__ probs_in,
              double* __restrict__ probs_ws, const int32_t* __restrict__ targets,
              const int32_t* __restrict__ in_len, const int32_t* __restrict__ tgt_len, int T, int V,
              int Lmax, int blank, float grad_scale, float* __restrict__ nll,
              float* __restrict__ dlogits, double* __restrict__ lattice, int* __restrict__ lat_exp) {
    extern __shared__ double smem_d[];
    const int b = blockIdx.x;
    const int warp = threadIdx.x >> 5;
    const int RS = ctc_row_stride(V);
    int Tb = in_len ? in_len[b] : T;
    Tb = min(max(Tb, 0), T);
    int L = tgt_len ? tgt_len[b] : Lmax;
    L = min(max(L, 0), Lmax);
    float* dlog_u = dlogits + (size_t)b * T * V;
    if (!kAccum)                                          // rows beyond the utterance carry no gradient
        for (int i = Tb * V + threadIdx.x; i < T * V; i += blockDim.x) dlog_u[i] = 0.0f;
    if (Tb == 0) {
        if (threadIdx.x == 0) nll[b] = L == 0 ? 0.0f : INFINITY;
        return;
    }
    double* pw = probs_ws + (size_t)b * T * RS;
    for (int t = threadIdx.x; t < Tb; t += blockDim.x)
        softmax_row_f64(logits ? logits + ((size_t)b * T + t) * V : nullptr,
                        probs_in ? probs_in + ((size_t)b * T + t) * V : nullptr, pw + (size_t)t * RS, V, RS);
    __syncthreads();
    auto mid = [] { __syncthreads(); };
    if (warp >= 2) {                                      // only two warps walk the lattice
        mid();
        return;
    }
    double* stage = smem_d + (size_t)warp * (2 * kChunk * RS);
    int* racc = reinterpret_cast<int*>(smem_d + (size_t)2 * (2 * kChunk * RS)) + warp * (V + 2);
    double* lat_u = lattice + (size_t)b * T * (SPL * 32);
    int* exp_u = lat_exp + (size_t)b * T;
    const int32_t* lab_u = targets + (size_t)b * Lmax;
    if (warp == 0)
        ctc_direction<SPL, true, kAccum, false, kChunk>(pw, lab_u, Tb, L, V, RS, blank, grad_scale, nll + b, dlog_u,
                                                        lat_u, exp_u, stage, racc, mid);
    else
        ctc_direction<SPL, false, kAccum, false, kChunk>(pw, lab_u, Tb, L, V, RS, blank, grad_scale, nll + b, dlog_u,
                                                         lat_u, exp_u, stage, racc, mid);
}

#define PGASR_CTC_KERNEL(name, chunk)                                                                                 \
    template <int SPL, bool kAccum>                                                                                   \
    __global__ void __launch_bounds__(kCtcThreads)                                                                    \
    name(const float* __restrict__ logits, const float* __restrict__ probs_in, double* __restrict__ probs_ws,         \
         const int32_t* __restrict__ targets, const int32_t* __restrict__ in_len, const int32_t* __restrict__ tgt_len, \
         int T, int V, int Lmax, int blank, float grad_scale, float* __restrict__ nll, float* __restrict__ dlogits,   \
         double* __restrict__ lattice, int* __restrict__ lat_exp) {                                                   \
        ctc_utterance<SPL, kAccum, chunk>(logits, probs_in, probs_ws, targets, in_len, tgt_len, T, V, Lmax, blank,    \
                                          grad_scale, nll, dlogits, lattice, lat_exp);                                \
    }
PGASR_CTC_KERNEL(ctc_kernel, kCtcChunk)           // V <= 196: 32 frames per batch
PGASR_CTC_KERNEL(ctc_wide_kernel, kCtcChunkWide)  // 196 < V <= 256: 16 frames per batch
#undef PGASR_CTC_KERNEL

// dynamic shared memory of the classic kernel: two warps x two staged batches of kChunk rows, and the two warps'
// label-column accumulators
static size_t ctc_smem_bytes(int V, int chunk) {
    return (size_t)2 * (2 * chunk * ctc_row_stride(V)) * sizeof(double) + (size_t)2 * (V + 2) * sizeof(int);
}
constexpr size_t kCtcMaxSmem = 200 * 1024;

struct CtcWs { size_t lat, probs, exps, total; };
static CtcWs ctc_ws(int B, int T, int V, int spl) {
    CtcWs w;
    w.lat = align_up((size_t)B * T * spl * 32 * sizeof(double), 256);
    w.probs = align_up((size_t)B * T * ctc_row_stride(V) * sizeof(double), 256);
    w.exps = align_up((size_t)B * T * sizeof(int), 256);
    w.total = w.lat + w.probs + w.exps;
    return w;
}

template <int SPL>
static int launch_ctc(const float* logits, const float* probs, const int32_t* targets, const int32_t* in_len,
                      const int32_t* tgt_len, int B, int T, int V, int Lmax, int blank, float grad_scale,
                      int accumulate, float* nll, float* dlogits, char* base, const CtcWs& w, cudaStream_t st) {
    double* lattice = reinterpret_cast<double*>(base);
    double* probs_ws = reinterpret_cast<double*>(base + w.lat);
    int* lat_exp = reinterpret_cast<int*>(base + w.lat + w.probs);
    // 32 staged frames per batch while they fit (every V <= 196), else 16
    const bool wide = ctc_smem_bytes(V, kCtcChunk) > kCtcMaxSmem;
    const size_t smem = ctc_smem_bytes(V, wide ? kCtcChunkWide : kCtcChunk);
    if (smem > kCtcMaxSmem) return PGASR_ERR_UNSUPPORTED;
    using Kern = void (*)(const float*, const float*, double*, const int32_t*, const int32_t*, const int32_t*, int, int,
                          int, int, float, float*, float*, double*, int*);
    const Kern k = wide ? (accumulate ? ctc_wide_kernel<SPL, true> : ctc_wide_kernel<SPL, false>)
                        : (accumulate ? ctc_kernel<SPL, true> : ctc_kernel<SPL, false>);
    if (smem > 48 * 1024) PGASR_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<B, kCtcThreads, smem, st>>>(logits, probs, probs_ws, targets, in_len, tgt_len, T, V, Lmax, blank, grad_scale,
                                    nll, dlogits, lattice, lat_exp);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

}  // namespace pgasr

// one call runs either the single-launch kernel (CTC role only; its workspace + 256 B for its loss scalar) or the
// classic kernel: the two layouts share the buffer
extern "C" size_t pgasr_ctc_workspace_bytes(int B, int T, int V, int Lmax) {
    using namespace pgasr;
    const int spl = ctc_spl(Lmax);
    if (spl == 0 || B < 0 || T <= 0 || V <= 0) return 0;
    const size_t fused = (fused_capability(T, V, 1, Lmax) & 1) ? align256(fused_workspace_bytes(B, T, V, 1, Lmax)) + 256 : 0;
    const size_t classic = ctc_ws(B, T, V, spl).total;
    return fused > classic ? fused : classic;
}

extern "C" int pgasr_ctc_loss_grad(const float* logits, const float* probs, const int32_t* targets,
                                   const int32_t* in_len, const int32_t* tgt_len, int B, int T, int V,
                                   int Lmax, int blank, float grad_scale, int accumulate, float* nll,
                                   float* dlogits, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace pgasr;
    if ((!logits && !probs) || !targets || !nll || !dlogits || !workspace || B < 0 || T <= 0 || V <= 0 ||
        Lmax <= 0 || blank < 0 || blank >= V)
        return PGASR_ERR_INVALID_ARG;
    const int spl = ctc_spl(Lmax);
    if (spl == 0) return PGASR_ERR_UNSUPPORTED;
    const CtcWs w = ctc_ws(B, T, V, spl);
    if (workspace_bytes < pgasr_ctc_workspace_bytes(B, T, V, Lmax)) return PGASR_ERR_WORKSPACE;
    if (B == 0) return PGASR_OK;
    cudaStream_t st = as_stream(stream);
    const bool fusable = logits && (fused_capability(T, V, 1, Lmax) & 1) && B + 4 <= 16384;
    const size_t fused_bytes = (fused_capability(T, V, 1, Lmax) & 1) ? align256(fused_workspace_bytes(B, T, V, 1, Lmax)) + 256 : 0;
    if (fusable && !accumulate) {
        // the walker / gradient-worker kernel of the fused step, CTC role only (3x the classic kernel at T = 500);
        // it takes the softmax from the logits itself (`probs` is only a shortcut for the classic kernel)
        FusedArgs a;
        a.logits = logits; a.targets = targets; a.in_len = in_len; a.tgt_len = tgt_len; a.uniforms = nullptr;
        a.seed = 0; a.B = B; a.T = T; a.V = V; a.K = 1; a.Lmax = Lmax; a.blank = blank;
        a.reward_mode = 0; a.baseline_mode = 1; a.baseline_value = 0.0f;
        a.w_pg = 0.0f; a.w_ctc = grad_scale * (float)B;   // the kernel scales the rows by w_ctc / B
        a.do_pg = 0; a.do_ctc = 1;
        a.loss = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + fused_bytes - 256);
        a.dlogits = dlogits; a.rewards = nullptr; a.logp = nullptr; a.hyp_len = nullptr; a.dist = nullptr;
        a.nll = nll; a.samples = nullptr; a.to_go = nullptr; a.r_pos = nullptr;
        PGASR_CUDA_TRY(cudaMemsetAsync(workspace, 0, (size_t)2 * (4 + B) * sizeof(unsigned), st));   // arm both control blocks
        return fused_step(a, workspace, st);
    }
    char* base = reinterpret_cast<char*>(workspace);
    switch (spl) {
        case 4: return launch_ctc<4>(logits, probs, targets, in_len, tgt_len, B, T, V, Lmax, blank, grad_scale, accumulate, nll, dlogits, base, w, st);
        case 8: return launch_ctc<8>(logits, probs, targets, in_len, tgt_len, B, T, V, Lmax, blank, grad_scale, accumulate, nll, dlogits, base, w, st);
        case 16: return launch_ctc<16>(logits, probs, targets, in_len, tgt_len, B, T, V, Lmax, blank, grad_scale, accumulate, nll, dlogits, base, w, st);
        default: return launch_ctc<32>(logits, probs, targets, in_len, tgt_len, B, T, V, Lmax, blank, grad_scale, accumulate, nll, dlogits, base, w, st);
    }
}
