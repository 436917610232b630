// The whole loss step behind one C-ABI call (upstream call site: criterion(model_out, t) followed by
// loss.backward(), model.py:235-237), plus the small ABI utilities.
#include <cmath>
#include <cstdlib>

#include "fused_args.cuh"
#include "words_core.cuh"

namespace pgasr {



thread_local int g_last_cuda_error = 0;
thread_local unsigned long long g_launches = 0;

size_t align256(size_t x) { return (x + 255) / 256 * 256; }

struct StepWorkspace {
    uint8_t* samples; uint8_t* hyps;
    int32_t* hyp_len; int32_t* dist;
    float* logp; float* rewards; float* adv; float* loss_terms; float* nll; float* probs;
    void* ctc; size_t ctc_bytes; size_t total;
};

// The one predicate carve(), pgasr_pg_ctc_step_workspace_bytes and the step share: the single-launch kernel takes
// the shape AND the batch fits its control block (4 + B words per block, two blocks inside the 128 KB that
// pgasr_pg_ctc_step_workspace_init clears).  Larger batches chain the stand-alone kernels.
constexpr int kFusedMaxB = 16380;
static int step_fused_capability(int B, int T, int V, int K, int Lmax) {
    return B <= kFusedMaxB ? fused_capability(T, V, K, Lmax) : 0;
}

static StepWorkspace carve(void* base, int B, int T, int V, int K, int Lmax) {
    StepWorkspace w;
    char* p = reinterpret_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { char* r = p ? p + off : nullptr; off += align256(bytes); return r; };
    const size_t BK = (size_t)B * K;
    w.samples = reinterpret_cast<uint8_t*>(take(BK * T));
    w.hyps = reinterpret_cast<uint8_t*>(take(BK * T));
    w.hyp_len = reinterpret_cast<int32_t*>(take(BK * 4));
    w.dist = reinterpret_cast<int32_t*>(take(BK * 4));
    w.logp = reinterpret_cast<float*>(take(BK * 4));
    w.rewards = reinterpret_cast<float*>(take(BK * 4));
    w.adv = reinterpret_cast<float*>(take(BK * 4));
    w.loss_terms = reinterpret_cast<float*>(take((size_t)B * 4));
    w.nll = reinterpret_cast<float*>(take((size_t)B * 4));
    w.probs = reinterpret_cast<float*>(take((size_t)B * T * V * 4));
    // the classic CTC kernel is only chained when the single-launch kernel cannot take the shape
    w.ctc_bytes = (step_fused_capability(B, T, V, K, Lmax) & 1) ? 256 : pgasr_ctc_workspace_bytes(B, T, V, Lmax);
    w.ctc = take(w.ctc_bytes);
    w.total = off;
    return w;
}

// loss = w_pg / (B K) * sum_b loss_terms[b] + w_ctc / B * sum_b nll[b]; one warp, fixed order.
__global__ void finalize_loss_kernel(const float* __restrict__ loss_terms, const float* __restrict__ nll,
                                     int B, int K, float w_pg, float w_ctc, float* __restrict__ loss) {
    float a = 0.0f, c = 0.0f;
    for (int b = threadIdx.x; b < B; b += 32) {
        if (loss_terms) a += loss_terms[b];
        if (nll) c += nll[b];
    }
    a = warp_sum(a);
    c = warp_sum(c);
    if (threadIdx.x == 0) {
        float l = 0.0f;
        if (loss_terms) l += w_pg * a / ((float)B * (float)K);
        if (nll) l += w_ctc * c / (float)B;
        loss[0] = l;
    }
}

}  // namespace pgasr

extern "C" int pgasr_abi_version(void) { return PGASR_ABI_VERSION; }

extern "C" const char* pgasr_status_string(int status) {
    switch (status) {
        case PGASR_OK: return "ok";
        case PGASR_ERR_INVALID_ARG: return "invalid argument";
        case PGASR_ERR_UNSUPPORTED: return "unsupported size for this build";
        case PGASR_ERR_NO_DEVICE: return "no sm_100 CUDA device";
        case PGASR_ERR_WORKSPACE: return "workspace too small";
        case PGASR_ERR_CUDA: return "CUDA error (see pgasr_last_cuda_error)";
        default: return "unknown status";
    }
}

extern "C" int pgasr_last_cuda_error(void) { return pgasr::g_last_cuda_error; }

extern "C" uint64_t pgasr_launch_count(void) { return pgasr::g_launches; }



extern "C" int pgasr_device_check(void) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return PGASR_ERR_NO_DEVICE;
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
        return PGASR_ERR_NO_DEVICE;
    return major == 10 ? PGASR_OK : PGASR_ERR_NO_DEVICE;
}

// layout of ONE lane: [fused-kernel workspace (control block first)][scratch of the stand-alone kernels]; the workspace
// holds three lanes (pgasr_pg_ctc_step_multi runs consecutive steps on three streams, each with its own lane)
namespace pgasr {
static size_t step_lane_bytes(int B, int T, int V, int K, int Lmax) {
    if (B < 0 || T <= 0 || V <= 0 || K <= 0 || Lmax <= 0) return 0;
    const size_t fused = step_fused_capability(B, T, V, K, Lmax) ? align256(fused_workspace_bytes(B, T, V, K, Lmax)) : 0;
    const StepWorkspace w = carve(nullptr, B, T, V, K, Lmax);
    if (w.ctc_bytes == 0) return 0;
    return align256(fused + w.total);
}
}  // namespace pgasr

namespace pgasr {
constexpr int kMaxLanes = 4;
// lanes of the workspace = steps of one pgasr_pg_ctc_step_multi call in flight at once (3: long runs measure the same
// with 2, 3 or 4, a 20-step region is 3 % shorter with 3 than with 2 -- the drain is smoother; PGASR_LANES=1..4 for A/B runs)
static int step_lanes() {
    static const int n = [] {
        const char* e = getenv("PGASR_LANES");
        const int v = e ? atoi(e) : 3;
        return v < 1 ? 1 : v > kMaxLanes ? kMaxLanes : v;
    }();
    return n;
}
}  // namespace pgasr

extern "C" size_t pgasr_pg_ctc_step_workspace_bytes(int B, int T, int V, int K, int Lmax) {
    return (size_t)pgasr::step_lanes() * pgasr::step_lane_bytes(B, T, V, K, Lmax);
}

extern "C" int pgasr_pg_ctc_step_workspace_init(void* workspace, size_t workspace_bytes, void* stream) {
    if (!workspace) return PGASR_ERR_INVALID_ARG;
    // The control blocks of a fused workspace have to start at zero; the kernel re-arms its block after every step.
    // The first lane's blocks sit at the front (2 * (4 + kFusedMaxB) words = 128 KB at most) and are cleared here; any
    // other fused workspace inside the range (the second lane, whose offset depends on the shape) is cleared on the
    // launching stream the first time a step uses it -- which it will be again after this call, because the host-side
    // records of every workspace in the range are dropped here (a recycled pointer therefore starts afresh).
    const size_t ctrl = (size_t)2 * (4 + pgasr::kFusedMaxB) * sizeof(unsigned);
    const size_t n = workspace_bytes < ctrl ? workspace_bytes : ctrl;
    PGASR_CUDA_TRY(cudaMemsetAsync(workspace, 0, n, pgasr::as_stream(stream)));
    pgasr::fused_workspace_reset(workspace, workspace_bytes);
    return PGASR_OK;
}

namespace pgasr {

struct StepParams {
    int B, T, V, K, Lmax, blank, reward_mode, baseline_mode;
    float baseline_value, w_pg, w_ctc;
    int word_sep;            // -1: entry points without word modes (reward_mode <= PGASR_REWARD_MAX)
    float temperature = 1.0f, w_ent = 0.0f;   // exploration (pgasr_pg_ctc_step_multi_ex)
};

static bool word_mode(int reward_mode) {
    return reward_mode == PGASR_REWARD_NEG_WED || reward_mode == PGASR_REWARD_NEG_WER;
}

static int step_check(const StepParams& q, const void* workspace, size_t workspace_bytes) {
    if (!workspace || q.B <= 0 || q.T <= 0 || q.V <= 0 || q.K <= 0 || q.Lmax <= 0 || q.blank < 0 || q.blank >= q.V)
        return PGASR_ERR_INVALID_ARG;
    const bool words = q.word_sep >= 0 && q.word_sep < q.V && q.word_sep != q.blank;
    if (q.word_sep != -1 && !words) return PGASR_ERR_INVALID_ARG;   // (pgasr_pg_ctc_step_multi_ws: the separator)
    if (q.reward_mode < 0 || (q.reward_mode > PGASR_REWARD_MAX && !(words && word_mode(q.reward_mode))) ||
        q.baseline_mode < 0 || q.baseline_mode > 3)
        return PGASR_ERR_INVALID_ARG;
    if (q.K > 64 || q.V > kMaxV) return PGASR_ERR_UNSUPPORTED;
    const size_t need = pgasr_pg_ctc_step_workspace_bytes(q.B, q.T, q.V, q.K, q.Lmax);
    if (need == 0) return PGASR_ERR_UNSUPPORTED;
    if (workspace_bytes < need) return PGASR_ERR_WORKSPACE;
    if ((reinterpret_cast<uintptr_t>(workspace) & 255u) != 0) return PGASR_ERR_INVALID_ARG;
    return PGASR_OK;
}

// one step: one launch of the single-launch kernel when the shape fits, else the chain of stand-alone kernels
// entropy: the step's H_b output (pgasr_pg_ctc_step_multi_ex), or NULL
static int step_one(const StepParams& q, const pgasr_step_io& io, uint64_t seed, void* workspace, cudaStream_t st,
                    bool throughput = false, float* entropy = nullptr) {
    if (!io.logits || !io.targets || !io.loss || !io.dlogits) return PGASR_ERR_INVALID_ARG;
    void* stream = reinterpret_cast<void*>(st);
    const int B = q.B, T = q.T, V = q.V, K = q.K, Lmax = q.Lmax;
    const bool do_pg = q.w_pg != 0.0f, do_ctc = q.w_ctc != 0.0f;
    const int cap = step_fused_capability(B, T, V, K, Lmax);
    const bool words = word_mode(q.reward_mode);
    // word modes: the single-launch kernel when its word layout fits, else the PG part chains the stand-alone kernels
    const bool words_fused = words && do_pg && fused_word_capability(T, V, K, Lmax);
    const WordArgs wa = {q.word_sep, word_class_cap(Lmax, V)};
    // exploration variant only when it changes something: defaults launch the kernels they always launched
    const bool explore = do_pg && (q.temperature != 1.0f || q.w_ent != 0.0f || entropy);
    ExploreArgs x;
    x.theta = 1.0f / q.temperature;                        // theta = fl32(1 / tau)
    x.ent_c = q.w_ent / (float)B;
    x.ent_lt = q.w_ent != 0.0f ? q.w_ent * (float)K / q.w_pg : 0.0f;
    x.entropy = entropy;
    FusedArgs a;
    a.logits = io.logits; a.targets = io.targets; a.in_len = io.in_len; a.tgt_len = io.tgt_len; a.uniforms = io.uniforms;
    a.seed = seed; a.B = B; a.T = T; a.V = V; a.K = K; a.Lmax = Lmax; a.blank = q.blank;
    a.reward_mode = q.reward_mode; a.baseline_mode = q.baseline_mode; a.baseline_value = q.baseline_value;
    a.w_pg = q.w_pg; a.w_ctc = q.w_ctc; a.do_pg = do_pg; a.do_ctc = do_ctc;
    a.loss = io.loss; a.dlogits = io.dlogits; a.rewards = io.rewards; a.logp = io.logp; a.hyp_len = io.hyp_len;
    a.dist = io.dist; a.nll = io.nll; a.samples = io.samples; a.to_go = io.to_go; a.r_pos = io.r_pos;
    if ((do_pg || do_ctc) && (cap & 1) && (!do_pg || (cap & 2)) && (!words || !do_pg || words_fused)) {
        // one launch: heterogeneous CTAs (CTC role / PG role per utterance), see fused.cu
        return fused_step(a, workspace, st, throughput, words && do_pg ? &wa : nullptr, explore ? &x : nullptr);
    }
    if (do_pg && q.reward_mode == PGASR_REWARD_ED_TO_GO) return PGASR_ERR_UNSUPPORTED;   // (single-launch kernel only)
    // long utterances: the PG role's tiles do not fit one SM -- the PG part runs as the chain of stand-alone
    // kernels, the CTC part still as the single-launch kernel (tile streamed from the workspace) when it fits
    const size_t fused_bytes = cap ? align256(fused_workspace_bytes(B, T, V, K, Lmax)) : 0;
    StepWorkspace w = carve(reinterpret_cast<char*>(workspace) + fused_bytes, B, T, V, K, Lmax);
    if (w.ctc_bytes == 0) return PGASR_ERR_UNSUPPORTED;
    uint8_t* smp = io.samples ? io.samples : w.samples;
    float* lp = io.logp ? io.logp : w.logp;
    int32_t* hl = io.hyp_len ? io.hyp_len : w.hyp_len;
    int32_t* ds = io.dist ? io.dist : w.dist;
    float* rw = io.rewards ? io.rewards : w.rewards;
    float* nl = io.nll ? io.nll : w.nll;
    const bool dense = q.baseline_mode != PGASR_BASELINE_MEAN;   // sum_k A_k == 0 under the per-utterance mean
    int rc;
    if (do_pg || do_ctc) {
        // the sampler also produces the softmax the CTC lattice and the dense PG term read (exploration: it samples
        // softmax(theta z); the gradient kernel then forms p' itself and the CTC kernel its softmax of z)
        rc = explore ? softmax_sample_theta(io.logits, io.in_len, io.uniforms, seed, B, T, V, K, x.theta, smp, lp, nullptr, st)
                     : pgasr_softmax_sample(io.logits, io.in_len, io.uniforms, seed, B, T, V, K, smp, lp, w.probs, stream);
        if (rc) return rc;
    }
    if (do_pg) {
        rc = pgasr_collapse_u8(smp, io.in_len, K, B * K, T, q.blank, w.hyps, hl, stream);
        if (rc) return rc;
        if (words) {
            // word counts of the transcripts in the stand-alone nll scratch: unused when the caller takes nll, else first
            // written by the CTC part below, after the advantages have read them.  They are the lengths of the WER ratio.
            int32_t* nw = reinterpret_cast<int32_t*>(w.nll);
            rc = pgasr_word_edit_distance_u8(w.hyps, hl, B * K, T, io.targets, io.tgt_len, K, Lmax, q.word_sep, ds, nw,
                                             stream);
            if (rc) return rc;
            rc = pgasr_pg_advantages(ds, nw, lp, B, K, Lmax,
                                     q.reward_mode == PGASR_REWARD_NEG_WER ? PGASR_REWARD_NEG_CER : PGASR_REWARD_NEG_ED,
                                     q.baseline_mode, q.baseline_value, rw, w.adv, w.loss_terms, stream);
            if (rc) return rc;
        } else {
        rc = pgasr_edit_distance_u8(w.hyps, hl, B * K, T, io.targets, io.tgt_len, K, Lmax, V, ds, nullptr, stream);
        if (rc) return rc;
        rc = pgasr_pg_advantages(ds, io.tgt_len, lp, B, K, Lmax, q.reward_mode, q.baseline_mode, q.baseline_value, rw,
                                 w.adv, w.loss_terms, stream);
        if (rc) return rc;
        }
    }
    if (do_ctc && (cap & 1)) {
        a.do_pg = 0; a.rewards = nullptr; a.logp = nullptr; a.hyp_len = nullptr; a.dist = nullptr; a.samples = nullptr;
        a.nll = nl;
        rc = fused_step(a, workspace, st);                 // dlogits = (w_ctc / B) g_ctc, nll; loss is finalised below
        if (rc) return rc;
    } else if (do_ctc) {
        rc = pgasr_ctc_loss_grad(io.logits, explore ? nullptr : w.probs, io.targets, io.in_len, io.tgt_len, B, T, V, Lmax, q.blank,
                                 q.w_ctc / (float)B, 0, nl, io.dlogits, w.ctc, w.ctc_bytes, stream);
        if (rc) return rc;
    }
    if (do_pg && explore) {
        rc = pg_grad_explore(io.logits, smp, w.adv, io.in_len, B, T, V, K, q.w_pg / ((float)B * (float)K), dense,
                             do_ctc ? 1 : 0, x, w.loss_terms, io.dlogits, st);
        if (rc) return rc;
    } else if (do_pg) {
        rc = pgasr_pg_grad(smp, w.adv, dense ? w.probs : nullptr, io.in_len, B, T, V, K,
                           q.w_pg / ((float)B * (float)K), do_ctc ? 1 : 0, io.dlogits, stream);
        if (rc) return rc;
    }
    if (!do_pg && !do_ctc) PGASR_CUDA_TRY(cudaMemsetAsync(io.dlogits, 0, (size_t)B * T * V * sizeof(float), st));
    finalize_loss_kernel<<<1, 32, 0, st>>>(do_pg ? w.loss_terms : nullptr, do_ctc ? nl : nullptr, B, K, q.w_pg,
                                           q.w_ctc, io.loss);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

}  // namespace pgasr

extern "C" int pgasr_pg_ctc_step(const float* logits, const int32_t* targets, const int32_t* in_len,
                                 const int32_t* tgt_len, const float* uniforms, uint64_t seed, int B, int T,
                                 int V, int K, int Lmax, int blank, int reward_mode, int baseline_mode,
                                 float baseline_value, float w_pg, float w_ctc, float* loss, float* dlogits,
                                 float* rewards, float* logp, int32_t* hyp_len, int32_t* dist, float* nll,
                                 uint8_t* samples, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace pgasr;
    const StepParams q = {B, T, V, K, Lmax, blank, reward_mode, baseline_mode, baseline_value, w_pg, w_ctc, -1};
    if (!logits || !targets || !loss || !dlogits) return PGASR_ERR_INVALID_ARG;
    const int rc = step_check(q, workspace, workspace_bytes);
    if (rc) return rc;
    pgasr_step_io io;
    io.logits = logits; io.targets = targets; io.in_len = in_len; io.tgt_len = tgt_len; io.uniforms = uniforms;
    io.seed = 0; io.loss = loss; io.dlogits = dlogits; io.rewards = rewards; io.logp = logp; io.hyp_len = hyp_len;
    io.dist = dist; io.nll = nll; io.samples = samples; io.to_go = nullptr; io.r_pos = nullptr;
    return step_one(q, io, seed, workspace, as_stream(stream));
}

namespace pgasr {
// The extra streams of pgasr_pg_ctc_step_multi and the events that fork them from / join them to the caller's stream:
// one set per host thread and device, created on first use (the only objects the library keeps besides the
// control-block parity; they live as long as the thread).
struct AuxLane { cudaStream_t stream[kMaxLanes - 1]; cudaEvent_t fork, join[kMaxLanes - 1]; bool ok; };
static int aux_lane(AuxLane** out) {
    static thread_local AuxLane lanes[64] = {};
    int dev = 0;
    PGASR_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return PGASR_ERR_UNSUPPORTED;
    AuxLane& a = lanes[dev];
    if (!a.ok) {
        PGASR_CUDA_TRY(cudaEventCreateWithFlags(&a.fork, cudaEventDisableTiming));
        for (int i = 0; i < kMaxLanes - 1; ++i) {
            PGASR_CUDA_TRY(cudaStreamCreateWithFlags(&a.stream[i], cudaStreamNonBlocking));
            PGASR_CUDA_TRY(cudaEventCreateWithFlags(&a.join[i], cudaEventDisableTiming));
        }
        a.ok = true;
    }
    *out = &a;
    return PGASR_OK;
}
}  // namespace pgasr

// n steps with one call: the per-step cost on the host is one cudaLaunchKernelEx, nothing else (no Python, no
// allocation, no argument marshalling).  The steps of one call are independent by contract (no step's output is
// another step's input), so they rotate over the caller's stream and two more streams, each with its own lane
// of the workspace: consecutive steps OVERLAP -- the CTAs of step n + 1 fill the SMs step n leaves idle (2B of 148
// at the headline shape) and its tail -- while steps three apart stay ordered (same stream; programmatic dependent
// launch overlaps their launch latency).  The extra streams are forked from and joined back into `stream` with
// events, so to the caller the call is ordered on `stream` like any other.  PGASR_NO_OVERLAP=1: one stream.
namespace pgasr {
static int step_multi(const StepParams& q, const pgasr_step_io* steps, int n_steps, uint64_t seed_base,
                      void* workspace, size_t workspace_bytes, void* stream, float* const* entropy = nullptr);
}

extern "C" int pgasr_pg_ctc_step_multi(const pgasr_step_io* steps, int n_steps, uint64_t seed_base, int B, int T,
                                       int V, int K, int Lmax, int blank, int reward_mode, int baseline_mode,
                                       float baseline_value, float w_pg, float w_ctc, void* workspace,
                                       size_t workspace_bytes, void* stream) {
    using namespace pgasr;
    const StepParams q = {B, T, V, K, Lmax, blank, reward_mode, baseline_mode, baseline_value, w_pg, w_ctc, -1};
    return step_multi(q, steps, n_steps, seed_base, workspace, workspace_bytes, stream);
}

// the same with the word-level rewards (word_sep: the separator id; checked for every mode)
extern "C" int pgasr_pg_ctc_step_multi_ws(const pgasr_step_io* steps, int n_steps, uint64_t seed_base, int B, int T,
                                          int V, int K, int Lmax, int blank, int reward_mode, int baseline_mode,
                                          float baseline_value, float w_pg, float w_ctc, int word_sep, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    using namespace pgasr;
    if (word_sep < 0 || word_sep >= V || word_sep == blank) return PGASR_ERR_INVALID_ARG;
    const StepParams q = {B, T, V, K, Lmax, blank, reward_mode, baseline_mode, baseline_value, w_pg, w_ctc, word_sep};
    return step_multi(q, steps, n_steps, seed_base, workspace, workspace_bytes, stream);
}

// the same with the exploration controls and every reward mode (word_sep < 0: no separator, character modes only)
extern "C" int pgasr_pg_ctc_step_multi_ex(const pgasr_step_io* steps, int n_steps, uint64_t seed_base, int B, int T,
                                          int V, int K, int Lmax, int blank, int reward_mode, int baseline_mode,
                                          float baseline_value, float w_pg, float w_ctc, float* const* entropy,
                                          int word_sep, float temperature, float w_ent, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    using namespace pgasr;
    if (!std::isfinite(temperature) || !(temperature >= 0.01f && temperature <= 100.0f)) return PGASR_ERR_INVALID_ARG;
    if (!std::isfinite(w_ent) || !(w_ent >= 0.0f) || (w_ent > 0.0f && w_pg == 0.0f)) return PGASR_ERR_INVALID_ARG;
    if (word_sep >= 0 && (word_sep >= V || word_sep == blank)) return PGASR_ERR_INVALID_ARG;
    if (!steps || n_steps < 0) return PGASR_ERR_INVALID_ARG;
    if (entropy && w_pg == 0.0f)                           // (H_b comes from the PG role)
        for (int i = 0; i < n_steps; ++i)
            if (entropy[i]) return PGASR_ERR_INVALID_ARG;
    StepParams q = {B, T, V, K, Lmax, blank, reward_mode, baseline_mode, baseline_value, w_pg, w_ctc,
                    word_sep < 0 ? -1 : word_sep};
    q.temperature = temperature;
    q.w_ent = w_ent;
    return step_multi(q, steps, n_steps, seed_base, workspace, workspace_bytes, stream, entropy);
}

namespace pgasr {
static int step_multi(const StepParams& q, const pgasr_step_io* steps, int n_steps, uint64_t seed_base,
                      void* workspace, size_t workspace_bytes, void* stream, float* const* entropy) {
    const int B = q.B, T = q.T, V = q.V, K = q.K, Lmax = q.Lmax;
    if (!steps || n_steps < 0) return PGASR_ERR_INVALID_ARG;
    int rc = step_check(q, workspace, workspace_bytes);
    if (rc) return rc;
    static const bool no_overlap = getenv("PGASR_NO_OVERLAP") != nullptr;
    cudaStream_t s0 = as_stream(stream);
    const size_t lane_bytes = step_lane_bytes(B, T, V, K, Lmax);
    const int nl = (n_steps >= 2 && !no_overlap) ? (step_lanes() < n_steps ? step_lanes() : n_steps) : 1;
    AuxLane* aux = nullptr;
    if (nl > 1) {
        rc = aux_lane(&aux);
        if (rc) return rc;
        PGASR_CUDA_TRY(cudaEventRecord(aux->fork, s0));
        for (int l = 1; l < nl; ++l) PGASR_CUDA_TRY(cudaStreamWaitEvent(aux->stream[l - 1], aux->fork, 0));
    }
    for (int i = 0; i < n_steps; ++i) {
        const int l = i % nl;
        rc = step_one(q, steps[i], seed_base + steps[i].seed, reinterpret_cast<char*>(workspace) + (size_t)l * lane_bytes,
                      l ? aux->stream[l - 1] : s0, nl > 1, entropy ? entropy[i] : nullptr);
        if (rc) break;
    }
    for (int l = 1; l < nl; ++l) {                         // join, also after an error: the caller's stream stays the one order
        PGASR_CUDA_TRY(cudaEventRecord(aux->join[l - 1], aux->stream[l - 1]));
        PGASR_CUDA_TRY(cudaStreamWaitEvent(s0, aux->join[l - 1], 0));
    }
    return rc;
}
}  // namespace pgasr
