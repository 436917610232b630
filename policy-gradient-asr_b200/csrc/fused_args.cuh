// Arguments of the single-launch kernel (fused.cu) and the host-side entry points other translation units call.
#pragma once
#include "pgasr_common.cuh"

namespace pgasr {

struct FusedArgs {
    const float* logits; const int32_t* targets; const int32_t* in_len; const int32_t* tgt_len;
    const float* uniforms; unsigned long long seed;
    int B, T, V, K, Lmax, blank, reward_mode, baseline_mode;
    float baseline_value, w_pg, w_ctc;
    int do_pg, do_ctc;
    int pg_pair;             // a PG CTA serves two utterances (their edit distances side by side); grid = B + ceil(B / 2)
    int no_pdl;              // host side only: launch without programmatic stream serialisation (steps of a multi-step call)
    int bulk_tile;           // the roles' logits tiles arrive as ONE bulk copy (cp.async.bulk + mbarrier) instead of 16-byte cp.async
    int cdf_smem;            // PG role: the per-frame CDF rows live in shared memory ([T][33] fp32, V <= 32, tile mode) -- rolled
                             // loops and a binary search instead of 32 registers and a select tree (fused_impl.cuh P1)
    float* loss; float* dlogits;
    float* rewards; float* logp; int32_t* hyp_len; int32_t* dist; float* nll; uint8_t* samples;   // optional
    int16_t* to_go; int8_t* r_pos;                                                                // optional (reward-to-go)
    unsigned* ctrl;          // [0] role ticket, [1] done ticket, [4 + b] CTC-done flag of utterance b
    double* lattice; int* lat_exp; float* loss_terms; float* nll_ws;
    float* tile_g;           // global-tile mode: [B][T + 2][RS] fp32 softmax rows (guard row before and after)
};

// Word-level rewards (reward_mode PGASR_REWARD_NEG_WED / _NEG_WER): a kernel argument of its own, next to FusedArgs, so
// that the character-mode kernels keep their parameter block
struct WordArgs {
    int sep;                 // id of the word separator, in [0, V), != blank
    int cap;                 // word_class_cap(Lmax, V): distinct transcript words a hypothesis can match
};

// Exploration controls (DESIGN.md "exploration spec"): the PG role samples from and trains softmax(theta z), with an
// entropy bonus.  A kernel argument of its own, like WordArgs, so the default kernels keep their parameter block.
struct ExploreArgs {
    float theta;             // fl32(1 / temperature)
    float ent_c;             // beta / B: the entropy term's gradient is ent_c theta p' (log p' + H_bt)
    float ent_lt;            // beta K / w_pg: subtracted (times H_b) from the utterance's loss term
    float* entropy;          // [B] H_b in nats, optional
};

// Entropy terms of the exploration variant with 0 log 0 = 0: a class whose p' is 0 (underflow, or a logit of -inf, where
// log p' = -inf) contributes 0 to H and gets gradient 0, instead of 0 * -inf = NaN.
__device__ __forceinline__ float ent_plogp(float p, float lp) { return p > 0.0f ? p * lp : 0.0f; }
__device__ __forceinline__ float ent_grad(float p, float c) { return p > 0.0f ? p * c : 0.0f; }

// shared-memory bytes of one utterance's block in a PG CTA (fused_impl.cuh: fused_pg_role; fused.cu sizes with it)
template <int W, int kThreads>
__host__ __device__ inline size_t pg_u_bytes(int T, int V, int K) {
    const int Tp = (T + 15) & ~15, Tp2 = (T / 2 + 16) & ~15;
    size_t off = (size_t)2 * K * Tp + (size_t)K * Tp2 + (size_t)2 * (V + 1) * W * 4 + (size_t)((K + 7) & ~7) * (W * 32 + 2) * 2;
    off = (off + 15) & ~(size_t)15;
    off += (size_t)(kThreads / 32) * 64 * 8 + 3 * 64 * 4 + 16;
    return (off + 15) & ~(size_t)15;
}

// bit 0: the CTC role fits (tile in shared memory or streamed from the workspace), bit 1: the PG role fits too
int fused_capability(int T, int V, int K, int Lmax);
// 0 when the fused kernel cannot take this shape at all
size_t fused_workspace_bytes(int B, int T, int V, int K, int Lmax);
// a.do_pg must be 0 when the PG role does not fit; the control block at the start of `workspace` must be zero
// (armed once: the kernel re-arms it when it finishes)
// throughput: the step is one of several independent ones in flight (pgasr_pg_ctc_step_multi): PG CTAs take two
// utterances each -- less SM time per step, a longer single step; a step on its own keeps one utterance per PG CTA
// word (non-NULL): the word-level rewards, a.do_pg set; the PG role must fit in its word layout (fused_word_capability)
// explore (non-NULL): the exploration variant of the PG role (a.do_pg set)
int fused_step(FusedArgs& a, void* workspace, cudaStream_t st, bool throughput = false, const WordArgs* word = nullptr,
               const ExploreArgs* explore = nullptr);
// the PG role of the word-level rewards fits an SM (logits tile in shared memory); otherwise the step chains the
// stand-alone kernels for the PG part
bool fused_word_capability(int T, int V, int K, int Lmax);
size_t align256(size_t x);
void fused_workspace_reset(const void* workspace, size_t bytes);   // forget the control-block parity of every fused workspace in the range
// chain path of the exploration variant: the sampler on theta z (sampler.cu); the PG gradient with the theta factor,
// the entropy term and H_b, which it also folds into loss_terms (pg.cu)
int softmax_sample_theta(const float* logits, const int32_t* in_len, const float* uniforms, uint64_t seed, int B, int T,
                         int V, int K, float theta, uint8_t* samples, float* logp, float* probs, cudaStream_t st);
int pg_grad_explore(const float* logits, const uint8_t* samples, const float* adv, const int32_t* in_len, int B, int T,
                    int V, int K, float scale, bool dense, int accumulate, const ExploreArgs& x, float* loss_terms,
                    float* dlogits, cudaStream_t st);

}  // namespace pgasr
