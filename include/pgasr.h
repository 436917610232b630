/*
 * pgasr.h -- C ABI of libpgasr_b200.so: the PG-loss + CTC hot path of Policy-Gradient-ASR on B200.
 *
 * The upstream project is pure Python: its "plugin interface" for this path is a handful of Python
 * functions and one nn.Module slot (SURVEY.md section 8b).  This header is what those bind to.  Every
 * entry point is extern "C", takes plain device pointers and sizes, allocates nothing, keeps no
 * global state (exceptions: the control-block parity of a step workspace lane and the per-thread extra streams of
 * pgasr_pg_ctc_step_multi, see there), enqueues its work on the
 * caller's stream (a cudaStream_t passed as void*; NULL = the
 * legacy default stream) and returns a pgasr_status.  All pointers are device pointers borrowed until
 * the stream work completes, unless a parameter says "host".  There is no CPU fallback: without a
 * sm_100 device every compute call returns PGASR_ERR_NO_DEVICE / a CUDA error.
 *
 * Upstream interface each entry point stands in for (paths relative to the upstream repository):
 *   pgasr_edit_distance_u8 / _i32   metrics.py:4-21     edit_dist(s1, s2) -> (distance, len(s1))
 *   pgasr_collapse_u8               CTCdecoder.py:119-131 collapse_fn(preds)  (+ blank drop, :41)
 *   pgasr_edit_distance_u8 last_col policy_grad.py:10-15  reward(): ED(y*, yhat[:t]) for every t
 *   pgasr_nll_sum_forward/backward  loss.py:13-17       customNLLLoss.forward(inp, target)
 *   pgasr_softmax_sample            (no upstream code)  K hypotheses per utterance from the posteriors
 *   pgasr_pg_advantages / _pg_grad  (no upstream code)  reward, baseline, REINFORCE gradient
 *   pgasr_ctc_loss_grad             (no upstream code)  CTC alpha-beta loss and gradient
 *   pgasr_pg_ctc_step               model.py:235-237    criterion(model_out, t); loss.backward()
 *                                                       -- the whole loss step in one call
 *   pgasr_host_*                    model.py:317-320    the same step on HOST arrays, pipelined
 *   pgasr_ctc_beam_search           CTCdecoder.py:41-116 CTCDecoder.decode(probs, beam_size, blank)
 * The Python binding a maintainer adds is shown in INTEGRATION.md.
 *
 * Layouts (all contiguous, batch first as upstream: batch_first=True, model.py:44,55):
 *   logits / probs / dlogits  [B,T,V] fp32      targets [B,Lmax] int32, padded with 0 (data.py:99)
 *   in_len [B], tgt_len [B] int32               uniforms [B,K,T] fp32 in [0,1)
 *   samples / hyps [B,K,T] uint8 (V <= 256)     hyp_len / dist [B,K] int32
 *   logp / rewards / adv [B,K] fp32             nll [B] fp32
 */
#ifndef PGASR_H_
#define PGASR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGASR_ABI_VERSION 1

#if defined(__GNUC__)
#define PGASR_API __attribute__((visibility("default")))
#else
#define PGASR_API
#endif

typedef enum {
    PGASR_OK = 0,
    PGASR_ERR_INVALID_ARG = -1,   /* NULL pointer, negative size, size over a documented limit */
    PGASR_ERR_UNSUPPORTED = -2,   /* legal request this build has no kernel for (e.g. V > 64 sampler) */
    PGASR_ERR_NO_DEVICE = -3,     /* no CUDA device of compute capability 10.x */
    PGASR_ERR_WORKSPACE = -4,     /* workspace too small; ask pgasr_*_workspace_bytes */
    PGASR_ERR_CUDA = -5           /* a CUDA call failed; pgasr_last_cuda_error() has the code */
} pgasr_status;

/* reward_mode: R = -ED  |  R = -ED/len(ref)  (the CER ratio of metrics.py:24-25)  |  per-position rewards
 * r_i = -(ED(ref, hyp[:i+1]) - ED(ref, hyp[:i])) (policy_grad.py:10-15) credited to the frames that can still
 * influence them: reward-to-go G_t = sum over the symbols emitted at frames >= t (DESIGN.md "reward-to-go spec") */
enum { PGASR_REWARD_NEG_ED = 0, PGASR_REWARD_NEG_CER = 1, PGASR_REWARD_ED_TO_GO = 2, PGASR_REWARD_MAX = 2 };
/* word-level reward_mode (pgasr_pg_ctc_step_multi_ws only): R = -ED_w | R = -ED_w / n_w (the WER ratio of
 * metrics.py:23-31), ED_w = Levenshtein distance between the WORD sequences of transcript and collapsed hypothesis,
 * n_w = number of transcript words.  Words: the ids split at every occurrence of the separator id word_sep, exactly
 * as Python's str.split(" ") splits a string (empty words kept: count(sep) + 1 words; the empty transcript is one
 * empty word, so n_w >= 1).  Equals the upstream string split when every alphabet entry is one character
 * (DESIGN.md "word reward spec").  PGASR_REWARD_MAX stays the bound of the entry points without word_sep. */
enum { PGASR_REWARD_NEG_WED = 3, PGASR_REWARD_NEG_WER = 4 };
/* baseline_mode: none | mean over the utterance's K samples | leave-one-out mean | external scalar */
enum { PGASR_BASELINE_NONE = 0, PGASR_BASELINE_MEAN = 1, PGASR_BASELINE_LOO = 2, PGASR_BASELINE_VALUE = 3 };

PGASR_API int         pgasr_abi_version(void);
PGASR_API const char* pgasr_status_string(int status);
PGASR_API int         pgasr_last_cuda_error(void);          /* cudaError_t of the last failing CUDA call (thread local) */
PGASR_API uint64_t    pgasr_launch_count(void);             /* kernels launched so far by the calling thread */
PGASR_API int         pgasr_device_check(void);             /* PGASR_OK iff the current device is sm_10x */

/* ---- a6: fused softmax + inverse-CDF categorical sampler ------------------------------------
 * samples[b,k,t] ~ Categorical(softmax(logits[b,t,:])) for t < in_len[b] (0 beyond), from
 * uniforms[b,k,t] when given, else Philox4x32-10(seed; counter (t, b, k/4, 'PGAS'), lane k%4).
 * logp[b,k] = sum_t log_softmax(logits[b,t,:])[samples[b,k,t]].  probs (optional) receives the
 * softmax.  Bit-exact contract: DESIGN.md "sampler spec".  V <= 64, K <= 64.                   */
PGASR_API int pgasr_softmax_sample(const float* logits, const int32_t* in_len, const float* uniforms,
                         uint64_t seed, int B, int T, int V, int K,
                         uint8_t* samples, float* logp, float* probs, void* stream);

/* ---- a3: repeat merge then blank drop on N rows of length <= T -------------------------------
 * Row r has length seq_len[r / rows_per_len] (seq_len NULL: T).  blank < 0: merge repeats only
 * (exactly collapse_fn).  out rows are zero filled beyond out_len[r].                          */
PGASR_API int pgasr_collapse_u8(const uint8_t* seqs, const int32_t* seq_len, int rows_per_len, int N, int T,
                      int blank, uint8_t* out, int32_t* out_len, void* stream);

/* ---- a1/a4: Levenshtein distance, N hypothesis rows against N/rows_per_ref references --------
 * dist[r] = ED(refs[r / rows_per_ref, :ref_len], hyps[r, :hyp_len[r]]), unit costs.
 * _u8: tokens < vocab <= 256, ref_len <= 512; bit-parallel (Myers/Hyyro) one thread per row.
 *      last_col (optional) [N, hyp_stride+1] int32 receives ED(ref, hyp[:i]) for i = 0..hyp_len.
 * _i32: arbitrary int32 tokens (word ids, code points), anti-diagonal wavefront in shared memory,
 *      one CTA per row; ref_len <= 4096.                                                       */
PGASR_API int pgasr_edit_distance_u8(const uint8_t* hyps, const int32_t* hyp_len, int N, int hyp_stride,
                           const int32_t* refs, const int32_t* ref_len, int rows_per_ref,
                           int ref_stride, int vocab, int32_t* dist, int32_t* last_col, void* stream);
/* ---- word edit distance: the same rows split into words at the separator id sep ---------------
 * dist[r] = ED_w(refs[r / rows_per_ref, :ref_len], hyps[r, :hyp_len[r]]): Levenshtein distance over the word
 * sequences (words compared by their ids; split semantics of PGASR_REWARD_NEG_WED), unit costs.
 * ref_words (optional) [N / rows_per_ref] receives n_w = count(sep in ref) + 1 per reference: passed as the tgt_len
 * of pgasr_pg_advantages with PGASR_REWARD_NEG_CER it gives the WER reward -ED_w / n_w.  ref_len <= 511
 * (ref_stride <= 511), rows_per_ref <= 1024.  One CTA per reference, one warp per row.                         */
PGASR_API int pgasr_word_edit_distance_u8(const uint8_t* hyps, const int32_t* hyp_len, int N, int hyp_stride,
                                const int32_t* refs, const int32_t* ref_len, int rows_per_ref, int ref_stride,
                                int sep, int32_t* dist, int32_t* ref_words, void* stream);
PGASR_API int pgasr_edit_distance_i32(const int32_t* hyps, const int32_t* hyp_len, int N, int hyp_stride,
                            const int32_t* refs, const int32_t* ref_len, int rows_per_ref,
                            int ref_stride, int32_t* dist, void* stream);

/* ---- a7: rewards, baseline, advantages and the per-utterance PG loss terms -------------------
 * rewards/adv [B,K]; loss_terms[b] = -sum_k adv[b,k] * logp[b,k].                              */
PGASR_API int pgasr_pg_advantages(const int32_t* dist, const int32_t* tgt_len, const float* logp,
                        int B, int K, int Lmax, int reward_mode, int baseline_mode,
                        float baseline_value, float* rewards, float* adv, float* loss_terms,
                        void* stream);
/* dlogits[b,t,v] (+)= scale * ( probs[b,t,v] * sum_k adv[b,k] - sum_k adv[b,k] [samples[b,k,t]==v] )
 * for t < in_len[b], 0 beyond.  probs may be NULL when the dense term vanishes (mean baseline). */
PGASR_API int pgasr_pg_grad(const uint8_t* samples, const float* adv, const float* probs,
                  const int32_t* in_len, int B, int T, int V, int K, float scale, int accumulate,
                  float* dlogits, void* stream);

/* ---- a8: CTC alpha-beta loss and gradient ------------------------------------------------------
 * nll[b] = -log p(targets[b] | logits[b]); dlogits (+)= grad_scale * d nll[b] / d logits[b].
 * probs: softmax of logits if the caller already has it (pgasr_softmax_sample), else NULL and the
 * kernel computes it into its workspace.  No valid alignment: nll = +inf, zero gradient.
 * With logits given, accumulate == 0 and V <= 64 this is the CTC role of the single-launch kernel below (walker and
 * gradient-worker warps, any T); otherwise the classic one-CTA-per-utterance kernel.
 * Lmax <= 511.  workspace: pgasr_ctc_workspace_bytes(B,T,V,Lmax) bytes, 256-byte aligned.       */
PGASR_API size_t pgasr_ctc_workspace_bytes(int B, int T, int V, int Lmax);
PGASR_API int pgasr_ctc_loss_grad(const float* logits, const float* probs, const int32_t* targets,
                        const int32_t* in_len, const int32_t* tgt_len, int B, int T, int V, int Lmax,
                        int blank, float grad_scale, int accumulate, float* nll, float* dlogits,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- a5: customNLLLoss (loss.py:13-17) ---------------------------------------------------------
 * inp [L,B,V] log-probs, target [B,L] int64.  loss = sum_i mean_b(-inp[i,b,target[b,i]]),
 * ignoring entries equal to ignore_index (any value, e.g. torch's -100; PGASR_NO_IGNORE for none).  A target
 * outside [0,V) that is not ignored makes the loss NaN (torch raises there); nothing is read out of bounds.
 * backward: grad_inp = grad_out * d loss / d inp (dense write, zero elsewhere).                 */
#define PGASR_NO_IGNORE (-2147483647 - 1)
PGASR_API int pgasr_nll_sum_forward(const float* inp, const int64_t* target, int L, int B, int V,
                          int ignore_index, float* loss, void* stream);
PGASR_API int pgasr_nll_sum_backward(const int64_t* target, const float* grad_out, int L, int B, int V,
                           int ignore_index, float* grad_inp, void* stream);

/* ---- the whole step (what criterion(model_out, t) + loss.backward() cost upstream) ------------
 * sample -> collapse -> edit distance -> reward -> baseline -> REINFORCE gradient, plus CTC, with
 *   loss[0]  = w_pg * L_pg + w_ctc * mean_b nll[b]
 *   dlogits  = w_pg * g_pg + (w_ctc / B) * g_ctc                     (written once, not accumulated)
 * Optional outputs (NULL to skip): rewards, logp, hyp_len, dist, nll, samples.
 * workspace: pgasr_pg_ctc_step_workspace_bytes(B,T,V,K,Lmax) bytes (three lanes, see pgasr_pg_ctc_step_multi), 256-byte
 * aligned, armed ONCE with pgasr_pg_ctc_step_workspace_init before its first use (and again after a step that returned
 * an error); one workspace serves one stream at a time.  The step kernel is launched with programmatic stream
 * serialisation: back-to-back steps on one stream overlap the launch of step n+1 with the tail of step n (the CTAs of
 * n+1 wait on the grid dependency before they touch any input or output); for that a lane holds two control blocks that
 * consecutive launches use alternately -- the library remembers, per lane pointer, which one is next (host side).
 * V <= 64 (register-resident fast paths up to 32 classes), K <= 64.  One kernel launch for every shape whose sample
 * buffers fit an SM (2.5 K T <= ~200 KB); targets / in_len / tgt_len and the small outputs may live in pinned host
 * memory mapped into the device (they are read once per CTA / written once).                       */
PGASR_API size_t pgasr_pg_ctc_step_workspace_bytes(int B, int T, int V, int K, int Lmax);
/* (init also forgets which control block the workspace pointer used last, so a freed and recycled pointer is safe) */
PGASR_API int pgasr_pg_ctc_step_workspace_init(void* workspace, size_t workspace_bytes, void* stream);
PGASR_API int pgasr_pg_ctc_step(const float* logits, const int32_t* targets, const int32_t* in_len,
                      const int32_t* tgt_len, const float* uniforms, uint64_t seed,
                      int B, int T, int V, int K, int Lmax, int blank,
                      int reward_mode, int baseline_mode, float baseline_value,
                      float w_pg, float w_ctc,
                      float* loss, float* dlogits, float* rewards, float* logp, int32_t* hyp_len,
                      int32_t* dist, float* nll, uint8_t* samples,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---- n steps with one call (micro-batches of one optimiser step; a bench loop) ---------------------------
 * steps: HOST array of n_steps records of DEVICE pointers, same meaning as the arguments of pgasr_pg_ctc_step
 * (optional ones may be NULL); step i samples with Philox(seed_base + steps[i].seed).  Per step the host does one
 * kernel launch and nothing else.
 * The steps of one call must be INDEPENDENT: no step's output buffer may be another step's input or output.  They
 * are enqueued in rotation on `stream` and on two more streams the library forks from `stream` (event) and joins back
 * into it before the call returns, each with its own lane of the workspace, so consecutive steps overlap on the GPU
 * while, to the caller, everything is ordered on `stream` as usual.  The extra streams and their events are created
 * on first use, one set per calling host thread and device, and live as long as the thread (together with the
 * control-block parity above this is all the state the library keeps).  PGASR_NO_OVERLAP=1 in the environment keeps
 * every step on `stream`.  The steps of a multi-step call are launched in plain stream order (no programmatic
 * serialisation: with three lanes in flight it only parked the next step's CTAs on SMs another lane could use).
 * reward_mode PGASR_REWARD_ED_TO_GO (single-launch kernel with the logits tile in shared memory only; else
 * PGASR_ERR_UNSUPPORTED): to_go [B,K,T] int16 and r_pos [B,K,T] int8 (optional) receive the reward-to-go of every
 * frame and the per-position reward of every collapsed symbol (zero beyond hyp_len); rewards = len(ref) - ED.   */
typedef struct pgasr_step_io {
    const float* logits; const int32_t* targets; const int32_t* in_len; const int32_t* tgt_len;
    const float* uniforms; uint64_t seed;
    float* loss; float* dlogits;
    float* rewards; float* logp; int32_t* hyp_len; int32_t* dist; float* nll; uint8_t* samples;
    int16_t* to_go; int8_t* r_pos;
} pgasr_step_io;
PGASR_API int pgasr_pg_ctc_step_multi(const pgasr_step_io* steps, int n_steps, uint64_t seed_base,
                            int B, int T, int V, int K, int Lmax, int blank,
                            int reward_mode, int baseline_mode, float baseline_value,
                            float w_pg, float w_ctc,
                            void* workspace, size_t workspace_bytes, void* stream);
/* The same with the word-level rewards: reward_mode may also be PGASR_REWARD_NEG_WED / _NEG_WER, word_sep is the id
 * of the word separator (the space of the alphabet), in [0, V) and != blank (else PGASR_ERR_INVALID_ARG; it is
 * checked, and ignored, for the character modes too).  The only entry point that takes the word modes; they are
 * rejected everywhere else.  dist receives ED_w, hyp_len stays the length of the collapsed hypothesis in ids.  Same
 * workspace (pgasr_pg_ctc_step_workspace_bytes) and kernel launches as the character modes: the single-launch kernel
 * when its word-mode shared memory fits an SM, else the chain of stand-alone kernels with
 * pgasr_word_edit_distance_u8.  Lmax <= 511.                                                                    */
PGASR_API int pgasr_pg_ctc_step_multi_ws(const pgasr_step_io* steps, int n_steps, uint64_t seed_base,
                            int B, int T, int V, int K, int Lmax, int blank,
                            int reward_mode, int baseline_mode, float baseline_value,
                            float w_pg, float w_ctc, int word_sep,
                            void* workspace, size_t workspace_bytes, void* stream);
/* The same with the exploration controls (DESIGN.md "exploration spec"): the PG role samples from and trains the
 * tempered policy softmax(z / temperature), theta = fl32(1 / temperature), and the loss gains an entropy bonus:
 *   loss = w_pg L_pg + w_ctc mean_b nll_b - w_ent (1/B) sum_b H_b,   H_b = sum_{t < in_len[b]} H(softmax(theta z_bt))
 * in nats.  The CTC term stays on the untempered logits.  entropy: HOST array of n_steps DEVICE pointers to [B] fp32
 * that receive H_b (the array or any element may be NULL; an element needs w_pg != 0).  word_sep < 0: no separator
 * (character modes only); word_sep >= 0: as in pgasr_pg_ctc_step_multi_ws.  Every reward mode is accepted.
 * PGASR_ERR_INVALID_ARG before any CUDA call: temperature non-finite or outside [0.01, 100], w_ent non-finite or < 0,
 * w_ent > 0 or an entropy output with w_pg == 0, a bad separator.  With temperature 1, w_ent 0 and no entropy output
 * the step is exactly the one pgasr_pg_ctc_step_multi (_ws) runs.  Same workspace.                                */
PGASR_API int pgasr_pg_ctc_step_multi_ex(const pgasr_step_io* steps, int n_steps, uint64_t seed_base,
                            int B, int T, int V, int K, int Lmax, int blank,
                            int reward_mode, int baseline_mode, float baseline_value,
                            float w_pg, float w_ctc, float* const* entropy, int word_sep,
                            float temperature, float w_ent,
                            void* workspace, size_t workspace_bytes, void* stream);

/* ---- CTC prefix beam search (upstream CTCdecoder.py:41-116, CTCDecoder.decode) -----------------------
 * probs [N,T,V] fp64 post-softmax (upstream takes the post-softmax array and works in Python floats), frames
 * t >= in_len[n] ignored (in_len NULL: T).  labels [N,T] int32 receives the best prefix of each utterance (zero
 * filled beyond label_len[n]), nll[n] = -log(p_blank + p_non_blank) of that prefix, as upstream returns.
 * One CTA per utterance; V <= 64, beam <= 128.  workspace: pgasr_ctc_beam_search_workspace_bytes(N,T,V,beam).  */
PGASR_API size_t pgasr_ctc_beam_search_workspace_bytes(int N, int T, int V, int beam);
PGASR_API int pgasr_ctc_beam_search(const double* probs, const int32_t* in_len, int N, int T, int V, int beam,
                          int blank, int32_t* labels, int32_t* label_len, double* nll,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- the step on HOST buffers (upstream hands the metric/reward code host arrays: model.py:317-320) ----
 * A pipeline owns the device buffers for `depth` steps in flight, three streams (copy-in, compute, copy-out)
 * and the step workspace; create/destroy are the only calls that allocate.  submit() takes HOST pointers
 * (page-locked for the copies to be asynchronous: pgasr_host_pin, or any pinned allocation), enqueues
 * H2D -> pgasr_pg_ctc_step -> D2H and returns a ticket without waiting; it blocks only when the step
 * submitted `depth` steps earlier has not finished.  wait(ticket) returns once the outputs of every step up to
 * `ticket` are in the caller's host buffers (ticket < 0: all submitted steps).  in_len_h / tgt_len_h may be
 * NULL (full lengths), rewards_h / nll_h may be NULL.  Sampling is Philox(seed).  One pipeline serves one host
 * thread at a time.  Host input buffers may be reused as soon as wait() for that step returns.            */
typedef struct pgasr_host_pipeline pgasr_host_pipeline;
PGASR_API int pgasr_host_create(int B, int T, int V, int K, int Lmax, int depth, pgasr_host_pipeline** out);
PGASR_API int pgasr_host_destroy(pgasr_host_pipeline* p);
PGASR_API int pgasr_host_submit(pgasr_host_pipeline* p, const float* logits_h, const int32_t* targets_h,
                      const int32_t* in_len_h, const int32_t* tgt_len_h, uint64_t seed, int blank,
                      int reward_mode, int baseline_mode, float baseline_value, float w_pg, float w_ctc,
                      float* loss_h, float* dlogits_h, float* rewards_h, float* nll_h, int64_t* ticket);
PGASR_API int pgasr_host_wait(pgasr_host_pipeline* p, int64_t ticket);
PGASR_API int pgasr_host_pin(void* ptr, size_t bytes);      /* cudaHostRegister / cudaHostUnregister */
PGASR_API int pgasr_host_unpin(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* PGASR_H_ */
