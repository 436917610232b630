// Host side of the single-launch kernel: what fits where (fused_plan), workspace layout, dispatch to the per-SPL
// translation units (fused_spl4/8/16/32.cu, which instantiate fused_impl.cuh).
#include <cstdlib>
#include <mutex>
#include <map>

#include "ctc_core.cuh"
#include "fused_args.cuh"
#include "words_core.cuh"

namespace pgasr {

constexpr int kFusedMaxK = 64;
int launch_fused_spl4(int mode, FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word,
                       const ExploreArgs* explore);
int launch_fused_spl8(int mode, FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word,
                       const ExploreArgs* explore);
int launch_fused_spl16(int mode, FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word,
                        const ExploreArgs* explore);
int launch_fused_spl32(int mode, FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word,
                        const ExploreArgs* explore);

constexpr size_t kFusedSmemLimit = 220 * 1024;

// Host-side state of the library: which of a fused workspace's two control blocks its next step uses (ordered map:
// pgasr_pg_ctc_step_workspace_init drops every entry inside the range it is given, so a recycled pointer starts
// afresh).  A fused workspace seen for the first time gets its control blocks zeroed on the launching stream.
static std::mutex g_parity_mu;
static std::map<uintptr_t, unsigned> g_parity;
static unsigned workspace_parity(const void* ws, bool* fresh) {
    std::lock_guard<std::mutex> lk(g_parity_mu);
    auto it = g_parity.find(reinterpret_cast<uintptr_t>(ws));
    *fresh = it == g_parity.end();
    if (*fresh) it = g_parity.emplace(reinterpret_cast<uintptr_t>(ws), 0u).first;
    return it->second++ & 1u;
}
void fused_workspace_reset(const void* ws, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_parity_mu);
    const uintptr_t lo = reinterpret_cast<uintptr_t>(ws);
    g_parity.erase(g_parity.lower_bound(lo), g_parity.lower_bound(lo + (bytes ? bytes : 1)));
}

struct FusedWs { size_t ctrl, lat, exps, terms, nll, tile, total; };

static FusedWs fused_ws(int B, int T, int V, int spl, bool gt) {
    FusedWs w;
    w.ctrl = align_up((size_t)2 * (4 + B) * sizeof(unsigned), 256);   // two control blocks, used alternately
    w.lat = align_up((size_t)B * T * spl * 32 * sizeof(double), 256);
    w.exps = align_up((size_t)B * T * sizeof(int), 256);
    w.terms = align_up((size_t)B * sizeof(float), 256);
    w.nll = align_up((size_t)B * sizeof(float), 256);
    w.tile = gt ? align_up((size_t)B * (T + 2) * ctc_row_stride_f32(V) * sizeof(float), 256) : 0;
    w.total = w.ctrl + w.lat + w.exps + w.terms + w.nll + w.tile;
    return w;
}

// block workers (ctc_core.cuh): tile with an odd row stride, rings of 10 frames, two transposed occupancy matrices per
// direction, the class-ordered label list
static size_t ctc_role_smem_bw(int T, int V, int spl) {
    const int RS = (V + 1) | 1;
    const size_t tile = (((size_t)(T + 4) * RS * sizeof(float) + 15) & ~(size_t)15);
    const size_t ring = spl == 4 ? grad_ring_bytes<4, kBwNB>() : grad_ring_bytes<8, kBwNB>();
    const size_t gam = 2 * (spl == 4 ? bw_gam_bytes<4>() : bw_gam_bytes<8>());
    return tile + 128 /* matrix alignment */ + 2 * ring + gam + (size_t)(2 * V + 1 + 512 + 512) * sizeof(int) + 16 +
           (size_t)2 * kBwGB * kBwListWords * sizeof(unsigned) + (size_t)2 * kBwGB * 8 + (size_t)2 * kBwGB * bw_stage_bytes();
}

static size_t ctc_role_smem(int T, int V, int spl, int threads, bool gt) {
    const int RS = ctc_row_stride_f32(V);
    const size_t ring = spl == 4 ? grad_ring_bytes<4>() : spl == 8 ? grad_ring_bytes<8>() : spl == 16 ? grad_ring_bytes<16>() : grad_ring_bytes<32>();
    const int G = (threads / 32 - 2) / 2, per = (batch_of(spl) + G - 1) / G;
    const size_t pring = (size_t)kPRows * (RS <= 32 ? 32 : RS <= 64 ? 64 : 128) * 4;
    const size_t tile = gt ? 3 * pring /* two rings + alignment slack */ : (((size_t)(T + 4) * RS * sizeof(float) + 15) & ~(size_t)15);
    return tile + 2 * ring + (size_t)2 * G * per * 16 * spl * sizeof(int) + (size_t)(2 * V + 1 + 512 + 512) * sizeof(int);
}

static size_t pg_cdf_bytes(int threads) { return (size_t)threads * 33 * sizeof(float) + 16; }
// (mirrors the carve-up of fused_pg_role: the tile, one block per utterance of the CTA, reward-to-go arrays, CDF rows)
static size_t pg_role_smem(int T, int V, int K, int spl, int threads, bool stream, bool togo = false, bool cdf = false, int nutt = 1) {
    const int Tp = (T + 15) & ~15, W = spl / 2;
    const size_t ub = W == 2 ? pg_u_bytes<2, 512>(T, V, K) : W == 4 ? pg_u_bytes<4, 512>(T, V, K) :
                      W == 8 ? pg_u_bytes<8, 512>(T, V, K) : pg_u_bytes<16, 256>(T, V, K);
    size_t pg = (stream ? 0 : (((size_t)T * V * 4 + 15) & ~(size_t)15)) + (size_t)nutt * ub + 16;
    // reward-to-go: log-sum-exp per frame, chunk counters, the last column / reward-to-go of every sample (int16)
    if (togo) pg += (size_t)Tp * 4 + (size_t)(threads / 32) * 64 * 4 + (size_t)K * (Tp + 16) * 2;
    if (cdf) pg += pg_cdf_bytes(threads);
    return pg;
}

// Word modes: the match tables have max(V, cap) + 1 rows (cap = word_class_cap), and the tail region holds
// max(CDF rows, word-phase scratch): the scratch is used after P1, where the CDF rows are dead.
static size_t pg_role_smem_word(int T, int V, int K, int Lmax, int spl, int threads, bool cdf, int nutt) {
    const int W = spl / 2, cap = word_class_cap(Lmax, V), Vp = V > cap ? V : cap;
    const size_t ub = W == 2 ? pg_u_bytes<2, 512>(T, Vp, K) : W == 4 ? pg_u_bytes<4, 512>(T, Vp, K) :
                      W == 8 ? pg_u_bytes<8, 512>(T, Vp, K) : pg_u_bytes<16, 256>(T, Vp, K);
    const size_t pg = (((size_t)T * V * 4 + 15) & ~(size_t)15) + (size_t)nutt * ub + 16;
    const size_t scratch = word_tail_bytes(T, Lmax, cap, nutt, threads / 32);
    const size_t cdfb = cdf ? pg_cdf_bytes(threads) : 0;
    return pg + (cdfb > scratch ? cdfb : scratch);
}

// What the single-launch kernel can take for this shape.
struct FusedPlan { int spl, threads; bool ctc_ok, gt, pg_ok, stream, bw; };

static FusedPlan fused_plan(int T, int V, int K, int Lmax) {
    FusedPlan pl;
    pl.spl = ctc_spl(Lmax);
    pl.threads = pl.spl >= 32 ? 256 : 512;             // 32 states per lane need the 255-register budget
    pl.ctc_ok = pl.gt = pl.pg_ok = pl.stream = pl.bw = false;
    if (pl.spl == 0 || V > kMaxV || K > kFusedMaxK) return pl;
    // each role keeps its [T][..] tile in shared memory when it fits one SM, else it streams; the streaming PG role
    // is only instantiated next to the streaming CTC role, so a PG role that has to stream makes the CTC role stream
    const bool ctc_tile = ctc_role_smem(T, V, pl.spl, pl.threads, false) <= kFusedSmemLimit;
    const bool ctc_gt = ctc_role_smem(T, V, pl.spl, pl.threads, true) <= kFusedSmemLimit;
    const bool pg_tile = pg_role_smem(T, V, K, pl.spl, pl.threads, false) <= kFusedSmemLimit;
    const bool pg_stream = pg_role_smem(T, V, K, pl.spl, pl.threads, true) <= kFusedSmemLimit;
    if (ctc_tile && (pg_tile || !(ctc_gt && pg_stream))) {
        pl.ctc_ok = true;
        pl.pg_ok = pg_tile;
        // block workers when their (larger) shared-memory layout fits too; PGASR_NO_BW=1 keeps the round-1 workers (A/B)
        static const bool no_bw = getenv("PGASR_NO_BW") != nullptr;
        pl.bw = !no_bw && V <= 32 && pl.spl <= 8 && pl.threads == 512 && ctc_role_smem_bw(T, V, pl.spl) <= kFusedSmemLimit;
    } else if (ctc_gt) {
        pl.ctc_ok = pl.gt = true;
        if (pg_tile) pl.pg_ok = true;
        else if (pg_stream) pl.pg_ok = pl.stream = true;
    }
    return pl;
}

// bit 0: the CTC role fits (tile in shared memory or streamed from the workspace), bit 1: the PG role fits too
int fused_capability(int T, int V, int K, int Lmax) {
    const FusedPlan pl = fused_plan(T, V, K, Lmax);
    return (pl.ctc_ok ? 1 : 0) | (pl.pg_ok ? 2 : 0);
}

bool fused_word_capability(int T, int V, int K, int Lmax) {
    const FusedPlan pl = fused_plan(T, V, K, Lmax);
    return pl.ctc_ok && pl.pg_ok && !pl.stream &&
           pg_role_smem_word(T, V, K, Lmax, pl.spl, pl.threads, false, 1) <= kFusedSmemLimit;
}

// 0 when the fused kernel cannot take this shape at all (the caller then chains the stand-alone kernels)
size_t fused_workspace_bytes(int B, int T, int V, int K, int Lmax) {
    const FusedPlan pl = fused_plan(T, V, K, Lmax);
    if (!pl.ctc_ok) return 0;
    return fused_ws(B, T, V, pl.spl, pl.gt).total;
}

// a.do_pg must be 0 when the PG role does not fit (fused_capability bit 1)
int fused_step(FusedArgs& a, void* workspace, cudaStream_t st, bool throughput, const WordArgs* word,
               const ExploreArgs* explore) {
    const FusedPlan pl = fused_plan(a.T, a.V, a.K, a.Lmax);
    if (!pl.ctc_ok || (a.do_pg && !pl.pg_ok)) return PGASR_ERR_UNSUPPORTED;
    const FusedWs w = fused_ws(a.B, a.T, a.V, pl.spl, pl.gt);
    char* p = reinterpret_cast<char*>(workspace);
    // Consecutive launches on one workspace alternate between its two control blocks: under programmatic dependent
    // launch the CTAs of step n + 1 take their role tickets while step n is still running on its own block.  (Step
    // n + 2 is launched only after every CTA of step n + 1 has passed its grid-dependency wait, i.e. after step n
    // completed and re-armed the block.)  The parity lives on the host, per workspace.
    bool fresh = false;
    const unsigned parity = workspace_parity(workspace, &fresh);
    if (fresh) PGASR_CUDA_TRY(cudaMemsetAsync(workspace, 0, w.ctrl, st));
    a.ctrl = reinterpret_cast<unsigned*>(p) + (size_t)parity * (4 + a.B);
    p += w.ctrl;
    a.lattice = reinterpret_cast<double*>(p);            p += w.lat;
    a.lat_exp = reinterpret_cast<int*>(p);               p += w.exps;
    a.loss_terms = reinterpret_cast<float*>(p);          p += w.terms;
    a.nll_ws = reinterpret_cast<float*>(p);              p += w.nll;
    a.tile_g = pl.gt ? reinterpret_cast<float*>(p) : nullptr;
    size_t smem = !a.do_ctc ? 0 : pl.bw ? ctc_role_smem_bw(a.T, a.V, pl.spl) : ctc_role_smem(a.T, a.V, pl.spl, pl.threads, pl.gt);
    const bool stream = a.do_pg && pl.stream;
    const bool togo = a.do_pg && a.reward_mode == PGASR_REWARD_ED_TO_GO;
    if (togo && stream) return PGASR_ERR_UNSUPPORTED;      // (reward-to-go needs the logits tile in shared memory)
    // The 60 KB logits tile of either role arrives as ONE TMA bulk copy (cp.async.bulk + mbarrier) when the 16-byte
    // alignment rules hold, instead of 3750 16-byte cp.async from 512 threads: measured A/B (same box) softmax-tile phase
    // 7.58 k -> 7.04 k cycles, PG tile load 2.24 k -> 1.67 k, step 38.3 -> 38.0 us.  PGASR_NO_BULK_TILE=1: cp.async path.
    static const bool no_bulk_tile = getenv("PGASR_NO_BULK_TILE") != nullptr;
    a.bulk_tile = !no_bulk_tile && (((size_t)a.T * a.V * 4) & 15) == 0 && ((reinterpret_cast<uintptr_t>(a.logits) & 15) == 0);
    a.cdf_smem = 0;
    a.pg_pair = 0;
    // Steps of a multi-step call run on three streams: a dependent launch then only brings the next step's CTAs onto SMs
    // early, where they sit at the grid-dependency wait (2.4 us per CTA, measured) while another lane's CTAs could run.
    // Measured on one box, 3 lanes: 34.75 / 34.54 us per step with it, 34.23 / 34.27 without (20-step region 36.26 / 35.97
    // against 35.78 / 35.66).  Single steps keep it (back-to-back launches on one stream).  PGASR_PDL_THROUGHPUT=1: keep (A/B)
    static const bool pdl_tp = getenv("PGASR_PDL_THROUGHPUT") != nullptr;
    a.no_pdl = throughput && !pdl_tp;
    if (!a.do_pg) word = nullptr, explore = nullptr;
    if (word) {
        // word modes: the same decisions as below on the word layout; the streaming PG role has no word phase
        if (stream || !fused_word_capability(a.T, a.V, a.K, a.Lmax)) return PGASR_ERR_UNSUPPORTED;
        static const bool no_pair = getenv("PGASR_NO_PAIR") != nullptr;
        if (throughput && !no_pair && a.B >= 2 && a.V <= 32 &&
            pg_role_smem_word(a.T, a.V, a.K, a.Lmax, pl.spl, pl.threads, true, 2) <= kFusedSmemLimit)
            a.pg_pair = 1;
        const int nutt = a.pg_pair ? 2 : 1;
        size_t pg = pg_role_smem_word(a.T, a.V, a.K, a.Lmax, pl.spl, pl.threads, false, nutt);
        if (pg > kFusedSmemLimit) return PGASR_ERR_UNSUPPORTED;
        static const bool no_cdf = getenv("PGASR_NO_CDF_SMEM") != nullptr;
        const size_t pg_cdf = pg_role_smem_word(a.T, a.V, a.K, a.Lmax, pl.spl, pl.threads, true, nutt);
        if (!no_cdf && a.V <= 32 && pg_cdf <= kFusedSmemLimit) {
            a.cdf_smem = 1;
            pg = pg_cdf;
        }
        smem = smem > pg ? smem : pg;
    } else
    if (a.do_pg) {
        // two utterances per PG CTA (their edit distances side by side) when the step is one of several in flight and both
        // blocks fit: measured 39.3 -> 36.5 us per step overlapped, but 58 -> 63 us for a step on its own (the pair CTA
        // outlasts the CTC CTA), hence not for single steps.  PGASR_NO_PAIR=1: never (A/B)
        static const bool no_pair = getenv("PGASR_NO_PAIR") != nullptr;
        if (throughput && !no_pair && !stream && !togo && a.B >= 2 && a.V <= 32 &&
            pg_role_smem(a.T, a.V, a.K, pl.spl, pl.threads, stream, togo, true, 2) <= kFusedSmemLimit)
            a.pg_pair = 1;
        size_t pg = pg_role_smem(a.T, a.V, a.K, pl.spl, pl.threads, stream, togo, false, a.pg_pair ? 2 : 1);
        if (pg > kFusedSmemLimit) return PGASR_ERR_UNSUPPORTED;
        // the CDF rows in shared memory when they fit next to everything else (PGASR_NO_CDF_SMEM=1: register path, A/B)
        static const bool no_cdf = getenv("PGASR_NO_CDF_SMEM") != nullptr;
        if (!no_cdf && !stream && a.V <= 32 && pg + pg_cdf_bytes(pl.threads) <= kFusedSmemLimit) {
            a.cdf_smem = 1;
            pg += pg_cdf_bytes(pl.threads);
        }
        smem = smem > pg ? smem : pg;
    }
    const int mode = pl.bw ? 3 : !pl.gt ? 0 : !stream ? 1 : 2;   // tiles in shared memory | CTC streams | both stream | block workers
    switch (pl.spl) {
        case 4: return launch_fused_spl4(mode, a, smem, st, word, explore);
        case 8: return launch_fused_spl8(mode, a, smem, st, word, explore);
        case 16: return launch_fused_spl16(mode, a, smem, st, word, explore);
        default: return launch_fused_spl32(mode, a, smem, st, word, explore);
    }
}

}  // namespace pgasr
