// CTC alpha-beta lattice walker shared by the standalone CTC kernel (ctc.cu) and the fused step kernel
// (fused.cu).  See ctc.cu for the design notes; spec = DESIGN.md "CTC spec" (SURVEY.md 8a row a8).
#pragma once
#include "pgasr_common.cuh"

namespace pgasr {

constexpr int kCtcChunk = 32;     // frames staged per cp.async batch (staged mode); must be even
constexpr int kCtcChunkWide = 16; // the same for rows too wide for kCtcChunk frames (ctc.cu: V > 196)

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc));
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__host__ __device__ inline int ctc_row_stride(int V) { return (V + 2) & ~1; }   // doubles per probability row (classic kernel)
// floats per probability row of the walker / worker kernel: a multiple of 4 (16-byte cp.async pieces) with at least
// one zero slot after the V classes (what label states beyond the transcript read)
__host__ __device__ inline int ctc_row_stride_f32(int V) { return (V + 4) & ~3; }

constexpr double kCtcMagic = 6755399441055744.0;       // 2^52 + 2^51: low word of (x + magic) = round(x)
constexpr double kCtcFix = 1073741824.0;               // occupancies and probabilities in 2^-30 fixed point
constexpr float kCtcUnfix = 9.31322574615478515625e-10f;

// softmax of one frame into an fp64 row of RS slots; slots V..RS-1 are zero (slot V is what label states
// beyond the transcript read).
__device__ __forceinline__ void softmax_row_f64(const float* __restrict__ z, const float* __restrict__ p_in,
                                                double* __restrict__ o, int V, int RS) {
    if (p_in) {
        for (int v = 0; v < V; ++v) o[v] = (double)p_in[v];
    } else {
        float m = -INFINITY;
        for (int v = 0; v < V; ++v) m = fmaxf(m, z[v]);
        float s = 0.0f;
        for (int v = 0; v < V; ++v) s += __expf(z[v] - m);
        const float inv = 1.0f / s;
        for (int v = 0; v < V; ++v) o[v] = (double)(__expf(z[v] - m) * inv);
    }
    for (int v = V; v < RS; ++v) o[v] = 0.0;
}

template <int SPL>
struct CtcLane {
    double a[SPL];            // alpha-hat / beta-hat of states lane*SPL + j (after the emission)
    double skipm[SPL / 2];    // odd state 2i+1: 1.0 if its two-state transition is legal, else 0.0
    int loff[SPL / 2];        // odd state 2i+1: slot of its class in a probability row (V = the zero slot)
    int E;                    // true value = hat value * 2^E
};

struct GradNorm {
    double invZ0;             // 2^30 / Z0, Z0 = sum_s alpha beta' at the first gradient frame
    int E0;                   // exponent sum (own + other) at that frame
    bool have;                // Z0 measured
    bool dead;                // Z0 == 0: no valid alignment
};

__device__ __forceinline__ double pow2i(int e) {       // 2^e, e clamped to the normal range
    e = max(-1022, min(1023, e));
    return __hiloint2double((1023 + e) << 20, 0);
}

template <int SPL, bool kAlpha>
__device__ __forceinline__ void ctc_lane_init(CtcLane<SPL>& st, const int32_t* __restrict__ lab_u, int L, int V) {
    const int lane = threadIdx.x & 31;
    st.E = 0;
#pragma unroll
    for (int i = 0; i < SPL / 2; ++i) {
        const int li = (lane * SPL) / 2 + i;              // label index of odd state lane*SPL + 2i + 1
        int c = li < L ? lab_u[li] : -1;
        // a label id outside [0,V) reads the zero slot like a state beyond the transcript: its emission probability is
        // 0 in every frame, so the utterance has no valid alignment (nll = +inf, zero gradient) instead of a read of
        // the neighbouring row
        if (c >= V) c = -2;
        st.loff[i] = c >= 0 ? c : V;
        bool legal;
        if (kAlpha) legal = c >= 0 && li >= 1 && lab_u[li - 1] != c;
        else legal = c >= 0 && li + 1 < L && lab_u[li + 1] != c;
        st.skipm[i] = legal ? 1.0 : 0.0;
    }
#pragma unroll
    for (int j = 0; j < SPL; ++j) st.a[j] = 0.0;
}

// One frame.  `row`: the fp64 probability row of frame t (shared memory).  kGrad: second half -- `o` holds the
// other direction's pre-emission sums of this frame (exponent eo); the values of the next frame are prefetched
// into `on` / `eon`.  !kGrad: first half -- this direction's pre-emission sums are stored for the other one.
template <int SPL, bool kAlpha, bool kGrad, bool kAccum>
__device__ __forceinline__ void ctc_step(CtcLane<SPL>& st, GradNorm& gn, int step, int t, bool more, int S, int V,
                                         int blank, const double* row, double* __restrict__ lat_u,
                                         int* __restrict__ exp_u, float grad_scale, float* __restrict__ dlog_u,
                                         int* racc, const double (&o)[SPL], int eo, double (&on)[SPL], int& eon) {
    const int lane = threadIdx.x & 31;
    const bool edge = kAlpha ? lane == 0 : lane == 31;

    if (kGrad && more) {                                  // prefetch the next frame's values (used one step later)
        const int tn = kAlpha ? t + 1 : t - 1;
        const double* lp = lat_u + (size_t)tn * (SPL * 32) + lane;
#pragma unroll
        for (int j = 0; j < SPL; ++j) on[j] = lp[j * 32];
        eon = exp_u[tn];
    }

    // ---- pre-emission sums, in place -----------------------------------------------------------
    if (step == 0) {
#pragma unroll
        for (int j = 0; j < SPL; ++j) {
            const int s = lane * SPL + j;
            const bool on_ = kAlpha ? (s <= 1 && s < S) : (s < S && s >= S - 2);
            st.a[j] = on_ ? 1.0 : 0.0;
        }
    } else if (kAlpha) {
        double h = __shfl_up_sync(kFull, st.a[SPL - 1], 1);
        h = edge ? 0.0 : h;
#pragma unroll
        for (int j = SPL - 1; j >= 2; --j) {
            if (j & 1) st.a[j] = fma(st.skipm[j >> 1], st.a[j - 2], st.a[j] + st.a[j - 1]);
            else st.a[j] = st.a[j] + st.a[j - 1];
        }
        st.a[1] = fma(st.skipm[0], h, st.a[1] + st.a[0]);
        st.a[0] = st.a[0] + h;
    } else {
        double h0 = __shfl_down_sync(kFull, st.a[0], 1);
        double h1 = __shfl_down_sync(kFull, st.a[1], 1);
        h0 = edge ? 0.0 : h0;
        h1 = edge ? 0.0 : h1;
#pragma unroll
        for (int j = 0; j < SPL - 2; ++j) {
            if (j & 1) st.a[j] = fma(st.skipm[j >> 1], st.a[j + 2], st.a[j] + st.a[j + 1]);
            else st.a[j] = st.a[j] + st.a[j + 1];
        }
        st.a[SPL - 2] = st.a[SPL - 2] + st.a[SPL - 1];
        st.a[SPL - 1] = fma(st.skipm[SPL / 2 - 1], h1, st.a[SPL - 1] + h0);
    }

    if (!kGrad) {
        double* lp = lat_u + (size_t)t * (SPL * 32) + lane;
#pragma unroll
        for (int j = 0; j < SPL; ++j) lp[j * 32] = st.a[j];
        if (lane == 0) exp_u[t] = st.E;
    }

    // ---- emission ------------------------------------------------------------------------------
    const double pb = row[blank];
#pragma unroll
    for (int j = 0; j < SPL; ++j) st.a[j] *= (j & 1) ? row[st.loff[j >> 1]] : pb;

    // ---- gradient row of frame t ---------------------------------------------------------------
    if (kGrad) {
        // occupancies in 2^-30 fixed point, with the normalising power of two split between the two factors so that
        // a(s) o(s) cannot underflow fp64 on its own (same scheme as the gradient workers of the fused kernel)
        if (!gn.have) {                                   // first gradient frame: fix the normalisation
            int emax = -1;
#pragma unroll
            for (int j = 0; j < SPL; ++j) {
                const int ax = (__double2hiint(st.a[j]) >> 20) & 0x7ff, ox = (__double2hiint(o[j]) >> 20) & 0x7ff;
                if (ax && ox) emax = max(emax, ax + ox);
            }
            emax = __reduce_max_sync(kFull, emax);
            gn.dead = emax < 0;
            const int ex0 = gn.dead ? 0 : 2046 - emax;
            const double s1 = pow2i(ex0 >> 1), s2 = pow2i(ex0 - (ex0 >> 1));
            double z = 0.0;
#pragma unroll
            for (int j = 0; j < SPL; ++j) z += (st.a[j] * s1) * (o[j] * s2);
            const double Z0 = warp_sum(z);
            gn.have = true;
            gn.dead = gn.dead || !(Z0 > 0.0);
            gn.invZ0 = gn.dead ? 0.0 : kCtcFix / Z0;
            gn.E0 = st.E + eo - ex0;
        }
        const int ex = st.E + eo - gn.E0;
        const int h1 = (ex >> 1) - 15;
        const double s1 = gn.invZ0 * pow2i(h1), s2 = pow2i(ex - h1);
        double w[SPL];
        double zb = 0.0;
#pragma unroll
        for (int j = 0; j < SPL; ++j) {
            w[j] = (st.a[j] * s1) * (o[j] * s2);
            if (!(j & 1)) zb += w[j];
        }
        const int gb = __reduce_add_sync(kFull, __double2loint(zb + kCtcMagic));
#pragma unroll
        for (int j = 1; j < SPL; j += 2) atomicAdd(&racc[st.loff[j >> 1]], __double2loint(w[j] + kCtcMagic));
        __syncwarp();
        float* out = dlog_u + (size_t)t * V;
        for (int v = lane; v < V; v += 32) {
            const int occ = v == blank ? gb : racc[v];
            racc[v] = 0;
            const int pfix = __double2loint(fma(row[v], kCtcFix, kCtcMagic));
            float g = grad_scale * ((float)(pfix - occ) * kCtcUnfix);
            g = gn.dead ? 0.0f : g;
            out[v] = kAccum ? out[v] + g : g;
        }
        __syncwarp();
    }

    // ---- exact power-of-two rescale every 4 steps ------------------------------------------------
    if ((step & 3) == 3) {
        int mx = 0;
#pragma unroll
        for (int j = 0; j < SPL; ++j) mx = max(mx, __double2hiint(st.a[j]));
        mx = __reduce_max_sync(kFull, mx);
        if (mx >= 0x00100000) {
            const int e = (mx >> 20) - 1023;
            const double sc = __hiloint2double((1023 - e) << 20, 0);
            st.E += e;
#pragma unroll
            for (int j = 0; j < SPL; ++j) st.a[j] *= sc;
        }
    }
}

// Steps [step_lo, step_hi) of one direction.  kTile: `probs` is a shared-memory tile [Tb][RS] of the whole
// utterance; else it is the global fp64 workspace and rows are staged through `stage` with cp.async.
template <int SPL, bool kAlpha, bool kGrad, bool kAccum, bool kTile, int kChunk = kCtcChunk>
__device__ __forceinline__ void ctc_frames(CtcLane<SPL>& st, GradNorm& gn, int step_lo, int step_hi, int Tb, int S,
                                           int V, int RS, int blank, const double* probs,
                                           double* __restrict__ lat_u, int* __restrict__ exp_u, float grad_scale,
                                           float* __restrict__ dlog_u, double* stage, int* racc) {
    const int lane = threadIdx.x & 31;
    if (step_lo >= step_hi) return;
    double oa[SPL], ob[SPL];
    int ea = 0, eb = 0;
    if (kGrad) {
        const int t = kAlpha ? step_lo : Tb - 1 - step_lo;
        const double* lp = lat_u + (size_t)t * (SPL * 32) + lane;
#pragma unroll
        for (int j = 0; j < SPL; ++j) oa[j] = lp[j * 32];
        ea = exp_u[t];
    }
    if (kTile) {
        int step = step_lo;
        for (; step + 1 < step_hi; step += 2) {
            const int t = kAlpha ? step : Tb - 1 - step;
            const int t2 = kAlpha ? t + 1 : t - 1;
            ctc_step<SPL, kAlpha, kGrad, kAccum>(st, gn, step, t, true, S, V, blank, probs + (size_t)t * RS, lat_u,
                                                 exp_u, grad_scale, dlog_u, racc, oa, ea, ob, eb);
            ctc_step<SPL, kAlpha, kGrad, kAccum>(st, gn, step + 1, t2, step + 2 < step_hi, S, V, blank,
                                                 probs + (size_t)t2 * RS, lat_u, exp_u, grad_scale, dlog_u, racc, ob,
                                                 eb, oa, ea);
        }
        if (step < step_hi) {
            const int t = kAlpha ? step : Tb - 1 - step;
            ctc_step<SPL, kAlpha, kGrad, kAccum>(st, gn, step, t, false, S, V, blank, probs + (size_t)t * RS, lat_u,
                                                 exp_u, grad_scale, dlog_u, racc, oa, ea, ob, eb);
        }
        return;
    }

    auto issue_chunk = [&](int lo, int buf) {             // steps [lo, hi) -> contiguous frames
        const int hi = min(lo + kChunk, step_hi);
        const int f0 = kAlpha ? lo : Tb - hi;
        const char* src = reinterpret_cast<const char*>(probs + (size_t)f0 * RS);
        char* dst = reinterpret_cast<char*>(stage + (size_t)buf * kChunk * RS);
        const int n16 = (hi - lo) * RS / 2;
        for (int i = lane; i < n16; i += 32) cp_async16(dst + (size_t)i * 16, src + (size_t)i * 16);
        cp_async_commit();
    };
    int buf = 0;
    issue_chunk(step_lo, 0);
    for (int lo = step_lo; lo < step_hi; lo += kChunk, buf ^= 1) {
        const int hi = min(lo + kChunk, step_hi);
        if (hi < step_hi) {
            issue_chunk(hi, buf ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncwarp();
        const double* chunk = stage + (size_t)buf * kChunk * RS;
        int step = lo;
        for (; step + 1 < hi; step += 2) {                // chunks hold an even number of frames except the last
            const int t = kAlpha ? step : Tb - 1 - step;
            const int t2 = kAlpha ? t + 1 : t - 1;
            const double* row = chunk + (size_t)(kAlpha ? step - lo : hi - 1 - step) * RS;
            const double* row2 = kAlpha ? row + RS : row - RS;
            ctc_step<SPL, kAlpha, kGrad, kAccum>(st, gn, step, t, true, S, V, blank, row, lat_u, exp_u, grad_scale,
                                                 dlog_u, racc, oa, ea, ob, eb);
            ctc_step<SPL, kAlpha, kGrad, kAccum>(st, gn, step + 1, t2, step + 2 < step_hi, S, V, blank, row2, lat_u,
                                                 exp_u, grad_scale, dlog_u, racc, ob, eb, oa, ea);
        }
        if (step < hi) {
            const int t = kAlpha ? step : Tb - 1 - step;
            const double* row = chunk + (size_t)(kAlpha ? step - lo : hi - 1 - step) * RS;
            ctc_step<SPL, kAlpha, kGrad, kAccum>(st, gn, step, t, false, S, V, blank, row, lat_u, exp_u, grad_scale,
                                                 dlog_u, racc, oa, ea, ob, eb);
        }
        __syncwarp();
    }
}

// One whole direction: first half (store), mid-point barrier, second half (gradient rows), and for alpha the
// negative log-likelihood.  `mid_barrier()` must synchronise the alpha and the beta warp (and make their global
// stores visible to each other).
template <int SPL, bool kAlpha, bool kAccum, bool kTile, int kChunk, typename Barrier>
__device__ __forceinline__ void ctc_direction(const double* probs, const int32_t* __restrict__ lab_u, int Tb, int L,
                                              int V, int RS, int blank, float grad_scale,
                                              float* __restrict__ nll_out, float* __restrict__ dlog_u,
                                              double* __restrict__ lat_u, int* __restrict__ exp_u, double* stage,
                                              int* racc, Barrier mid_barrier) {
    const int lane = threadIdx.x & 31;
    const int S = 2 * L + 1;
    const int tm = Tb / 2;
    CtcLane<SPL> st;
    ctc_lane_init<SPL, kAlpha>(st, lab_u, L, V);
    for (int v = lane; v <= V; v += 32) racc[v] = 0;
    __syncwarp();
    GradNorm gn;
    gn.have = false; gn.dead = false; gn.invZ0 = 0.0; gn.E0 = 0;
    // steps 0..Tb-1 visit frames 0..Tb-1 (alpha) or Tb-1..0 (beta)
    const int n_first = kAlpha ? tm : Tb - tm;
    ctc_frames<SPL, kAlpha, false, kAccum, kTile, kChunk>(st, gn, 0, n_first, Tb, S, V, RS, blank, probs, lat_u, exp_u,
                                                  grad_scale, dlog_u, stage, racc);
    mid_barrier();
    ctc_frames<SPL, kAlpha, true, kAccum, kTile, kChunk>(st, gn, n_first, Tb, Tb, S, V, RS, blank, probs, lat_u, exp_u,
                                                 grad_scale, dlog_u, stage, racc);
    if (kAlpha) {
        double fin = 0.0;
#pragma unroll
        for (int j = 0; j < SPL; ++j) {
            const int s = lane * SPL + j;
            if (s < S && s >= S - 2) fin += st.a[j];
        }
        fin = warp_sum(fin);
        if (lane == 0)
            *nll_out = fin > 0.0 ? (float)(-(log(fin) + (double)st.E * 0.69314718055994530942)) : INFINITY;
    }
}

inline int ctc_spl(int Lmax) {
    const int S = 2 * Lmax + 1;
    if (S <= 4 * 32) return 4;
    if (S <= 8 * 32) return 8;
    if (S <= 16 * 32) return 16;
    if (S <= 32 * 32) return 32;
    return 0;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace pgasr

// =====================================================================================================
// Split walker (fused kernel, probability tile in shared memory): the two recurrence warps carry ONLY the
// recurrence; in their second half they hand each frame's post-emission values to gradient worker warps through
// a double-buffered shared-memory ring, in batches of kBatch frames guarded by named barriers (bar.arrive /
// bar.sync: waiting warps sleep in hardware, and the only memory fence is the barrier itself, once per batch --
// a per-frame release store costs a MEMBAR that drains the 8 pending STS, ~300 cycles, measured).  The workers
// turn the values into gradient rows; frames are independent there, so G workers per direction work on G frames
// at once.  A warp issues in order, so taking the gradient's latencies (lattice loads, redux, shared atomics,
// row stores) out of the recurrence warp is what shortens the frame time.
// =====================================================================================================
namespace pgasr {

// frames per hand-off batch (two batches in flight per direction); 32 states per lane make a frame 8 KB, so the
// rings of that variant hold fewer frames
// (up to 8 states per lane: 14 frames, so each of the 7 workers owns TWO frames of a batch and runs them side by
// side -- a worker frame is ~170 dependent instructions at ~7 cycles each, measured; one frame at a time left the
// workers, not the walkers, as the bound of the second half)
template <int SPL>
constexpr int kBatchOf = SPL >= 32 ? 4 : SPL >= 16 ? 7 : 14;
inline int batch_of(int spl) { return spl >= 32 ? 4 : spl >= 16 ? 7 : 14; }
template <int SPL>
constexpr int kWalkUnroll = kBatchOf<SPL> % 7 == 0 ? 7 : kBatchOf<SPL>;   // frames per unrolled group of the walker

template <int SPL, int NB = kBatchOf<SPL>>
struct GradRing {
    double* slots;                // [2 * NB][SPL*16]: the LABEL states of a frame ([SPL/4][32 lanes] double2)
    int* eslot;                   // [2 * kBatch] exponent of the published values
    double* norm;                 // [2]: 2^30 / Z0, then (int) E0 and (int) dead -- written by the walker, see ctc_walk_publish_norm
    int bar_full;                 // named barrier ids: bar_full + k, bar_empty + k for buffer k in {0, 1}
    int bar_empty;
    const int* cls_off;           // [V + 1] CSR over classes: label positions li with lab[li] == v
    const int* cls_pos;           // [L]
    bool dbg;                     // PGASR_TIMING: this CTA records phase stamps
};

// Label positions grouped by class (counting sort), built once per utterance by one warp.  The gradient workers
// sum the label occupancies of a class by walking its list: shared-memory atomics cost ~2 cycles per lane on
// the one atomic unit of the SM (measured: 8 worker warps x 4 ATOMS per frame made the atomics the bottleneck).
__device__ __forceinline__ void ctc_build_class_lists(const int32_t* __restrict__ lab_u, int L, int V, int* cls_off,
                                                      int* cls_pos, int* scratch /* V ints */) {
    const int lane = threadIdx.x & 31;
    for (int v = lane; v <= V; v += 32) cls_off[v] = 0;
    for (int v = lane; v < V; v += 32) scratch[v] = 0;
    __syncwarp();
    for (int li = lane; li < L; li += 32) {
        const int c = lab_u[li];
        if (c >= 0 && c < V) atomicAdd(&cls_off[c + 1], 1);
    }
    __syncwarp();
    if (lane == 0)
        for (int v = 0; v < V; ++v) cls_off[v + 1] += cls_off[v];
    __syncwarp();
    for (int li = lane; li < L; li += 32) {
        const int c = lab_u[li];
        if (c >= 0 && c < V) cls_pos[cls_off[c] + atomicAdd(&scratch[c], 1)] = li;
    }
    __syncwarp();
}

template <int SPL, int NB = kBatchOf<SPL>>
__host__ __device__ inline size_t grad_ring_bytes() {
    // slots + exponents + the normalisation block
    return (size_t)2 * NB * SPL * 16 * 8 + (((size_t)2 * NB * 4 + 15) & ~(size_t)15) + 16;
}

template <int SPL, int NB = kBatchOf<SPL>>
__device__ __forceinline__ GradRing<SPL, NB> grad_ring_carve(unsigned char* p, int bar_base) {   // p 16-byte aligned
    GradRing<SPL, NB> r;
    r.slots = reinterpret_cast<double*>(p);
    r.eslot = reinterpret_cast<int*>(p + (size_t)2 * NB * SPL * 16 * 8);
    r.norm = reinterpret_cast<double*>(p + (size_t)2 * NB * SPL * 16 * 8 + (((size_t)2 * NB * 4 + 15) & ~(size_t)15));
    r.bar_full = bar_base;
    r.bar_empty = bar_base + 2;
    r.dbg = false;
    return r;
}

__device__ __forceinline__ void named_bar_sync(int id, int count) {
    asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int count) {
    asm volatile("bar.arrive %0, %1;\n" ::"r"(id), "r"(count) : "memory");
}

// pre-emission sums in place; h0 (and h1 for beta) are the halo values fetched from the neighbour lane
template <int SPL, bool kAlpha>
__device__ __forceinline__ void ctc_presum(CtcLane<SPL>& st, double h0, double h1) {
    if (kAlpha) {
#pragma unroll
        for (int j = SPL - 1; j >= 2; --j) {
            if (j & 1) st.a[j] = fma(st.skipm[j >> 1], st.a[j - 2], st.a[j] + st.a[j - 1]);
            else st.a[j] = st.a[j] + st.a[j - 1];
        }
        st.a[1] = fma(st.skipm[0], h0, st.a[1] + st.a[0]);
        st.a[0] = st.a[0] + h0;
    } else {
#pragma unroll
        for (int j = 0; j < SPL - 2; ++j) {
            if (j & 1) st.a[j] = fma(st.skipm[j >> 1], st.a[j + 2], st.a[j] + st.a[j + 1]);
            else st.a[j] = st.a[j] + st.a[j + 1];
        }
        st.a[SPL - 2] = st.a[SPL - 2] + st.a[SPL - 1];
        st.a[SPL - 1] = fma(st.skipm[SPL / 2 - 1], h1, st.a[SPL - 1] + h0);
    }
}

// (not volatile: the probability tile is read-only while the walkers run, the scheduler may move these loads)
__device__ __forceinline__ double lds_f64(unsigned addr) {
    double v;
    asm("ld.shared.f64 %0, [%1];\n" : "=d"(v) : "r"(addr));
    return v;
}

// L2 residency hints for the half-lattice (written once, read once ~30 us later, then dead; the workspace is reused
// every step): stores ask L2 to keep the lines (evict_last), the single read demotes them (evict_first).  Without
// the hints ~11 MB of the 52 MB lattice were written back to DRAM per step before they were read (ncu).
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ void st_lattice(double2* ptr, double x, double y, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;\n" ::"l"(ptr), "d"(x), "d"(y), "l"(pol) : "memory");
}
// 32-byte flavours (sm_100: STG/LDG.256): a lane's four label values of a frame in one access.  Lattice rows with
// 8 or more states per lane are laid out [SPL/8][32 lanes][2 double2] so that they apply; SPL 4 keeps [32 lanes] double2.
__device__ __forceinline__ void st_lattice4(double2* ptr, double x, double y, double z, double w, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.v4.f64 [%0], {%1, %2, %3, %4}, %5;\n" ::"l"(ptr), "d"(x), "d"(y), "d"(z), "d"(w), "l"(pol) : "memory");
}
__device__ __forceinline__ void ld_lattice4(const double2* ptr, unsigned long long pol, double2& lo, double2& hi) {
    asm volatile("ld.global.cg.L2::cache_hint.v4.f64 {%0, %1, %2, %3}, [%4], %5;\n"
                 : "=d"(lo.x), "=d"(lo.y), "=d"(hi.x), "=d"(hi.y) : "l"(ptr), "l"(pol));
}
template <int SPL>
__device__ __forceinline__ int lat_lane_off(int lane) { return SPL >= 8 ? 2 * lane : lane; }   // in double2 units
__device__ __forceinline__ double2 ld_lattice(const double2* ptr, unsigned long long pol) {
    double2 v;
    asm volatile("ld.global.cg.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;\n" : "=d"(v.x), "=d"(v.y) : "l"(ptr), "l"(pol));
    return v;
}

// volatile flavour for the streaming ring: ordered after the cp.async waits (volatile asm keeps its order)
__device__ __forceinline__ double lds_f64_v(unsigned addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];\n" : "=d"(v) : "r"(addr) : "memory");
    return v;
}
// The probability tile of the walker / worker kernel is fp32 (the softmax is computed in fp32, so nothing is lost):
// a lane's 4-byte read of "its" class within a 128-byte row never collides on a bank with the other lanes' reads
// (8-byte reads of a 256-byte row were 2-3 wavefronts each), and the tile takes half the shared memory.
__device__ __forceinline__ float lds_f32_v(unsigned addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];\n" : "=f"(v) : "r"(addr) : "memory");
    return v;
}

// Recurrence warp of one direction over the whole utterance (tile mode).  G: workers of this direction.
// Lattice / ring layout per frame: [SPL/2][32 lanes] double2, so each lane moves 16 bytes per access and a warp
// access is one coalesced 512 B line.  The frame body is branch free and unrolled four times; every frame uses
// the same code (frame 0 starts from a virtual "previous" vector that the recurrence maps onto the CTC start
// states), so the only branches left are the loop, the rescale test and the batch barriers.
template <int SPL, bool kAlpha>
struct CtcWalk {
    CtcLane<SPL> st;
    double h0, h1;                // halo value for the frame about to be computed (h1: unused, kept zero)
    double skip_prev;             // beta: skip factor of the PREVIOUS lane's last label state into this lane's state 1
    double pb_n, p_n[SPL / 2];    // probabilities of the frame about to be computed   (both sets were loaded TWO frames
    float pb_m, p_m[SPL / 2];     // probabilities of the frame after it                ahead of their use; widened to
                                  //                                                    fp64 one frame after the load)
    unsigned pa_b, pa[SPL / 2];   // running shared-memory addresses of this lane's probabilities: two frames on
    int rstride;
    bool edge;
    bool act;                     // this lane holds at least one state < S (lanes beyond never touch the lattice)
    unsigned long long l2pol;     // L2 cache policy of the lattice stores
    // global-tile mode (long utterances): the probability rows stream from global memory through a 32-row ring
    unsigned ring_base, ring_mask;        // shared-memory address of the ring (aligned to its size), size - 1
    const float* tile_g;                  // row 0 of this utterance's fp32 tile in global memory (guard rows around it)
    int gstep, row_next, row_dir, row_lo, row_hi, RS, RSR;
};

constexpr int kPRows = 32;        // rows of the streaming ring
constexpr int kPGroup = 8;        // rows per cp.async group

// rows [first, first + kPGroup) in walking order -> ring slots (row & 31); one 16-byte cp.async per lane and piece
template <int SPL, bool kAlpha>
__device__ __forceinline__ void ctc_walk_issue_group(CtcWalk<SPL, kAlpha>& w, unsigned ring_generic_lo) {
    (void)ring_generic_lo;
    const int lane = threadIdx.x & 31;
    const int per_row = w.RS / 4;                         // 16-byte pieces per row
    for (int i = lane; i < kPGroup * per_row; i += 32) {
        const int r = i / per_row, c = i - r * per_row;
        int row = w.row_next + w.row_dir * r;
        row = min(max(row, w.row_lo), w.row_hi);          // guard rows: loaded, never used
        const unsigned dst = w.ring_base + (unsigned)(((row & (kPRows - 1)) * w.RSR + 4 * c) * 4);
        const float* src = w.tile_g + (ptrdiff_t)row * w.RS + 4 * c;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(src));
    }
    cp_async_commit();
    w.row_next += w.row_dir * kPGroup;
}


// One value crosses each lane boundary per frame.  alpha: the neighbour's last state (it feeds both of this lane's
// first two states).  beta: the lane's last (label) state needs the next lane's first TWO states, b(s+1) and
// skip * b(s+2); the next lane knows that skip factor (skip_prev) and sends the sum, so it is one shuffle as well.
template <int SPL, bool kAlpha>
__device__ __forceinline__ void ctc_walk_halo(CtcWalk<SPL, kAlpha>& w) {
    if (kAlpha) {
        w.h0 = __shfl_up_sync(kFull, w.st.a[SPL - 1], 1);
    } else {
        w.h0 = __shfl_down_sync(kFull, fma(w.skip_prev, w.st.a[1], w.st.a[0]), 1);
    }
    w.h0 = w.edge ? 0.0 : w.h0;
    w.h1 = 0.0;
}

template <int SPL, bool kAlpha>
__device__ __forceinline__ void ctc_walk_rescale(CtcWalk<SPL, kAlpha>& w) {
    int mx = 0;
#pragma unroll
    for (int j = 0; j < SPL; ++j) mx = max(mx, __double2hiint(w.st.a[j]));
    mx = __reduce_max_sync(kFull, mx);
    if (mx >= 0x00100000) {
        const int e = (mx >> 20) - 1023;
        const double sc = __hiloint2double((1023 - e) << 20, 0);
        w.st.E += e;
#pragma unroll
        for (int j = 0; j < SPL; ++j) w.st.a[j] *= sc;
        w.h0 *= sc;
        w.h1 *= sc;
    }
}

// kFirst: store the pre-emission sums to the lattice (dst = global), else the post-emission values to the ring
// (dst = shared).  dst advances by `dstride` double2 per frame; edst (exponent per frame) by estride ints.
// Only the LABEL states (odd j) are published: the blank column of the gradient follows from sum_s gamma_t(s) = 1
// (in 2^-30 fixed point: 2^30 minus the label occupancies), so neither the lattice nor the ring carries the blank
// states.  kMid: the direction's last first-half frame -- its blank states are stored too (second half of the
// lattice row), because the other walker measures Z0 = sum_s alpha beta' over ALL states there, once.
template <int SPL, bool kAlpha, bool kFirst, bool kGT = false, bool kMid = false>
__device__ __forceinline__ void ctc_walk_frame(CtcWalk<SPL, kAlpha>& w, double2*& dst, ptrdiff_t dstride, int*& edst,
                                               int estride, bool lane0) {
    if (kGT) {
        // every 8 frames: the two groups about to be read are complete, the slot of the group just left is refilled
        if ((w.gstep & (kPGroup - 1)) == 0) {
            cp_async_wait<1>();
            __syncwarp();
            ctc_walk_issue_group<SPL, kAlpha>(w, 0u);
        }
        ++w.gstep;
    }
    // The loads are volatile asm issued two frames before their values are multiplied in: measured on the bare frame
    // loop (tools/walk_probe.cu) plain loads cost 127 cycles per frame wherever they are written (ptxas sinks them next
    // to their consumers), volatile loads one frame ahead 94, two frames ahead 79; the arithmetic alone is 52.
    double p[SPL / 2];
    const double pb = w.pb_n;
#pragma unroll
    for (int i = 0; i < SPL / 2; ++i) p[i] = w.p_n[i];
    w.pb_n = (double)w.pb_m;
#pragma unroll
    for (int i = 0; i < SPL / 2; ++i) w.p_n[i] = (double)w.p_m[i];
    w.pb_m = lds_f32_v(w.pa_b);
#pragma unroll
    for (int i = 0; i < SPL / 2; ++i) w.p_m[i] = lds_f32_v(w.pa[i]);
    if (kGT) {
        w.pa_b = w.ring_base | ((w.pa_b + w.rstride) & w.ring_mask);
#pragma unroll
        for (int i = 0; i < SPL / 2; ++i) w.pa[i] = w.ring_base | ((w.pa[i] + w.rstride) & w.ring_mask);
    } else {
        w.pa_b += w.rstride;
#pragma unroll
        for (int i = 0; i < SPL / 2; ++i) w.pa[i] += w.rstride;
    }
    ctc_presum<SPL, kAlpha>(w.st, w.h0, w.h1);
#ifndef EXP_NO_LATSTORE
    if (kFirst) {
        if (w.act) {
            if constexpr (SPL >= 8) {
#pragma unroll
                for (int j2 = 0; j2 < SPL / 8; ++j2)
                    st_lattice4(dst + j2 * 64, w.st.a[8 * j2 + 1], w.st.a[8 * j2 + 3], w.st.a[8 * j2 + 5], w.st.a[8 * j2 + 7], w.l2pol);
                if (kMid) {
#pragma unroll
                    for (int j2 = 0; j2 < SPL / 8; ++j2)
                        st_lattice4(dst + (SPL / 4) * 32 + j2 * 64, w.st.a[8 * j2], w.st.a[8 * j2 + 2], w.st.a[8 * j2 + 4],
                                    w.st.a[8 * j2 + 6], w.l2pol);
                }
            } else {
                st_lattice(dst, w.st.a[1], w.st.a[3], w.l2pol);
                if (kMid) st_lattice(dst + 32, w.st.a[0], w.st.a[2], w.l2pol);
            }
        }
    }
#endif
#pragma unroll
    for (int j = 0; j < SPL; ++j) w.st.a[j] *= (j & 1) ? p[j >> 1] : pb;
    ctc_walk_halo<SPL, kAlpha>(w);
    if (!kFirst) {
#pragma unroll
        for (int jj = 0; jj < SPL / 4; ++jj) dst[jj * 32] = make_double2(w.st.a[4 * jj + 1], w.st.a[4 * jj + 3]);
    }
    if (lane0) *edst = w.st.E;
    dst += dstride;
    edst += estride;
}

// The walker's first second-half frame: Z0 = sum over ALL states of (own post-emission value) x (the other direction's
// pre-emission sum), the one place the blank states of the other direction are needed (it stored them at its last
// first-half frame, kMid).  The product a(s) o(s) can underflow fp64 on its own when alpha and beta peak far apart,
// so the normalising power of two is split between the two factors (same scheme as the workers' occupancies).
// Result -> shared memory: norm[0] = 2^30 / Z0 (0 when no alignment exists), then int E0, int dead.
template <int SPL, bool kAlpha>
__device__ __forceinline__ void ctc_walk_publish_norm(const CtcWalk<SPL, kAlpha>& w, const double* lat_row,
                                                      const int* exp_p, double* norm) {
    const int lane = threadIdx.x & 31;
    const double2* lp = reinterpret_cast<const double2*>(lat_row) + lat_lane_off<SPL>(lane);
    double o[SPL];
#pragma unroll
    for (int jj = 0; jj < SPL / 4; ++jj) {
        double2 lab = make_double2(0.0, 0.0), blk = make_double2(0.0, 0.0);
        if (w.act) {
            const int off = SPL >= 8 ? (jj >> 1) * 64 + (jj & 1) : jj * 32;   // (see st_lattice4)
            lab = __ldcg(lp + off);
            blk = __ldcg(lp + (SPL / 4) * 32 + off);
        }
        o[4 * jj] = blk.x; o[4 * jj + 1] = lab.x; o[4 * jj + 2] = blk.y; o[4 * jj + 3] = lab.y;
    }
    const int eo = __ldcg(exp_p);
    int emax = -1;                                        // largest exponent-field sum of a product with both factors > 0
#pragma unroll
    for (int j = 0; j < SPL; ++j) {
        const int ax = (__double2hiint(w.st.a[j]) >> 20) & 0x7ff, ox = (__double2hiint(o[j]) >> 20) & 0x7ff;
        if (ax && ox) emax = max(emax, ax + ox);
    }
    emax = __reduce_max_sync(kFull, emax);
    bool dead = emax < 0;
    const int ex0 = dead ? 0 : 2046 - emax;               // brings the largest product to about 2^0
    const double s1 = pow2i(ex0 >> 1), s2 = pow2i(ex0 - (ex0 >> 1));
    double z = 0.0;
#pragma unroll
    for (int j = 0; j < SPL; ++j) z += (w.st.a[j] * s1) * (o[j] * s2);
    const double Z0 = warp_sum(z);
    dead = dead || !(Z0 > 0.0);
    if (lane == 0) {
        norm[0] = dead ? 0.0 : kCtcFix / Z0;
        reinterpret_cast<int*>(norm)[2] = w.st.E + eo - ex0;
        reinterpret_cast<int*>(norm)[3] = dead ? 1 : 0;
    }
}

// kGT: `tile` is row 0 of the utterance's tile in GLOBAL memory ([T] rows of RS doubles between two guard rows),
// `pring` the 32-row shared-memory ring of this walker (aligned to its size, row stride RSR doubles).
template <int SPL, int G, bool kAlpha, bool kGT = false, int NB = kBatchOf<SPL>, typename Barrier>
__device__ __forceinline__ void ctc_walk_tile(const float* tile, const int32_t* __restrict__ lab_u, int Tb, int L,
                                              int V, int RS, int blank, float* __restrict__ nll_out,
                                              double* __restrict__ lat_u, int* __restrict__ exp_u,
                                              GradRing<SPL, NB> ring, Barrier mid_barrier, float* pring = nullptr,
                                              int RSR = 0, int T = 0) {
    constexpr int kGroup = 32 * (1 + G);                  // this warp + its workers
    // frames per unrolled group of the second half: TWO.  Unrolling the whole batch (8 frames, ~3 KB of code) measured
    // 3 % slower per step than groups of 4 or 2 (36.3 / 35.3 / 35.2 us): six code streams share the SM's instruction
    // caches and the walkers showed instruction-fetch stalls (18 % of their second-half samples).
#ifdef PGASR_WALK_UNROLL
    constexpr int kWU = NB % PGASR_WALK_UNROLL == 0 ? PGASR_WALK_UNROLL : NB;
#else
    constexpr int kWU = NB % 2 == 0 ? 2 : NB % 7 == 0 ? 7 : NB;
#endif
    const int lane = threadIdx.x & 31;
    const bool lane0 = lane == 0;
    const int S = 2 * L + 1;
    const int tm = Tb / 2;
    const int n_first = kAlpha ? tm : Tb - tm;
    const int n2 = Tb - n_first;
    CtcWalk<SPL, kAlpha> w;
    ctc_lane_init<SPL, kAlpha>(w.st, lab_u, L, V);
    w.edge = kAlpha ? lane == 0 : lane == 31;
    w.act = lane * SPL < S;
    w.l2pol = l2_policy_evict_last();
    w.skip_prev = 0.0;
    if (!kAlpha && lane > 0) {
        const int li = (lane * SPL) / 2 - 1;              // last label of the previous lane; this lane's state 1 is label li + 1
        if (li + 1 < L && lab_u[li + 1] != lab_u[li]) w.skip_prev = 1.0;
    }
    const bool dbg = ring.dbg && lane == 0;
    PGASR_STAMP(dbg, kAlpha ? 10 : 14);

    const int t0 = kAlpha ? 0 : Tb - 1;
    unsigned row0;
    if (kGT) {
        w.tile_g = tile; w.RS = RS; w.RSR = RSR;
        w.ring_base = (unsigned)__cvta_generic_to_shared(pring);
        w.ring_mask = (unsigned)(kPRows * RSR * 4 - 1);
        w.rstride = kAlpha ? RSR * 4 : -RSR * 4;
        w.row_dir = kAlpha ? 1 : -1;
        w.row_lo = -1; w.row_hi = T;
        w.row_next = t0;
        w.gstep = 0;
        // three groups in flight, the first two complete before the first frame
        ctc_walk_issue_group<SPL, kAlpha>(w, 0u);
        ctc_walk_issue_group<SPL, kAlpha>(w, 0u);
        ctc_walk_issue_group<SPL, kAlpha>(w, 0u);
        cp_async_wait<1>();
        __syncwarp();
        row0 = w.ring_base + (unsigned)((t0 & (kPRows - 1)) * RSR * 4);
    } else {
        w.rstride = kAlpha ? RS * 4 : -RS * 4;
        row0 = (unsigned)__cvta_generic_to_shared(tile) + (unsigned)(t0 * RS * 4);
    }
    // every tile load below takes its address from this opaque copy, so none of them (plain asm, free to be
    // scheduled) can be moved above this point, i.e. above the barrier that published the tile
    asm volatile("mov.u32 %0, %0;\n" : "+r"(row0) : : "memory");
    {
        // frame 0 and frame 1 now, the running addresses point at frame 2
        const unsigned row1 = kGT ? (w.ring_base | ((row0 + w.rstride) & w.ring_mask)) : row0 + w.rstride;
        const unsigned row2 = kGT ? (w.ring_base | ((row1 + w.rstride) & w.ring_mask)) : row1 + w.rstride;
        // (in ring mode row0 is ring_base + slot * row bytes: the column offsets below stay inside the row)
        w.pb_n = (double)lds_f32_v(row0 + (unsigned)(blank * 4));
        w.pb_m = lds_f32_v(row1 + (unsigned)(blank * 4));
        w.pa_b = row2 + (unsigned)(blank * 4);
#pragma unroll
        for (int i = 0; i < SPL / 2; ++i) {
            w.p_n[i] = (double)lds_f32_v(row0 + (unsigned)(w.st.loff[i] * 4));
            w.p_m[i] = lds_f32_v(row1 + (unsigned)(w.st.loff[i] * 4));
            w.pa[i] = row2 + (unsigned)(w.st.loff[i] * 4);
        }
    }
    // virtual vector before the first frame: the recurrence turns it into the CTC start (alpha: states 0,1;
    // beta: states S-1,S-2) -- see DESIGN.md "CTC spec"
#pragma unroll
    for (int j = 0; j < SPL; ++j) {
        const int s = lane * SPL + j;
        w.st.a[j] = (kAlpha ? s == 0 : s == S - 1) ? 1.0 : 0.0;
    }
    w.h0 = w.h1 = 0.0;
    ctc_walk_halo<SPL, kAlpha>(w);

    // ---- first half: pre-emission sums go to the lattice for the other direction -----------------
    {
        double2* lp = reinterpret_cast<double2*>(lat_u + (size_t)t0 * (SPL * 32)) + lat_lane_off<SPL>(lane);
        const ptrdiff_t lstride = kAlpha ? (SPL / 2) * 32 : -(SPL / 2) * 32;
        int* ep = exp_u + t0;
        const int estride = kAlpha ? 1 : -1;
        int step = 0;
        for (; step + 4 <= n_first - 1; step += 4) {
#pragma unroll
            for (int u = 0; u < 4; ++u) ctc_walk_frame<SPL, kAlpha, true, kGT>(w, lp, lstride, ep, estride, lane0);
            if (step & 4) ctc_walk_rescale<SPL, kAlpha>(w);
        }
        for (; step < n_first - 1; ++step) ctc_walk_frame<SPL, kAlpha, true, kGT>(w, lp, lstride, ep, estride, lane0);
        if (n_first > 0) ctc_walk_frame<SPL, kAlpha, true, kGT, true>(w, lp, lstride, ep, estride, lane0);   // + blank states
        ctc_walk_rescale<SPL, kAlpha>(w);
    }
    PGASR_STAMP(dbg, kAlpha ? 11 : 15);
    mid_barrier();
    PGASR_STAMP(dbg, kAlpha ? 12 : 16);

    // ---- second half: post-emission values go to the workers in batches of kBatch frames -----------
    for (int q = 0; q < n2; q += NB) {
        const int buf = (q / NB) & 1;
        if (q >= 2 * NB) named_bar_sync(ring.bar_empty + buf, kGroup);
        double2* sp = reinterpret_cast<double2*>(ring.slots + (size_t)(buf * NB) * (SPL * 16)) + lane;
        int* ep = ring.eslot + buf * NB;
        const int nfr = min(NB, n2 - q);
        if (q == 0) {
            // first frame of the second half: measure Z0 against the other direction's full row and publish the
            // normalisation for the workers (they read it after the first bar_full)
            ctc_walk_frame<SPL, kAlpha, false, kGT>(w, sp, (SPL / 4) * 32, ep, 1, lane0);
            const int tf = kAlpha ? n_first : Tb - 1 - n_first;
            ctc_walk_publish_norm<SPL, kAlpha>(w, lat_u + (size_t)tf * (SPL * 32), exp_u + tf, ring.norm);
            for (int u = 1; u < nfr; ++u) ctc_walk_frame<SPL, kAlpha, false, kGT>(w, sp, (SPL / 4) * 32, ep, 1, lane0);
        } else if (nfr == NB) {
            for (int u0 = 0; u0 < NB; u0 += kWU) {
#pragma unroll
                for (int u = 0; u < kWU; ++u) ctc_walk_frame<SPL, kAlpha, false, kGT>(w, sp, (SPL / 4) * 32, ep, 1, lane0);
            }
        } else {
            for (int u = 0; u < nfr; ++u) ctc_walk_frame<SPL, kAlpha, false, kGT>(w, sp, (SPL / 4) * 32, ep, 1, lane0);
        }
        named_bar_arrive(ring.bar_full + buf, kGroup);
        ctc_walk_rescale<SPL, kAlpha>(w);
    }
    PGASR_STAMP(dbg, kAlpha ? 13 : 17);
    if (kGT) cp_async_wait<0>();                          // nothing of this warp may still be landing in the ring

    if (kAlpha) {
        double fin = 0.0;
#pragma unroll
        for (int j = 0; j < SPL; ++j) {
            const int s = lane * SPL + j;
            if (s < S && s >= S - 2) fin += w.st.a[j];
        }
        fin = warp_sum(fin);
        if (lane == 0)
            *nll_out = fin > 0.0 ? (float)(-(log(fin) + (double)w.st.E * 0.69314718055994530942)) : INFINITY;
    }
}

// Gradient worker g of one direction: frames q with q % G == g of that direction's second half.  The frames a
// worker owns in one batch are processed side by side (separate accumulators) so their latencies overlap.
// The other direction's lattice rows come from L2 (~600 cycles): the loads for the NEXT batch are issued right
// after phase A has consumed the current ones, into the same registers, so they fly during phase B and the
// batch barrier.  (A two-register-set ping-pong issued the next loads BEFORE the current ones were consumed;
// both sets then shared hardware scoreboards and every batch waited out the full L2 latency -- measured:
// 48k of the 113k second-half cycles.)
template <int SPL, int G, bool kAlpha>
struct CtcWorker {
    static constexpr int kPer = (kBatchOf<SPL> + G - 1) / G;     // frames of a batch per worker (worker g: frames g, g+G, ..)
    double2 o[kPer][SPL / 4];     // the other direction's label states of the frame
    int eo[kPer];
    double prow[kPer];            // global-tile mode: p_t(lane) of the frame, fetched with the lattice row
    unsigned long long l2pol;     // L2 cache policy of the lattice loads (evict_first: the row is dead after this read)
    int tF[kPer], qF[kPer];       // frame and second-half index of the NEXT fetch of each owned frame (they advance by
                                  // a batch per fetch: no per-batch index arithmetic)
    int tB[kPer], qB[kPer];       // the same for the NEXT phase B (it runs one fetch behind)
    const double2* lat2;          // the utterance's lattice as double2, this lane's offset folded in
};

template <int SPL, int G, bool kAlpha>
__device__ __forceinline__ void ctc_worker_fetch_init(CtcWorker<SPL, G, kAlpha>& wk, int g, int n_first, int Tb,
                                                      const double* __restrict__ lat_u) {
    const int lane = threadIdx.x & 31;
    wk.lat2 = reinterpret_cast<const double2*>(lat_u) + lat_lane_off<SPL>(lane);
#pragma unroll
    for (int r = 0; r < CtcWorker<SPL, G, kAlpha>::kPer; ++r) {
        const int q = g + r * G;
        wk.qF[r] = wk.qB[r] = q < kBatchOf<SPL> ? q : (1 << 28);     // (a frame this worker never owns: always out of range)
        wk.tF[r] = wk.tB[r] = kAlpha ? n_first + q : Tb - 1 - n_first - q;
    }
}

template <int SPL, int G, bool kAlpha, bool kGT = false>
__device__ __forceinline__ void ctc_worker_fetch(CtcWorker<SPL, G, kAlpha>& wk, int n2, int S,
                                                 const int* __restrict__ exp_u, const float* tile = nullptr,
                                                 int RS = 0) {
    const int lane = threadIdx.x & 31;
    const bool act = lane * SPL < S;                      // the other direction never stored the lanes beyond S
    const unsigned long long pol = wk.l2pol;
#pragma unroll
    for (int r = 0; r < CtcWorker<SPL, G, kAlpha>::kPer; ++r) {
        const int t = wk.tF[r];
        const bool valid = wk.qF[r] < n2;                 // (beyond the utterance: nothing is loaded, zeros are used)
        const double2* lp = wk.lat2 + (size_t)t * (SPL * 16);
#ifdef EXP_NO_LATTICE
#pragma unroll
        for (int jj = 0; jj < SPL / 4; ++jj) wk.o[r][jj] = make_double2(1.0 + lane, 0.5);
        wk.eo[r] = 0; (void)lp;
#else
        if constexpr (SPL >= 8) {
#pragma unroll
            for (int j2 = 0; j2 < SPL / 8; ++j2) {
                wk.o[r][2 * j2] = wk.o[r][2 * j2 + 1] = make_double2(0.0, 0.0);
                if (act && valid) ld_lattice4(lp + j2 * 64, pol, wk.o[r][2 * j2], wk.o[r][2 * j2 + 1]);
            }
        } else {
            wk.o[r][0] = (act && valid) ? ld_lattice(lp, pol) : make_double2(0.0, 0.0);
        }
        wk.eo[r] = valid ? __ldcg(exp_u + t) : 0;
        if (kGT) wk.prow[r] = valid ? (double)__ldcg(tile + (size_t)t * RS + min(lane, RS - 1)) : 0.0;
#endif
        wk.qF[r] += kBatchOf<SPL>;
        wk.tF[r] += kAlpha ? kBatchOf<SPL> : -kBatchOf<SPL>;
    }
}

struct WorkerNorm { double invZ0; int E0; bool dead, have; long long tA, tB, tWait, tBusy; };

constexpr int kClsRegs = 12;      // label positions of this lane's class held in registers

// phase A: occupancies of every owned frame of batch nb; label states go to gam[frame][label index] and the
// blank total to gb[] (2^-30 fixed point).  When every worker owns the same number of frames per batch (kUncond)
// the frames are computed unconditionally, in ONE basic block, so that their dependent chains interleave; a frame
// beyond the end of the utterance then reads a stale ring slot and its results are never stored.
template <int SPL, int G, bool kAlpha>
__device__ __forceinline__ void ctc_worker_phase_a(const CtcWorker<SPL, G, kAlpha>& wk, WorkerNorm& nm, int nb, int g,
                                                   int n2, const GradRing<SPL>& ring, int* gam,
                                                   int (&gb)[(kBatchOf<SPL> + G - 1) / G]) {
    constexpr int kPer = CtcWorker<SPL, G, kAlpha>::kPer;
    constexpr int kGam = 16 * SPL;                        // ints per frame: SPL/2 label occupancies per lane
    constexpr bool kUncond = kBatchOf<SPL> % G == 0;
    const int lane = threadIdx.x & 31;
    // Occupancy of state s in 2^-30 fixed point = a(s) o(s) c with c = invZ0 2^(E + eo - E0).  The product
    // a(s) o(s) alone can underflow fp64 although both factors and the final value are in range (alpha and
    // beta peak far apart when T >> L with diffuse posteriors), so the power of two is split between the
    // two factors before they are multiplied: (a 2^h1) (o invZ0 2^h2), h1 + h2 = E + eo - E0.
    // Only the label states are handled; the blank column is 2^30 minus their sum (sum_s gamma_t(s) = 1).
    if constexpr (kUncond) {
        // stage by stage over the frames (loads, products, reductions, stores): the shared-memory stores of one
        // frame would otherwise fence the loads of the next (the compiler cannot tell the ring from gam)
        double2 av[kPer][SPL / 4];
        int E[kPer], wi[kPer][SPL / 2], ls[kPer];
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            const int slot = (nb & 1) * kBatchOf<SPL> + g + r * G;
            const double2* sp = reinterpret_cast<const double2*>(ring.slots + (size_t)slot * (SPL * 16)) + lane;
#pragma unroll
            for (int jj = 0; jj < SPL / 4; ++jj) av[r][jj] = sp[jj * 32];
            E[r] = ring.eslot[slot];
        }
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            const int ex = E[r] + wk.eo[r] - nm.E0;
            const int h1 = (ex >> 1) - 15;                // invZ0 <= 2^30 rides on the smaller half
            const double s1 = nm.invZ0 * pow2i(h1), s2 = pow2i(ex - h1);
            ls[r] = 0;
#pragma unroll
            for (int jj = 0; jj < SPL / 4; ++jj) {
                wi[r][2 * jj] = __double2loint((av[r][jj].x * s1) * (wk.o[r][jj].x * s2) + kCtcMagic);
                wi[r][2 * jj + 1] = __double2loint((av[r][jj].y * s1) * (wk.o[r][jj].y * s2) + kCtcMagic);
                ls[r] += wi[r][2 * jj] + wi[r][2 * jj + 1];
            }
        }
#pragma unroll
        for (int r = 0; r < kPer; ++r) gb[r] = (1 << 30) - __reduce_add_sync(kFull, ls[r]);
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            if constexpr (SPL >= 8) {
                int4* gr = reinterpret_cast<int4*>(gam + r * kGam) + lane * (SPL / 8);
#pragma unroll
                for (int i = 0; i < SPL / 8; ++i) gr[i] = make_int4(wi[r][4 * i], wi[r][4 * i + 1], wi[r][4 * i + 2], wi[r][4 * i + 3]);
            } else {
                reinterpret_cast<int2*>(gam + r * kGam)[lane] = make_int2(wi[r][0], wi[r][1]);
            }
        }
        (void)n2;
    } else {
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            const int qi = g + r * G;                     // frame of the batch
            gb[r] = 0;
            if (qi < kBatchOf<SPL> && nb * kBatchOf<SPL> + qi < n2) {
                const int slot = (nb & 1) * kBatchOf<SPL> + qi;
                const double2* sp = reinterpret_cast<const double2*>(ring.slots + (size_t)slot * (SPL * 16)) + lane;
                double2 av[SPL / 4];
#pragma unroll
                for (int jj = 0; jj < SPL / 4; ++jj) av[jj] = sp[jj * 32];
                const int E = ring.eslot[slot];
                const int ex = E + wk.eo[r] - nm.E0;
                const int h1 = (ex >> 1) - 15;
                const double s1 = nm.invZ0 * pow2i(h1), s2 = pow2i(ex - h1);
                int wi[SPL / 2];
                int ls = 0;
#pragma unroll
                for (int jj = 0; jj < SPL / 4; ++jj) {
                    wi[2 * jj] = __double2loint((av[jj].x * s1) * (wk.o[r][jj].x * s2) + kCtcMagic);
                    wi[2 * jj + 1] = __double2loint((av[jj].y * s1) * (wk.o[r][jj].y * s2) + kCtcMagic);
                    ls += wi[2 * jj] + wi[2 * jj + 1];
                }
                gb[r] = (1 << 30) - __reduce_add_sync(kFull, ls);
                if constexpr (SPL >= 8) {
                    int4* gr = reinterpret_cast<int4*>(gam + r * kGam) + lane * (SPL / 8);
#pragma unroll
                    for (int i = 0; i < SPL / 8; ++i) gr[i] = make_int4(wi[4 * i], wi[4 * i + 1], wi[4 * i + 2], wi[4 * i + 3]);
                } else {
                    reinterpret_cast<int2*>(gam + r * kGam)[lane] = make_int2(wi[0], wi[1]);
                }
            }
        }
    }
    __syncwarp();
}

// phase B: gradient rows; lane v sums the label occupancies of class v.  cpos[] entries beyond the class's
// count point at label slot 16*SPL-1, whose state 32*SPL-1 lies beyond S for every transcript (always 0), so the
// gather is branch free; cmax (warp uniform) bounds the rare tail of classes with more than kClsRegs labels.
template <int SPL, int G, bool kAlpha, bool kGT = false>
__device__ __forceinline__ void ctc_worker_phase_b(CtcWorker<SPL, G, kAlpha>& wk, const double (&prow)[(kBatchOf<SPL> + G - 1) / G],
                                                   const WorkerNorm& nm, int nb, int g, int n_first, int n2, int Tb,
                                                   const float* tile, int V, int RS, int blank, float grad_scale,
                                                   float* __restrict__ dlog_u, const GradRing<SPL>& ring,
                                                   const int* gam, const int (&gb)[(kBatchOf<SPL> + G - 1) / G], int ccnt, int cmax,
                                                   const int (&cpos)[kClsRegs]) {
    constexpr int kPer = (kBatchOf<SPL> + G - 1) / G;
    constexpr int kGam = 16 * SPL;
    constexpr bool kUncond = kBatchOf<SPL> % G == 0;
    const int lane = threadIdx.x & 31;
    if (V <= 32) {
        // the frames of this worker side by side: gathers, then the rare tail, then the rows
        int occ[kPer];
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            const int* gr = gam + r * kGam;
            int o1 = 0, o2 = 0;
#ifndef EXP_NO_PHASEB
#pragma unroll
            for (int i = 0; i < kClsRegs; i += 2) {
                if (i < cmax) {                            // warp uniform: no class of this transcript is longer
                    o1 += gr[cpos[i]];
                    o2 += gr[cpos[i + 1]];
                }
            }
#endif
            occ[r] = o1 + o2;
        }
#ifndef EXP_NO_PHASEB
        if (cmax > kClsRegs) {
#pragma unroll
            for (int r = 0; r < kPer; ++r)
                for (int i = kClsRegs; i < cmax; ++i)
                    occ[r] += i < ccnt ? gam[r * kGam + ring.cls_pos[ring.cls_off[lane] + i]] : 0;
        }
#endif
        const int lane_c = min(lane, RS - 1);
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            const bool valid = wk.qB[r] < n2;
            const int t = wk.tB[r];
            if (kUncond || valid) {
                const int oc = lane == blank ? gb[r] : occ[r];
                const double pv = kGT ? prow[r] : (valid ? (double)tile[t * RS + lane_c] : 0.0);
                const int pfix = __double2loint(fma(pv, kCtcFix, kCtcMagic));
                const float gval = nm.dead ? 0.0f : grad_scale * ((float)(pfix - oc) * kCtcUnfix);
                if (lane < V && valid) dlog_u[(size_t)t * V + lane] = gval;
            }
        }
    } else {
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            if (wk.qB[r] < n2) {
                const int t = wk.tB[r];
                const float* row = tile + (size_t)t * RS;
                float* out = dlog_u + (size_t)t * V;
                const int* gr = gam + r * kGam;
                for (int v = lane; v < V; v += 32) {
                    int occ = 0;
                    for (int i = ring.cls_off[v]; i < ring.cls_off[v + 1]; ++i) occ += gr[ring.cls_pos[i]];
                    if (v == blank) occ = gb[r];
                    const int pfix = __double2loint(fma((double)row[v], kCtcFix, kCtcMagic));
                    const float gval = grad_scale * ((float)(pfix - occ) * kCtcUnfix);
                    out[v] = nm.dead ? 0.0f : gval;
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
        wk.qB[r] += kBatchOf<SPL>;
        wk.tB[r] += kAlpha ? kBatchOf<SPL> : -kBatchOf<SPL>;
    }
    (void)nb; (void)g; (void)n_first; (void)Tb;
    __syncwarp();
}

template <int SPL, int G, bool kAlpha, bool kGT = false, typename Barrier>
__device__ __forceinline__ void ctc_grad_worker(int g, const float* tile, const int32_t* __restrict__ lab_u, int Tb,
                                                int L, int V, int RS, int blank, float grad_scale,
                                                float* __restrict__ dlog_u, const double* __restrict__ lat_u,
                                                const int* __restrict__ exp_u, GradRing<SPL> ring, int* gam,
                                                Barrier mid_barrier) {
    constexpr int kGroup = 32 * (1 + G);
    constexpr int kPer = (kBatchOf<SPL> + G - 1) / G;
    const int lane = threadIdx.x & 31;
    const int tm = Tb / 2;
    const int n_first = kAlpha ? tm : Tb - tm;
    const int n2 = Tb - n_first;
    // label positions of class `lane` (the classes beyond 32, if any, are walked from shared memory)
    int ccnt = 0, cpos[kClsRegs];
    if (lane < V) ccnt = ring.cls_off[lane + 1] - ring.cls_off[lane];
#pragma unroll
    for (int i = 0; i < kClsRegs; ++i) cpos[i] = (i < ccnt) ? ring.cls_pos[ring.cls_off[min(lane, V - 1)] + i] : 16 * SPL - 1;
    const int cmax = __reduce_max_sync(kFull, ccnt);
    (void)lab_u;
    mid_barrier();                                        // the other direction's half-lattice is complete
    WorkerNorm nm;
    nm.invZ0 = 0.0; nm.E0 = 0; nm.dead = false; nm.have = false;
    nm.tA = nm.tB = nm.tWait = nm.tBusy = 0;
    const int nbatch = (n2 + kBatchOf<SPL> - 1) / kBatchOf<SPL>;
    CtcWorker<SPL, G, kAlpha> wk;
    wk.l2pol = l2_policy_evict_first();
    int gb[kPer];
    const int S = 2 * L + 1;
    double prow[kPer];
    ctc_worker_fetch_init<SPL, G, kAlpha>(wk, g, n_first, Tb, lat_u);
    if (nbatch > 0) ctc_worker_fetch<SPL, G, kAlpha, kGT>(wk, n2, S, exp_u, tile, RS);
    for (int nb = 0; nb < nbatch; ++nb) {
        const int buf = nb & 1;
#ifdef PGASR_TIMING
        const long long w0 = clock64();
#endif
        named_bar_sync(ring.bar_full + buf, kGroup);
#ifdef PGASR_TIMING
        const long long w1 = clock64();
        nm.tWait += w1 - w0;
#endif
        if (nb == 0) {                                    // the walker measured Z0 on its first second-half frame
            nm.invZ0 = ring.norm[0];
            nm.E0 = reinterpret_cast<const int*>(ring.norm)[2];
            nm.dead = reinterpret_cast<const int*>(ring.norm)[3] != 0;
            nm.have = true;
        }
#ifndef EXP_NO_WORKER
        ctc_worker_phase_a<SPL, G, kAlpha>(wk, nm, nb, g, n2, ring, gam, gb);
#ifdef PGASR_TIMING
        const long long w2 = clock64();
        nm.tA += w2 - w1;
#endif
        if (kGT) {                                        // keep this batch's p_t(lane) before the registers are refilled
#pragma unroll
            for (int r = 0; r < kPer; ++r) prow[r] = wk.prow[r];
        }
        if (nb + 1 < nbatch) ctc_worker_fetch<SPL, G, kAlpha, kGT>(wk, n2, S, exp_u, tile, RS);
        ctc_worker_phase_b<SPL, G, kAlpha, kGT>(wk, prow, nm, nb, g, n_first, n2, Tb, tile, V, RS, blank, grad_scale,
                                                dlog_u, ring, gam, gb, ccnt, cmax, cpos);
#ifdef PGASR_TIMING
        nm.tB += clock64() - w2;
#endif
#endif
#ifdef PGASR_TIMING
        nm.tBusy += clock64() - w1;
#endif
        if (nb + 2 < nbatch) named_bar_arrive(ring.bar_empty + buf, kGroup);   // buffer may be overwritten
    }
#ifdef PGASR_TIMING
    if (ring.dbg && lane == 0 && g == 0) {
        g_dbg[kAlpha ? 20 : 22] = nm.tWait;
        g_dbg[kAlpha ? 21 : 23] = nm.tBusy;
        g_dbg[kAlpha ? 25 : 29] = nm.tA;
        g_dbg[kAlpha ? 26 : 30] = nm.tB;
    }
#endif
}

}  // namespace pgasr

// =====================================================================================================
// Block workers (round 2; up to 8 states per lane, probability tile in shared memory).
//
// What bounded the second half was the gradient ROW, not the lattice: with a lane per class a row is a gather of the
// class's label occupancies from arbitrary positions -- 8 to 12 bank-conflicting LDS per frame and warp, 27 of the ~40
// shared-memory wavefronts a frame cost -- and the SM's one shared-memory pipe was ~60 % busy, which is also what
// slowed the walkers from 130 to 180 cycles per frame.  Here the rows of a BLOCK of up to 32 consecutive frames are
// formed together with a lane per FRAME:
//   * A-workers (GA per direction) do what phase A did -- occupancy of every label state of a frame, 2^-30 fixed
//     point -- and store it TRANSPOSED into the block's matrix gam[label][frame slot] (bank = slot ^ (label / labels
//     per lane): conflict free for the A-worker's stores, one per label of the lane, and for the reads below).
//   * B-workers (GB per direction, block b belongs to B-worker b % GB and to matrix buffer b % GB) walk the
//     transcript's labels in CLASS ORDER (one warp-uniform list per utterance) and add gam[label][lane's frame] into
//     a per-class accumulator: one conflict-free LDS per label for 30 frames at once, no gather, no tail loop.  At
//     the end of a class the lane turns (p - occupancy) into the gradient entry and stores it in place of p_t(v) in
//     the probability tile (row stride odd: conflict free; nobody reads a row's probabilities after its frame has
//     been handed to the workers), and when the block is done its rows leave as one contiguous, coalesced copy.
// Per frame this is ~20 shared-memory wavefronts instead of ~40 and ~75 warp instructions instead of ~115.
// Hand-offs: walker -> A-workers through the ring as before (batches of 2 GA frames, named barriers); A-workers ->
// B-worker one named barrier per block (gam_full); B-worker -> A-workers a release/acquire counter in shared memory
// per matrix buffer (the B-worker is a block period ahead, so the wait is normally a single load).
// =====================================================================================================
#ifndef PGASR_BW_GA
#define PGASR_BW_GA 4
#endif
namespace pgasr {

// Warp w of the CTA runs on scheduler partition w % 4.  The walkers are warps 0 and 1; the occupancy (A) workers -- the
// fp64 work -- sit on partitions 2 and 3 only (warps 2,3,6,7,10,11,14,15: four per direction), the row (B) workers
// share the walkers' partitions (integer and shared-memory work), and the two warps left over idle at the barriers.
constexpr int kBwGA = PGASR_BW_GA;          // A-workers per direction (4: partitions 2/3 only; 5: the spare warp too)
constexpr int kBwGB = 2;          // B-workers per direction (= matrix buffers per direction), at most 3
constexpr int kBwNB = 2 * kBwGA;  // frames per ring batch: two per A-worker
constexpr int kBwBB = 32 / kBwNB; // ring batches per block
constexpr int kBwBlk = kBwBB * kBwNB;   // frames per block (<= 32: a lane per frame)

template <int SPL>
__host__ __device__ inline size_t bw_gam_bytes() { return (size_t)kBwGB * (16 * SPL) * 32 * sizeof(int); }   // per direction
__host__ __device__ inline size_t bw_stage_bytes() { return (size_t)kBwBlk * 32 * sizeof(float); }     // per B-worker, V <= 32

__device__ __forceinline__ int lds_acquire_s32(const int* p) {
    int v;
    asm volatile("ld.acquire.cta.shared.s32 %0, [%1];\n" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void sts_release_s32(int* p, int v) {
    asm volatile("st.release.cta.shared.s32 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}
// mbarrier (shared memory, CTA scope): the row worker's "matrix buffer consumed" signal.  A waiter sleeps in hardware
// inside try_wait (a spin on ld.acquire kept five warps per direction hammering the shared-memory pipe the row worker
// needs: it ran 4x slower than alone).
__device__ __forceinline__ void mbar_init(unsigned long long* b, int count) {
    asm volatile("mbarrier.init.shared.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* b) {
    asm volatile("mbarrier.arrive.release.cta.shared.b64 _, [%0];\n" ::"r"((unsigned)__cvta_generic_to_shared(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* b, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.acquire.cta.shared.b64 p, [%0], %1, 0x989680;\n"
        "@p bra DONE_%=;\n"
        "nanosleep.u32 256;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(b)), "r"(parity) : "memory");
}
__device__ __forceinline__ int lds_s32(unsigned addr) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1];\n" : "=r"(v) : "r"(addr) : "memory");
    return v;
}

// The transcript's label positions in class order (from the CSR lists of ctc_build_class_lists), as shared-memory
// ADDRESSES of the label's row in one matrix buffer with the frame-slot swizzle folded in:
// entry = base + row * 128 + (row / LPL) * 4, so that the address of (label, frame slot f) is entry ^ 4 f (base is
// 128-byte aligned: the xor stays inside the row).  One list per matrix buffer (2 directions x kBwGB buffers).
// The row worker walks the list in groups of 8, three groups per loop trip and two groups of prefetch, replacing every
// entry's occupancy by the running sum up to it; the list is padded to 3 ceil(groups / 3) + 2 groups with entries
// pointing at the spare row 16 SPL - 1 (its state lies beyond S for every transcript this variant takes; what lands
// there is never read back).
// info[0] = loop trips, info[4 + v] (16-byte aligned, 32 entries) = the LAST entry of the classes 0..v, i.e. where the
// running sum up to and including class v ends up (kBwNone when no label has a class <= v): a class's total is the
// difference of two of them.  One warp; V <= 32.
constexpr unsigned kBwNone = 0xffffffffu;
constexpr int kBwListWords = 256;     // per copy: the list (at most 23 groups) and, from word 192, info[36]
constexpr int kBwInfoAt = 192;
template <int SPL>
__device__ __forceinline__ void bw_build_list(const int* cls_off, const int* cls_pos, int V, unsigned* elist, int* info,
                                              unsigned base) {
    constexpr int LPL = SPL / 2, kRows = 16 * SPL;
    const int lane = threadIdx.x & 31;
    const int cnt = lane < V ? cls_off[lane + 1] - cls_off[lane] : 0;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int x = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += x;
    }
    const int start = incl - cnt;
    const int total = __shfl_sync(kFull, incl, 31);
    const unsigned ez = base + (unsigned)((kRows - 1) * 128 + ((kRows - 1) / LPL) * 4);
    if (lane < V) {
        const int src = cls_off[lane];
        for (int i = 0; i < cnt; ++i) {
            const int li = cls_pos[src + i];
            elist[start + i] = base + (unsigned)(li * 128 + (li / LPL) * 4);
        }
    }
    const int trips = ((total + 7) / 8 + 2) / 3;
    for (int i = total + lane; i < 8 * (3 * trips + 2); i += 32) elist[i] = ez;
    __syncwarp();
    info[4 + lane] = incl > 0 ? (int)elist[incl - 1] : (int)kBwNone;   // (lanes >= V repeat the last class: never used)
    if (lane == 0) info[0] = trips;
    __syncwarp();
}

// A-worker g (0 .. GA-1) of one direction: frames g and g + GA of every ring batch.
// (the direction is a run-time argument: both directions then execute the SAME instructions, which halves the
// helpers' footprint in the instruction cache -- the walkers showed instruction-fetch stalls next to six code streams)
template <int SPL, typename Barrier>
__device__ __forceinline__ void ctc_aworker(bool kAlpha, int g, int Tb, int L, const double* __restrict__ lat_u,
                                            const int* __restrict__ exp_u, GradRing<SPL, kBwNB> ring, int* gam,
                                            unsigned long long* done, int bar_gfull, Barrier mid_barrier) {
    constexpr int GA = kBwGA, GB = kBwGB, NB = kBwNB, kBB = kBwBB, LPL = SPL / 2, kRows = 16 * SPL;
    constexpr int kGroup = 32 * (1 + GA);
    const int lane = threadIdx.x & 31;
    const int tm = Tb / 2;
    const int n_first = kAlpha ? tm : Tb - tm;
    const int n2 = Tb - n_first;
    const int S = 2 * L + 1;
    const bool act = lane * SPL < S;                      // the other direction never stored the lanes beyond S
    mid_barrier();                                        // the other direction's half-lattice is complete
    const int nbatch = (n2 + NB - 1) / NB;
    const unsigned long long pol = l2_policy_evict_first();
    const double2* lat2 = reinterpret_cast<const double2*>(lat_u) + lat_lane_off<SPL>(lane);
    // The other direction's rows come from L2 through running pointers that stop at the worker's last frame (a frame
    // beyond the utterance re-reads that row; its results are never used).  Lanes beyond the transcript read memory the
    // other walker never wrote: whatever comes out lands in matrix rows no class list points at -- except the all-zero
    // row 16 SPL - 1 (lane 31's last label), which is forced to zero below.
    double2 o[2][SPL / 4];
    int eo[2], left[2];
    const char* lp[2];
    const int* ep[2];
    const ptrdiff_t lstep = (ptrdiff_t)(kAlpha ? NB : -NB) * (SPL * 16) * (ptrdiff_t)sizeof(double2);
    const int estep = kAlpha ? NB : -NB;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int q = g + r * GA;
        left[r] = q < n2 ? (n2 - 1 - q) / NB : 0;         // advances left
        const int qc = min(q, max(n2 - 1, 0));
        const int t = kAlpha ? n_first + qc : Tb - 1 - n_first - qc;
        lp[r] = reinterpret_cast<const char*>(lat2 + (size_t)t * (SPL * 16));
        ep[r] = exp_u + t;
    }
    auto fetch = [&]() {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const double2* l2p = reinterpret_cast<const double2*>(lp[r]);
            if constexpr (SPL >= 8) {
#pragma unroll
                for (int j2 = 0; j2 < SPL / 8; ++j2) ld_lattice4(l2p + j2 * 64, pol, o[r][2 * j2], o[r][2 * j2 + 1]);
            } else {
                o[r][0] = ld_lattice(l2p, pol);
            }
            eo[r] = __ldcg(ep[r]);
            const bool more = left[r] > 0;
            --left[r];
            lp[r] += more ? lstep : 0;
            ep[r] += more ? estep : 0;
        }
    };
    const bool zlast = lane == 31 && !act;
    if (nbatch > 0) fetch();
    double invZ0 = 0.0;
    int E0 = 0;
    // this lane's rows of a matrix buffer start at label LPL * lane; the frame slot is XORed with the lane
    int* const grow = gam + (LPL * lane) * 32;
    int blk = 0, bi = 0;                                  // block of this batch, batch within the block
#ifdef PGASR_TIMING
    long long tWait = 0, tSpin = 0, tBusy = 0;
#endif
    for (int nb = 0; nb < nbatch; ++nb) {
        const int buf = nb & 1;
#ifdef PGASR_TIMING
        const long long c0 = clock64();
#endif
        named_bar_sync(ring.bar_full + buf, kGroup);
#ifdef PGASR_TIMING
        const long long c1 = clock64();
        tWait += c1 - c0;
#endif
        if (nb == 0) {                                    // the walker measured Z0 on its first second-half frame
            invZ0 = ring.norm[0];
            E0 = reinterpret_cast<const int*>(ring.norm)[2];
        }
        const int gbuf = blk % GB;
        if (bi == 0 && blk >= GB) {                       // the buffer's previous block must have been consumed
            mbar_wait(done + gbuf, (unsigned)(blk / GB - 1) & 1u);   // phase k of the barrier = the buffer's k-th use consumed
        }
#ifdef PGASR_TIMING
        const long long c2 = clock64();
        tSpin += c2 - c1;
#endif
        double2 av[2][SPL / 4];
        int E[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int slot = buf * NB + g + r * GA;
            const double2* sp = reinterpret_cast<const double2*>(ring.slots + (size_t)slot * (SPL * 16)) + lane;
#pragma unroll
            for (int jj = 0; jj < SPL / 4; ++jj) av[r][jj] = sp[jj * 32];
            E[r] = ring.eslot[slot];
        }
        // the ring buffer is free as soon as this warp's values have LANDED in registers -- hand it back to the walker now
        // rather than after the products (the barrier id takes a never-true dependency on the loaded words, which is
        // what makes the warp wait for them)
        if (nb + 2 < nbatch) {
            int chk = E[0] & E[1];
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int jj = 0; jj < SPL / 4; ++jj) chk &= __double2hiint(av[r][jj].x) & __double2hiint(av[r][jj].y);
            named_bar_arrive(ring.bar_empty + buf + (chk == -1 ? 16 : 0), kGroup);   // (values are finite and >= 0: never -1)
        }
#ifndef EXP_A_IDLE
        int wi[2][LPL];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            // occupancy = a(s) o(s) invZ0 2^(E + eo - E0) in 2^-30 fixed point, the power of two split between the two
            // factors so that the product cannot underflow on its own (see ctc_worker_phase_a)
            const int ex = E[r] + eo[r] - E0;
            const int h1 = (ex >> 1) - 15;
            const double s1 = invZ0 * pow2i(h1), s2 = pow2i(ex - h1);
#pragma unroll
            for (int jj = 0; jj < SPL / 4; ++jj) {
                wi[r][2 * jj] = __double2loint((av[r][jj].x * s1) * (o[r][jj].x * s2) + kCtcMagic);
                wi[r][2 * jj + 1] = __double2loint((av[r][jj].y * s1) * (o[r][jj].y * s2) + kCtcMagic);
            }
            wi[r][LPL - 1] = zlast ? 0 : wi[r][LPL - 1];
        }
        int* const gb = grow + gbuf * (kRows * 32);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int f = bi * NB + g + r * GA;           // frame slot within the block
            int* const gp = gb + (f ^ lane);
#pragma unroll
#ifndef EXP_A_NOSTORE
            for (int j = 0; j < LPL; ++j) gp[j * 32] = wi[r][j];
#endif
        }
#else
        asm volatile("" :: "d"(o[0][0].x), "d"(o[1][0].y), "r"(eo[0] + eo[1]), "d"(invZ0), "r"(E0), "r"(zlast ? 1 : 0), "l"(grow), "r"(gbuf) : "memory");
#endif
        if (nb + 1 < nbatch) fetch();
        const bool last_of_block = bi == kBB - 1 || nb == nbatch - 1;
        if (last_of_block) {
            named_bar_arrive(bar_gfull + gbuf, 32 * (GA + 1));                 // the block's matrix is complete
            ++blk;
            bi = 0;
        } else {
            ++bi;
        }
#ifdef PGASR_TIMING
        tBusy += clock64() - c2;
#endif
    }
#ifdef PGASR_TIMING
    if (ring.dbg && lane == 0 && g == 0) {
        g_dbg[kAlpha ? 40 : 44] = tWait;
        g_dbg[kAlpha ? 41 : 45] = tSpin;
        g_dbg[kAlpha ? 42 : 46] = tBusy;
    }
#endif
}

// B-worker j (0 .. GB-1) of one direction: blocks j, j + GB, ...  Lane f = frame slot f of the block.
// The class-ordered label list is walked in groups of 8 entries, software pipelined (list words two groups ahead,
// occupancies one group ahead, three register sets rotating through a loop body of three groups): uniform 16-byte
// list loads, eight independent conflict-free occupancy loads, a running integer sum.  Where an entry carries the
// class-end flag the class's total (a difference of two running sums) is stored over that entry's occupancy -- one
// predicated store, no branch.  Afterwards the classes are independent: total and probability in, gradient entry out.
// (A first version branched to an in-loop "emit" at every class end: 4 control instructions per entry and a chain
// through the emit; 9.4k cycles per block.)
template <int SPL, typename Barrier>
__device__ __forceinline__ void ctc_bworker(bool kAlpha, int j, const float* tile, int RS, int Tb, int V, int blank,
                                            float grad_scale, float* __restrict__ dlog_u, const double* norm,
                                            unsigned long long* done, int bar_gfull, const unsigned* elist,
                                            const int* info, float* stage, Barrier mid_barrier, bool dbg = false) {
    constexpr int GA = kBwGA, GB = kBwGB, kBlk = kBwBlk;
    const int lane = threadIdx.x & 31;
    const int tm = Tb / 2;
    const int n_first = kAlpha ? tm : Tb - tm;
    const int n2 = Tb - n_first;
    mid_barrier();
    const int nblocks = (n2 + kBlk - 1) / kBlk;
    const unsigned fx = (unsigned)lane << 2;              // the frame-slot swizzle: address = entry ^ 4 lane
    const unsigned el_s = (unsigned)__cvta_generic_to_shared(elist);
    const unsigned cl_s = (unsigned)__cvta_generic_to_shared(info + 4);
    const unsigned st_s = (unsigned)__cvta_generic_to_shared(stage);
    const float gs30 = grad_scale * kCtcUnfix;
    const int ntrips = info[0];
    bool dead = false;
    int it = 0;
#ifdef PGASR_TIMING
    long long tWait = 0, tRows = 0, tCopy = 0, tPre = 0, tLoop = 0, nBlk = 0;
#endif
    for (int blk = j; blk < nblocks; blk += GB, ++it) {
#ifdef PGASR_TIMING
        const long long c0 = clock64();
#endif
        named_bar_sync(bar_gfull + j, 32 * (GA + 1));
#ifdef PGASR_TIMING
        const long long c1 = clock64();
        tWait += c1 - c0;
#endif
        if (it == 0) dead = reinterpret_cast<const int*>(norm)[3] != 0;
        const int q0 = blk * kBlk;
        const int nf = min(kBlk, n2 - q0);
        const bool valid = lane < nf;
        const int q = q0 + min(lane, nf - 1);
        const int t = kAlpha ? n_first + q : Tb - 1 - n_first - q;
        const int tlo = kAlpha ? n_first + q0 : Tb - 1 - n_first - q0 - (nf - 1);
        const unsigned prow = (unsigned)__cvta_generic_to_shared(tile + (size_t)t * RS);
        const float gmul = dead ? 0.0f : gs30;
        // ---- running integer sums over the class-ordered list: every entry's occupancy is replaced by the sum up to
        // and including it (load, add, store back to the same address: four instructions per label for 32 frames; a
        // version that stored only at class ends needed a compare, a select and two predicated instructions per entry)
#ifdef EXP_B_IDLE
        (void)prow; (void)gmul; (void)valid; (void)fx; (void)el_s; (void)cl_s; (void)ntrips;
        if (it > 0 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
        __syncwarp();
#else
        int acc = 0;
        unsigned E[3][8];
        int X[3][8];
        auto ld_list = [&](unsigned (&e)[8], unsigned addr) {
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];\n" : "=r"(e[0]), "=r"(e[1]), "=r"(e[2]), "=r"(e[3]) : "r"(addr));
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];\n" : "=r"(e[4]), "=r"(e[5]), "=r"(e[6]), "=r"(e[7]) : "r"(addr + 16u));
        };
        auto ld_occ = [&](int (&x)[8], unsigned (&e)[8]) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                e[u] ^= fx;                               // (this lane's slot of the entry's row)
                asm volatile("ld.shared.s32 %0, [%1];\n" : "=r"(x[u]) : "r"(e[u]));
            }
        };
        auto sum8 = [&](const int (&x)[8], const unsigned (&e)[8]) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                acc += x[u];
                asm volatile("st.shared.s32 [%0], %1;\n" ::"r"(e[u]), "r"(acc));
            }
        };
        ld_list(E[0], el_s);
        ld_list(E[1], el_s + 32u);
        ld_occ(X[0], E[0]);
#ifdef PGASR_TIMING
        asm volatile("" :: "r"(X[0][7]) : "memory");
        const long long ca = clock64();
#endif
        unsigned la = el_s + 64u;
        for (int g = 0; g < ntrips; ++g, la += 96u) {
            ld_occ(X[1], E[1]); ld_list(E[2], la);       sum8(X[0], E[0]);
            ld_occ(X[2], E[2]); ld_list(E[0], la + 32u); sum8(X[1], E[1]);
            ld_occ(X[0], E[0]); ld_list(E[1], la + 64u); sum8(X[2], E[2]);
        }
#ifdef PGASR_TIMING
        asm volatile("" :: "r"(acc) : "memory");
        const long long cb = clock64();
        tPre += ca - c1; tLoop += cb - ca; ++nBlk;
#endif
        // ---- the block's gradient rows, packed [frame][V] in this worker's staging buffer (= their layout in dlogits),
        // eight classes at a time: all loads of a batch first (the compiler keeps asm memory operations in source order,
        // so the batching has to be written out).  The previous block's bulk copy must have READ the buffer first.
        if (it > 0 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
        __syncwarp();
        const int row = kAlpha ? lane : nf - 1 - lane;   // this lane's frame within the block's rows, ascending in t
        const unsigned srow = st_s + 4u * (unsigned)(max(row, 0) * V);
        const unsigned zslot = (elist[8 * (3 * ntrips + 2) - 1]) ^ fx;   // (a padding entry: any valid address)
        int tot;                                          // sum of all label occupancies: where the last class ends
        {
            unsigned ce;
            asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(ce) : "r"(cl_s + 4u * (unsigned)(V - 1)));
            asm volatile("ld.shared.s32 %0, [%1];\n" : "=r"(tot) : "r"(ce == kBwNone ? zslot : ce ^ fx));
            tot = ce == kBwNone ? 0 : tot;
        }
        int prev = 0;                                     // running sum at the end of the previous class
        for (int v0 = 0; v0 < V; v0 += 8) {
            unsigned cl[8];
            ld_list(cl, cl_s + 4u * (unsigned)v0);
            const unsigned pa = prow + 4u * (unsigned)v0;
            int ps[8];
            float pv[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                asm volatile("ld.shared.s32 %0, [%1];\n" : "=r"(ps[u]) : "r"(cl[u] == kBwNone ? zslot : cl[u] ^ fx));
#pragma unroll
            for (int u = 0; u < 8; ++u)                   // (beyond V: the row's zero slot, in bounds)
                asm volatile("ld.shared.f32 %0, [%1];\n" : "=f"(pv[u]) : "r"(pa + 4u * (unsigned)min(u, V - v0)));
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int upto = cl[u] == kBwNone ? 0 : ps[u];
                const int oc = v0 + u == blank ? (1 << 30) - tot : upto - prev;   // the blank column: sum_s gamma_t(s) = 1
                prev = upto;
                const int pfix = __float2int_rn(pv[u] * (float)kCtcFix);
                const float gval = (float)(pfix - oc) * gmul;
                if (valid && v0 + u < V)
                    asm volatile("st.shared.f32 [%0], %1;\n" ::"r"(srow + 4u * (unsigned)(v0 + u)), "f"(gval) : "memory");
            }
        }
#endif
        // (the executing threads' shared-memory writes -> visible to the bulk-copy engine)
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(done + j);                          // the matrix buffer may be refilled
#ifdef PGASR_TIMING
        const long long c2 = clock64();
        tRows += c2 - c1;
#endif
        // ---- one bulk copy: the block's rows are contiguous in dlogits
        float* const out = dlog_u + (size_t)tlo * V;
        const unsigned bytes = (unsigned)(nf * V) * 4u;
        if (((reinterpret_cast<uintptr_t>(out) | bytes) & 15u) == 0u) {
            if (lane == 0) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n"
                             ::"l"(out), "r"(st_s), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
            }
        } else {
            for (int e = lane; e < nf * V; e += 32) out[e] = stage[e];
            __syncwarp();
        }
#ifdef PGASR_TIMING
        tCopy += clock64() - c2;
#endif
    }
    if (lane == 0) {                                      // the rows have to be in global memory before the CTA's flag
        asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
        asm volatile("fence.proxy.async;\n" ::: "memory");
    }
    __syncwarp();
#ifdef PGASR_TIMING
    if (dbg && lane == 0 && j == 0) {
        g_dbg[kAlpha ? 48 : 52] = tWait;
        g_dbg[kAlpha ? 49 : 53] = tRows;
        g_dbg[kAlpha ? 50 : 54] = tCopy;
        if (kAlpha) { g_dbg[56] = tPre; g_dbg[57] = tLoop; g_dbg[58] = nBlk; g_dbg[59] = ntrips; }
    }
#endif
}

}  // namespace pgasr
