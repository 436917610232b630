#pragma once
// (implementation header: included by fused_spl*.cu, one translation unit per states-per-lane variant)
// The whole PG + CTC loss step as ONE kernel launch (upstream call site: criterion(model_out, t) followed by
// loss.backward(), model.py:235-237; SURVEY.md rows a1-a8 chained).
//
// Grid = 2B CTAs that pick their role from an atomic ticket (tickets < B: CTC role of utterance `ticket`;
// the rest: PG role of utterance `ticket - B`), so the long-pole CTC CTAs are always resident before any PG CTA
// waits on them.  Both roles of an utterance run at the same time on different SMs:
//   CTC role: softmax of the utterance into an fp32 shared-memory tile, then warp 0 / warp 1 walk alpha / beta
//             (ctc_core.cuh) and write the CTC gradient rows; finally a release flag.
//   PG role:  logits tile -> shared memory (cp.async), one thread per frame: softmax CDF + K inverse-CDF draws
//             (Philox or injected uniforms), one warp per sample: ballot/popc collapse, one thread per sample:
//             bit-parallel Levenshtein against the transcript, warp 0: rewards / baseline / advantages, then the
//             REINFORCE gradient tile is built in place of the logits tile, the CTA acquires the CTC role's flag
//             and adds its tile onto the CTC rows with coalesced float4 read-modify-writes.
// The last CTA to finish (second ticket) reduces the loss in a fixed order and re-arms the control block.
// dlogits is written once by the CTC role and updated once by the PG role; every sum is order independent or
// fixed-order, so the step is bit-reproducible run to run.
#include <cstdlib>
#include <type_traits>

#include "ctc_core.cuh"
#include "fused_args.cuh"
#include "myers_core.cuh"
#include "words_core.cuh"

namespace pgasr {


__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(unsigned* p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}

constexpr int kFusedMaxK = 64;

#ifdef PGASR_TIMING
static __device__ unsigned long long g_cta_ns[2048][3];          // per ticket: start, role end, exit (globaltimer ns)
// per role (0 CTC, 1 PG), summed over every CTA since the last reset: CTAs, ns at the grid-dependency wait, ns from
// there to the exit, ns a PG CTA spent waiting for CTC flags -- what a CTA costs in SM time when steps overlap
static __device__ unsigned long long g_role_ns[2][4];
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
    return t;
}
#endif

// one bulk copy global -> shared memory, completion on an mbarrier (see fused.cu for the measured A/B)
__device__ __forceinline__ void bulk_load_tile(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
    const unsigned b = (unsigned)__cvta_generic_to_shared(bar), d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(b), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(d), "l"(gsrc), "r"(bytes), "r"(b) : "memory");
}

// Second ticket (thread 0 of a CTA, once): the CTA that draws the last one reduces the loss at the end of the kernel
// and re-arms the control block.  It is drawn as EARLY as the protocol allows -- by a CTC CTA right after it released
// its flag, by a PG CTA right after it acquired that flag and before its read-modify-write of dlogits -- so that the
// fence in front of it does not have to wait for 60 KB of freshly issued stores (that cost ~1 us at the end of the
// kernel).  Everything the last CTA reads (loss_terms[b], nll_ws[b]) was written by thread 0 of the owning CTA before
// this point; nobody reads a flag after its CTA drew this ticket, so re-arming the flags is safe.
__device__ __forceinline__ void draw_done_ticket(const FusedArgs& a, unsigned* s_last) {
    __threadfence();
    *s_last = atomicAdd(a.ctrl + 1, 1u) == gridDim.x - 1 ? 1u : 0u;
}

// One warp of the CTA that drew the last ticket: the loss in a fixed order, then the control block re-armed.
__device__ __forceinline__ void loss_reduce_and_rearm(const FusedArgs& a) {
    const int lane = threadIdx.x & 31;
    __threadfence();
    const float* nl = a.nll_ws;
    float pg = 0.0f, ct = 0.0f;
    for (int b = lane; b < a.B; b += 32) {
        if (a.do_pg) pg += __ldcg(a.loss_terms + b);
        if (a.do_ctc) ct += __ldcg(nl + b);
        a.ctrl[4 + b] = 0u;
    }
    pg = warp_sum(pg);
    ct = warp_sum(ct);
    if (lane == 0) {
        float l = 0.0f;
        if (a.do_pg) l += a.w_pg * pg / ((float)a.B * (float)a.K);
        if (a.do_ctc) l += a.w_ctc * ct / (float)a.B;
        a.loss[0] = l;
        a.ctrl[0] = 0u;
        a.ctrl[1] = 0u;
    }
}

// Number of entries of a non-decreasing 32-entry register array that are <= tau: a binary search written as a tree
// of selects (26 FSEL + 5 FSETP instead of 32 compare-and-add pairs).  Same count as the linear scan of the sampler
// spec because the CDF is non-decreasing (sums of non-negative terms, round to nearest).
__device__ __forceinline__ int cdf_count32(const float (&c)[32], float tau) {
    const bool b4 = c[15] <= tau;
    const float p3 = b4 ? c[23] : c[7];
    const bool b3 = p3 <= tau;
    const float q0 = b3 ? c[11] : c[3], q1 = b3 ? c[27] : c[19];
    const bool b2 = (b4 ? q1 : q0) <= tau;
    const float r0 = b2 ? c[5] : c[1], r1 = b2 ? c[13] : c[9], r2 = b2 ? c[21] : c[17], r3 = b2 ? c[29] : c[25];
    const float s0 = b3 ? r1 : r0, s1 = b3 ? r3 : r2;
    const bool b1 = (b4 ? s1 : s0) <= tau;
    float t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = b1 ? c[4 * i + 2] : c[4 * i];
    const float u0 = b2 ? t[1] : t[0], u1 = b2 ? t[3] : t[2], u2 = b2 ? t[5] : t[4], u3 = b2 ? t[7] : t[6];
    const float v0 = b3 ? u1 : u0, v1 = b3 ? u3 : u2;
    const bool b0 = (b4 ? v1 : v0) <= tau;
    return (b4 ? 16 : 0) + (b3 ? 8 : 0) + (b2 ? 4 : 0) + (b1 ? 2 : 0) + (b0 ? 1 : 0);
}

// One level of the binary search over a CDF row in shared memory, four draws side by side: off[u] is the row's
// shared-memory address plus four times the count so far (plain asm: free to be scheduled, ordered by the address).
template <int H>
__device__ __forceinline__ void cdf_search_step(unsigned (&off)[4], const float (&tau)[4]) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        float cv;
        asm("ld.shared.f32 %0, [%1+%2];\n" : "=f"(cv) : "r"(off[u]), "n"(4 * (H - 1)));
        off[u] += cv <= tau[u] ? 4u * H : 0u;
    }
}

// ------------------------------------------------------------------------------------------------ CTC role
// warp 0: alpha recurrence, warp 1: beta recurrence; every other warp is a gradient worker, even warps on the
// alpha side, odd warps on the beta side (G = (warps - 2) / 2 per direction).
// kGT (long utterances): the fp32 softmax tile does not fit in shared memory; it is written to the global
// workspace instead, the walkers stream it back through 32-row cp.async rings and the workers fetch their
// p_t(lane) with the lattice row.  Shared memory then no longer depends on T.
// kBW: block workers (ctc_core.cuh, "Block workers"): 5 occupancy workers and 2 row workers per direction instead of 7
// workers that do both; up to 8 states per lane, tile in shared memory, 512 threads.
template <int SPL, int kThreads, bool kGT, bool kBW = false>
__device__ void fused_ctc_role(const FusedArgs& a, int b, unsigned char* smem_raw, unsigned* s_last, unsigned long long* s_mbar) {
    static_assert(!kBW || (!kGT && SPL <= 8 && kThreads == 512 && (kBwGA == 4 || (kBwGA == 5 && kBwGB == 2)) && kBwGB <= 3), "block workers: tile mode only");
    constexpr int G = (kThreads / 32 - 2) / 2;             // gradient workers per direction
    constexpr int kPer = (kBatchOf<SPL> + G - 1) / G;      // frames of a batch per worker
    constexpr int kMidThreads = 32 * (2 + 2 * G);
    const int warp = threadIdx.x >> 5;
    const int T = a.T, V = a.V;
    PGASR_STAMP(b == 0 && threadIdx.x == 0, 6);
    // floats per tile row.  Block workers read and write the tile with a lane per FRAME, so consecutive rows must
    // fall into different banks: an odd stride with at least one zero slot after the V classes
    const int RS = kBW ? ((V + 1) | 1) : ctc_row_stride_f32(V);
    // shared-memory carve-up (see fused_smem)
    // [T][RS] between two pairs of guard rows: the walkers load the probabilities two frames ahead and run two rows
    // past either end (the guard values are loaded and never used)
    const int RSR = RS <= 32 ? 32 : RS <= 64 ? 64 : 128;                                  // ring row stride (power of two)
    const size_t pring_bytes = (size_t)kPRows * RSR * 4;
    float* tile;
    float* pring_a = nullptr;
    float* pring_b = nullptr;
    unsigned char* p;
    if (kGT) {
        tile = a.tile_g + ((size_t)b * (T + 2) + 1) * RS;
        // the dynamic shared memory window is 1 KB aligned at least; align the rings to their size by address
        const unsigned base = (unsigned)__cvta_generic_to_shared(smem_raw);
        const unsigned pad = (unsigned)((pring_bytes - (base & (pring_bytes - 1))) & (pring_bytes - 1));
        pring_a = reinterpret_cast<float*>(smem_raw + pad);
        pring_b = reinterpret_cast<float*>(smem_raw + pad + pring_bytes);
        p = smem_raw + pad + 2 * pring_bytes;
    } else {
        tile = reinterpret_cast<float*>(smem_raw) + 2 * RS;
        p = smem_raw + (((size_t)(T + 4) * RS * 4 + 15) & ~(size_t)15);
    }
    constexpr int kNB = kBW ? kBwNB : kBatchOf<SPL>;                    // frames per hand-off batch
    int* bw_gam = nullptr;
    if constexpr (kBW) {
        // block workers: the four occupancy matrices come first, 128-byte aligned BY ADDRESS (the frame-slot xor of the
        // row workers stays inside a 128-byte row)
        const unsigned at = (unsigned)__cvta_generic_to_shared(p);
        p += (128u - (at & 127u)) & 127u;
        bw_gam = reinterpret_cast<int*>(p);
    }
    unsigned char* const stage_base = p;
    if constexpr (kBW) p += 2 * bw_gam_bytes<SPL>();
    GradRing<SPL, kNB> ring_a = grad_ring_carve<SPL, kNB>(p, 2);        p += grad_ring_bytes<SPL, kNB>();
    GradRing<SPL, kNB> ring_b = grad_ring_carve<SPL, kNB>(p, 6);        p += grad_ring_bytes<SPL, kNB>();
    int* gam_all = reinterpret_cast<int*>(p);                           // [2 G workers][kPer frames][16 SPL]
    // (block workers: [2 directions][kBwGB buffers][16 SPL labels][32 frame slots])
    const size_t gam_bytes = kBW ? 2 * bw_gam_bytes<SPL>() : (size_t)2 * G * kPer * 16 * SPL * sizeof(int);
    if constexpr (!kBW) p += gam_bytes;
    int* cls_off = reinterpret_cast<int*>(p);                           // [V + 1]
    int* cls_scr = cls_off + (V + 1);                                   // [V] counting-sort scratch
    int* cls_pos = cls_scr + V;                                         // [512]
    int* lab_s = cls_pos + 512;                                         // [512] the transcript
    // block workers: one class-ordered label list per matrix buffer (16-byte aligned; bw_build_list), the buffers'
    // "consumed" mbarriers, one staging buffer per row worker
    unsigned* bw_lists = reinterpret_cast<unsigned*>((reinterpret_cast<uintptr_t>(lab_s + 512) + 15) & ~(uintptr_t)15);
    unsigned long long* bw_done = reinterpret_cast<unsigned long long*>(bw_lists + 2 * kBwGB * kBwListWords);   // [2][kBwGB]
    float* bw_stage = reinterpret_cast<float*>(bw_done + 2 * kBwGB);    // [2][kBwGB][32 frames][32]
    // The transcript and the lengths may live in mapped HOST memory (pgasr_host_*: a PCIe round trip per dependent
    // access), so everything is fetched here in one go and the transcript is used from shared memory afterwards.
    // the whole logits tile as one bulk load, issued before anything is known about the utterance's length (rows beyond it
    // are loaded and never used): the load then flies while the lengths and the transcript arrive
    const size_t stage_bytes = 2 * grad_ring_bytes<SPL, kNB>() + gam_bytes;
    const int stage_chunk = (int)(stage_bytes / ((size_t)V * 4)) & ~3;
    const bool early_bulk = a.bulk_tile && stage_chunk >= T;
    if (early_bulk && threadIdx.x == 0)
        bulk_load_tile(stage_base, a.logits + (size_t)b * T * V, (unsigned)((size_t)T * V * 4), s_mbar);
    for (int i = threadIdx.x; i < a.Lmax; i += kThreads) lab_s[i] = a.targets[(size_t)b * a.Lmax + i];
    int Tb = a.in_len ? a.in_len[b] : T;
    Tb = min(max(Tb, 0), T);
    int L = a.tgt_len ? a.tgt_len[b] : a.Lmax;
    L = min(max(L, 0), a.Lmax);
    float* dlog_u = a.dlogits + (size_t)b * T * V;
    float* nll_u = a.nll_ws + b;
    PGASR_STAMP(b == 0 && threadIdx.x == 0, 0);
    for (int i = Tb * V + threadIdx.x; i < T * V; i += kThreads) dlog_u[i] = 0.0f;
    if (Tb == 0) {
        if (early_bulk) mbar_wait(s_mbar, 0u);             // (nothing may still be landing in shared memory when the CTA ends)
        if (threadIdx.x == 0) *nll_u = L == 0 ? 0.0f : INFINITY;
    } else {
        ring_a.dbg = ring_b.dbg = (b == 0);
        PGASR_STAMP(b == 0 && threadIdx.x == 0, 1);
        // softmax tile.  The raw logits are staged through the (not yet used) ring region with cp.async, then one
        // thread per frame makes three passes over its row -- max, exp + sum, normalise -- visiting the classes in
        // a per-thread rotated order so that neither the staged reads (row stride V floats) nor the fp32 tile
        // writes (row stride RS floats) collide on a shared-memory bank.  (One warp per frame with a lane per
        // class was measured at twice the time, 17.9k against 9k cycles: 5 shuffles + a redux per frame.)
        const float* lg = a.logits + (size_t)b * T * V;
        {
            float* stage = reinterpret_cast<float*>(stage_base);
            const int chunk = stage_chunk;
            // (any float* is a valid logits pointer: the 16-byte copies need the base aligned too.  Every utterance's
            // base differs by T*V*4 bytes, so the predicate is the same for all of them)
            const bool al16 = ((reinterpret_cast<uintptr_t>(lg) | ((size_t)T * V * 4)) & 15) == 0;
            for (int c0 = 0; c0 < Tb; c0 += chunk) {
                const int n = min(chunk, Tb - c0);
                const float* src = lg + (size_t)c0 * V;
                const bool bulk = early_bulk;              // (then the one chunk is the whole utterance)
                if (bulk) {
                } else if (al16) {
                    const int n16 = n * V / 4, rem = n * V - n16 * 4;
                    for (int i = threadIdx.x; i < n16; i += kThreads)
                        cp_async16(reinterpret_cast<char*>(stage) + (size_t)i * 16,
                                   reinterpret_cast<const char*>(src) + (size_t)i * 16);
                    for (int i = threadIdx.x; i < rem; i += kThreads) cp_async4(stage + n16 * 4 + i, src + n16 * 4 + i);
                } else {
                    for (int i = threadIdx.x; i < n * V; i += kThreads) cp_async4(stage + i, src + i);
                }
                cp_async_commit();
                if (c0 == 0) {
                    // class lists of the transcript, built by warp 0 while the logits are in flight
                    __syncthreads();                           // the transcript is in shared memory
                    if (warp == 0) {
                        ctc_build_class_lists(lab_s, L, V, cls_off, cls_pos, cls_scr);
                        if constexpr (kBW) {
                            if (threadIdx.x < 2 * kBwGB) mbar_init(bw_done + threadIdx.x, 1);
                        }
                    }
                }
                if (bulk) mbar_wait(s_mbar, 0u);
                cp_async_wait<0>();
                __syncthreads();
                if constexpr (kBW) {
                    // the class lists are visible now: warp c writes the list of matrix buffer c (published by the
                    // barrier at the end of this chunk)
                    if (c0 == 0 && warp < 2 * kBwGB)
                        bw_build_list<SPL>(cls_off, cls_pos, V, bw_lists + warp * kBwListWords,
                                           reinterpret_cast<int*>(bw_lists + warp * kBwListWords + kBwInfoAt),
                                           (unsigned)__cvta_generic_to_shared(bw_gam + warp * (16 * SPL * 32)));
                }
                if (V > 32) {
                    // wide alphabets (33..64 classes): three plain passes over the staged row, no register-resident row
                    for (int t = threadIdx.x; t < n; t += kThreads) {
                        const float* zr = stage + (size_t)t * V;
                        float* orow = tile + (size_t)(c0 + t) * RS;
                        float m = -INFINITY, s = 0.0f;
                        for (int v = 0; v < V; ++v) m = fmaxf(m, zr[v]);
                        for (int v = 0; v < V; ++v) s += __expf(zr[v] - m);
                        const float inv = 1.0f / s;
                        for (int v = 0; v < V; ++v) orow[v] = __expf(zr[v] - m) * inv;
                        for (int v = V; v < RS; ++v) orow[v] = 0.0f;
                    }
                } else
                for (int t = threadIdx.x; t < n; t += kThreads) {
                    // the row lives in registers in rotated order (slot k holds class (k + t) & 31): the order does
                    // not matter for the max and the sum, every load / exp / store is independent of the others
                    const float* zr = stage + (size_t)t * V;
                    float* orow = tile + (size_t)(c0 + t) * RS;
                    // (block workers: the tile's row stride is odd, so the UNROTATED order is the conflict-free one for
                    // the writes; the staged reads are then two-way conflicted, 64 wavefronts per warp, once)
                    const int rot = kBW ? 0 : t;
                    float x[32];
#pragma unroll
                    for (int k = 0; k < 32; ++k) {
                        const int idx = (k + rot) & 31;
                        x[k] = idx < V ? zr[idx] : -INFINITY;
                    }
                    float m4[4] = {x[0], x[1], x[2], x[3]};
#pragma unroll
                    for (int k = 4; k < 32; ++k) m4[k & 3] = fmaxf(m4[k & 3], x[k]);
                    const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
                    float s4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
                    for (int k = 0; k < 32; ++k) {
                        x[k] = __expf(x[k] - m);                   // exp(-inf) = 0 for the unused slots
                        s4[k & 3] += x[k];
                    }
                    const float inv = 1.0f / ((s4[0] + s4[1]) + (s4[2] + s4[3]));
#pragma unroll
                    for (int k = 0; k < 32; ++k) {
                        const int idx = (k + rot) & 31;
                        if (idx < RS) orow[idx] = x[k] * inv;
                    }
                    for (int idx = 32; idx < RS; ++idx) orow[idx] = 0.0f;
                }
                if (kGT) __threadfence_block();            // the rows go to global memory: order them before the barrier
                __syncthreads();
            }
        }
        const int32_t* lab_u = lab_s;                      // (published by the barriers of the tile loop above,
        ring_a.cls_off = ring_b.cls_off = cls_off;         //  like the class lists)
        ring_a.cls_pos = ring_b.cls_pos = cls_pos;
        PGASR_STAMP(b == 0 && threadIdx.x == 0, 2);
        double* lat_u = a.lattice + (size_t)b * T * (SPL * 32);
        int* exp_u = a.lat_exp + (size_t)b * T;
        const float gs = a.w_ctc / (float)a.B;
        auto mid = [] {
            __threadfence_block();
            asm volatile("bar.sync 1, %0;\n" ::"n"(kMidThreads) : "memory");
        };
        const int g = (warp - 2) >> 1;
        if constexpr (kBW) {
            // even warps serve alpha, odd warps beta; w = warp / 2 is the warp's number within its direction: 0 the
            // walker, odd w the A-workers (scheduler partitions 2 / 3), even w the B-workers (the walker's partition)
#if defined(PGASR_ROLE_MAP) && PGASR_ROLE_MAP == 1
            // (A/B) both walkers on partition 0, the four B-workers on partition 1, A-workers on 2 / 3
            const int pp = warp & 3, ii = warp >> 2;
            const bool al = pp == 0 ? ii == 0 : pp == 1 ? ii < 2 : pp == 2;
            const bool walker = pp == 0 && ii < 2;
            const int bj = pp == 1 ? (ii & 1) : -1;
            const int ga = pp >= 2 ? ii : -1;
#elif defined(PGASR_ROLE_MAP) && PGASR_ROLE_MAP == 2
            // (A/B) walkers on partitions 0 / 1 as usual, but each walker shares its partition with the OTHER direction's B-workers
            const int w0 = warp >> 1;
            const bool isb = !(w0 & 1) && w0 >= 2 && (w0 >> 1) - 1 < kBwGB;
            const bool al = isb ? (warp & 1) : !(warp & 1);
            const bool walker = warp < 2;
            const int bj = isb ? (w0 >> 1) - 1 : -1;
            const int ga = (w0 & 1) ? (w0 >> 1) : -1;
#elif defined(PGASR_ROLE_MAP) && PGASR_ROLE_MAP == 3
            // (A/B) per direction: partition 0 / 1 = walker, B-worker 0, A-worker 0, spare; partition 2 / 3 = A-workers 1..3
            // and B-worker 1 (evens out the instruction load of the partitions: 99 / 87 per frame instead of 110 / 75)
            const bool al = !(warp & 1);
            const int w = warp >> 1;                   // 0..7 within the direction: partitions 0,2,0,2,0,2,0,2 (alpha)
            const bool walker = w == 0;
            const int bj = w == 2 ? 0 : w == 7 ? 1 : -1;
            const int ga = w == 4 ? 0 : w == 1 ? 1 : w == 3 ? 2 : w == 5 ? 3 : -1;
#else
            const bool al = !(warp & 1);
            const int w = warp >> 1;
            const bool walker = warp < 2;
            const int bj = (!(w & 1) && w >= 2 && (w >> 1) - 1 < kBwGB) ? (w >> 1) - 1 : -1;
            const int ga = (w & 1) ? (w >> 1) : (kBwGA == 5 && w == 6) ? 4 : -1;
#endif
            const int dirx = al ? 0 : 1;
            int* gam_d = bw_gam + dirx * (kBwGB * 16 * SPL * 32);
            unsigned long long* done_d = bw_done + dirx * kBwGB;
            const int bar_g = al ? 10 : 13;
            const unsigned* list_w = bw_lists + (dirx * kBwGB + max(bj, 0)) * kBwListWords;
            if (walker && al)
                ctc_walk_tile<SPL, kBwGA, true, false, kBwNB>(tile, lab_u, Tb, L, V, RS, a.blank, nll_u, lat_u, exp_u, ring_a, mid);
            else if (walker)
                ctc_walk_tile<SPL, kBwGA, false, false, kBwNB>(tile, lab_u, Tb, L, V, RS, a.blank, nll_u, lat_u, exp_u, ring_b, mid);
            else if (bj >= 0)
                ctc_bworker<SPL>(al, bj, tile, RS, Tb, V, a.blank, gs, dlog_u, al ? ring_a.norm : ring_b.norm, done_d, bar_g,
                                 list_w, reinterpret_cast<const int*>(list_w + kBwInfoAt),
                                 bw_stage + (dirx * kBwGB + bj) * (kBwBlk * 32), mid, b == 0);
            else if (ga >= 0)
                ctc_aworker<SPL>(al, ga, Tb, L, lat_u, exp_u, al ? ring_a : ring_b, gam_d, done_d, bar_g, mid);
            else
                mid();                                     // a spare warp: it only takes part in the CTA-wide barriers
        } else
        if (warp == 0)
            ctc_walk_tile<SPL, G, true, kGT>(tile, lab_u, Tb, L, V, RS, a.blank, nll_u, lat_u, exp_u, ring_a, mid, pring_a,
                                             RSR, T);
        else if (warp == 1)
            ctc_walk_tile<SPL, G, false, kGT>(tile, lab_u, Tb, L, V, RS, a.blank, nll_u, lat_u, exp_u, ring_b, mid,
                                              pring_b, RSR, T);
        else if (g < G && !(warp & 1))
            ctc_grad_worker<SPL, G, true, kGT>(g, tile, lab_u, Tb, L, V, RS, a.blank, gs, dlog_u, lat_u, exp_u, ring_a,
                                               gam_all + g * kPer * 16 * SPL, mid);
        else if (g < G)
            ctc_grad_worker<SPL, G, false, kGT>(g, tile, lab_u, Tb, L, V, RS, a.blank, gs, dlog_u, lat_u, exp_u, ring_b,
                                                gam_all + (G + g) * kPer * 16 * SPL, mid);
    }
    __threadfence();                                       // rows and nll visible device-wide before the flag
    __syncthreads();
#ifdef PGASR_TIMING
    // (a clock64 right behind the barrier would execute before the barrier releases, BAR.SYNC.DEFER_BLOCKING: take it
    // behind a shared-memory load)
    if (b == 0 && threadIdx.x == 0) { const unsigned x = *reinterpret_cast<volatile unsigned*>(s_last); asm volatile("" ::"r"(x) : "memory"); }
#endif
    PGASR_STAMP(b == 0 && threadIdx.x == 0, 3);
    // Thread 0's chain here is what every other warp of the CTA -- and the SM -- waits for (measured: 5.8 k cycles with a
    // release store, a second fence, the ticket and the nll copy one after the other).  One fence orders the CTA's rows, nll
    // and loss term before BOTH the flag and the ticket: the fence inside st.release, with the ticket behind it in program
    // order.  Flag store and ticket may then become visible in either order, which is fine: the last ticket of the grid
    // (whose CTA re-arms the flags) is drawn after this utterance's PG CTA drew its own, and that CTA has read the flag by
    // then.  Without a PG role nobody reads the flag: it is not set at all.  The caller's nll copy rides on another warp.
    if (threadIdx.x == 32 && a.nll) a.nll[b] = *nll_u;     // (possibly host memory; the loss reads nll_ws)
    if (threadIdx.x == 0) {
        if (a.do_pg) st_release(a.ctrl + 4 + b, 1u);
        else __threadfence();
        PGASR_STAMP(b == 0, 9);
        *s_last = atomicAdd(a.ctrl + 1, 1u) == gridDim.x - 1 ? 1u : 0u;
        PGASR_STAMP(b == 0, 7);
    }
}

// exploration variant: z' = fl32(z theta) over a logits tile in shared memory, float4 where the tile allows
template <int kThreads>
__device__ __forceinline__ void scale_tile(float* z, int n, float theta) {
    float4* z4 = reinterpret_cast<float4*>(z);
    const int n4 = n / 4;
    for (int i = threadIdx.x; i < n4; i += kThreads) {
        float4 x = z4[i];
        x.x = __fmul_rn(x.x, theta); x.y = __fmul_rn(x.y, theta); x.z = __fmul_rn(x.z, theta); x.w = __fmul_rn(x.w, theta);
        z4[i] = x;
    }
    for (int i = n4 * 4 + threadIdx.x; i < n; i += kThreads) z[i] = __fmul_rn(z[i], theta);
}

// ------------------------------------------------------------------------------------------------ PG role
// kStream (long utterances): no [T][V] tile in shared memory -- a thread reads its frame's logits straight from
// global memory, and the gradient rows are formed in registers and added to dlogits row by row.
// A PG CTA serves `nutt` utterances b0, b0 + 1 (two in the common mode, a.pg_pair): the sampling of the two runs one
// after the other on the one logits tile buffer, but their edit distances -- the phase that keeps only four warps of
// the CTA busy -- run side by side, so the pair costs one edit-distance phase instead of two.
struct PgU {
    int b, Tb, m;
    uint8_t *samples_s, *hyp_s, *hrev_s;
    uint32_t *peq, *peq_r;
    int16_t* fg_s;
    double* warp_acc;
    float* adv_s;
    int *hlen_s, *dist_s;
    float* misc_s;
};
// kWord (word-level rewards, DESIGN.md "word reward spec"): a word phase after P2 turns every collapsed hypothesis into
// its sequence of word classes, the transcript's words become the match table, and P3 runs over words.
// (the word arguments come as a parameter pack, empty for the character modes: their role keeps its exact signature --
// where it is not inlined, an extra parameter changes its call frame)
// kExp (exploration, DESIGN.md "exploration spec"): the logits are scaled by theta -- the tile once after its load, the
// streamed rows on read -- so P1 samples softmax(theta z); P5 multiplies the coefficients by theta and adds the
// entropy term, and writes H_b.  Its ExploreArgs come last in the same pack.
struct PgExtra { WordArgs w; ExploreArgs x; };
__device__ __forceinline__ PgExtra pg_extra() { return PgExtra{{-1, 0}, {1.0f, 0.0f, 0.0f, nullptr}}; }
__device__ __forceinline__ PgExtra pg_extra(const WordArgs& w) { return PgExtra{w, {1.0f, 0.0f, 0.0f, nullptr}}; }
__device__ __forceinline__ PgExtra pg_extra(const ExploreArgs& x) { return PgExtra{{-1, 0}, x}; }
__device__ __forceinline__ PgExtra pg_extra(const WordArgs& w, const ExploreArgs& x) { return PgExtra{w, x}; }
template <int W, int kThreads, bool kStream, bool kWord = false, bool kExp = false, typename... XA>
__device__ void fused_pg_role(const FusedArgs& a, int b0, int nutt, unsigned char* smem_raw, unsigned* s_last,
                              unsigned long long* s_mbar, const XA&... extra) {
    static_assert(sizeof...(XA) == (kWord ? 1 : 0) + (kExp ? 1 : 0), "WordArgs for the word modes, then ExploreArgs");
    const PgExtra px = pg_extra(extra...);
    const WordArgs wa = px.w;
    const float theta = px.x.theta;
    (void)theta;
    // a value of the frame's row as the policy sees it: streamed rows are scaled on read, the tile already is
    auto zv = [&](const float* z, int v) { return kExp && kStream ? __fmul_rn(z[v], theta) : z[v]; };
    constexpr int kWarps = kThreads / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int T = a.T, V = a.V, K = a.K;
    const int Tp = (T + 15) & ~15;
    const int Tp2 = (T / 2 + 16) & ~15;
    // rows of the match tables: the alphabet, or (word modes) the transcript's word classes
    const int Vp = kWord ? max(V, wa.cap) : V;

    // shared-memory carve-up: the logits tile (shared by the utterances of the CTA), one block per utterance, then the
    // reward-to-go arrays and the CDF rows
    float* ztile = reinterpret_cast<float*>(smem_raw);                                // [T][V] (tile mode only)
    const size_t off0 = kStream ? 0 : (((size_t)T * V * 4 + 15) & ~(size_t)15);
    const size_t ubytes = pg_u_bytes<W, kThreads>(T, Vp, K);
    auto pg_u = [&](int uu) {
        PgU X;
        X.b = b0 + uu;
        int Tb = a.in_len ? a.in_len[X.b] : T;
        X.Tb = min(max(Tb, 0), T);
        int m = a.tgt_len ? a.tgt_len[X.b] : a.Lmax;
        X.m = min(max(m, 0), a.Lmax);
        unsigned char* p = smem_raw + off0 + (size_t)uu * ubytes;
        size_t off = 0;
        X.samples_s = p + off;            off += (size_t)K * Tp;            // [K][Tp]
        X.hyp_s = p + off;                off += (size_t)K * Tp;            // [K][Tp]
        X.hrev_s = p + off;               off += (size_t)K * Tp2;           // [K][Tp2] second halves, reversed
        X.peq = reinterpret_cast<uint32_t*>(p + off);   off += (size_t)(Vp + 1) * W * 4;
        X.peq_r = reinterpret_cast<uint32_t*>(p + off); off += (size_t)(Vp + 1) * W * 4;   // reversed transcript
        X.fg_s = reinterpret_cast<int16_t*>(p + off);   off += (size_t)((K + 7) & ~7) * (W * 32 + 2) * 2;   // (idle groups of the last warp get their own scratch)
        off = (off + 15) & ~(size_t)15;
        X.warp_acc = reinterpret_cast<double*>(p + off); off += (size_t)kWarps * kFusedMaxK * 8;   // log-prob partial sums
        X.adv_s = reinterpret_cast<float*>(p + off);     off += kFusedMaxK * 4;
        X.hlen_s = reinterpret_cast<int*>(p + off);      off += kFusedMaxK * 4;
        X.dist_s = reinterpret_cast<int*>(p + off);      off += kFusedMaxK * 4;
        X.misc_s = reinterpret_cast<float*>(p + off);    // [0] sum of advantages; word modes: [1] n_w, [2] classes (int)
        return X;
    };
    size_t off = off0 + (size_t)nutt * ubytes;
    // reward-to-go mode: log-sum-exp of every frame (P1 -> P5) and, per sample, the last column of the edit-distance
    // table c[i] = ED(ref, hyp[:i]) (int16, i = 0..n), later overwritten in place by the reward-to-go of every frame
    const bool togo = a.reward_mode == PGASR_REWARD_ED_TO_GO;
    const int Tc = Tp + 16;
    float* lz_s = reinterpret_cast<float*>(smem_raw + off);      if (togo) off += (size_t)Tp * 4;
    int* warp_acc_i = reinterpret_cast<int*>(smem_raw + off);    if (togo) off += (size_t)kWarps * 64 * 4;   // emitted symbols before each 32-frame chunk
    int16_t* col_s = reinterpret_cast<int16_t*>(smem_raw + off); if (togo) off += (size_t)K * Tc * 2;   // [K][Tc]
    off = (off + 15) & ~(size_t)15;
    float* cdf_s = reinterpret_cast<float*>(smem_raw + off);     // [kThreads][33] (a.cdf_smem)
    // word modes: the scratch of the word phase (transcripts, one block per warp) in place of the CDF rows, dead by then
    unsigned char* const wtail = reinterpret_cast<unsigned char*>(cdf_s);
    (void)wtail;
    unsigned nload = 0;                                    // bulk tile loads so far (the mbarrier's phase)
    int ref_rr[2][2];

    // ======== sampling, one utterance after the other ========
    for (int uu = 0; uu < nutt; ++uu) {
        const PgU X = pg_u(uu);
        const int b = X.b, Tb = X.Tb, m = X.m;
        uint8_t* const samples_s = X.samples_s; uint8_t* const hyp_s = X.hyp_s; uint8_t* const hrev_s = X.hrev_s;
        uint32_t* const peq = X.peq; uint32_t* const peq_r = X.peq_r; int16_t* const fg_s = X.fg_s;
        double* const warp_acc = X.warp_acc; float* const adv_s = X.adv_s; int* const hlen_s = X.hlen_s;
        int* const dist_s = X.dist_s; float* const misc_s = X.misc_s;
        const float* const lg = a.logits + (size_t)b * T * V;
        const int32_t* const ref = a.targets + (size_t)b * a.Lmax;
        const bool dbg = b == 0 && threadIdx.x == 0;
        (void)dbg; (void)samples_s; (void)hyp_s; (void)hrev_s; (void)peq; (void)peq_r; (void)fg_s; (void)warp_acc; (void)adv_s;
        (void)hlen_s; (void)dist_s; (void)misc_s; (void)lg; (void)ref; (void)Tb; (void)m;
        int (&ref_r)[2] = ref_rr[uu];
        PGASR_STAMP(dbg, 30);
        // ---- P0: logits tile -> shared memory ------------------------------------------------------
        if (!kStream && a.bulk_tile) {
            if (threadIdx.x == 0) bulk_load_tile(ztile, lg, (unsigned)((size_t)T * V * 4), s_mbar);
        } else if (!kStream) {
            if (((reinterpret_cast<uintptr_t>(lg) | ((size_t)T * V * 4)) & 15) == 0) {
                const int n16 = T * V / 4;
                for (int i = threadIdx.x; i < n16; i += kThreads)
                    cp_async16(reinterpret_cast<char*>(ztile) + (size_t)i * 16, reinterpret_cast<const char*>(lg) + (size_t)i * 16);
            } else {
                for (int i = threadIdx.x; i < T * V; i += kThreads) cp_async4(ztile + i, lg + i);
            }
            cp_async_commit();
        }
        // the transcript may live in mapped host memory: fetch it now, it is needed after the sampling phase
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int j = threadIdx.x + q * kThreads;
            ref_r[q] = j < m ? ref[j] : -1;
        }
        for (int i = threadIdx.x; i < kWarps * kFusedMaxK; i += kThreads) warp_acc[i] = 0.0;
        for (int i = threadIdx.x; i < (Vp + 1) * W; i += kThreads) { peq[i] = 0u; peq_r[i] = 0u; }
        if (!kStream && a.bulk_tile) mbar_wait(s_mbar, nload++ & 1u);
        cp_async_wait<0>();
        __syncthreads();
        if constexpr (kExp && !kStream) {
            if (theta != 1.0f) {                           // z' = z theta, once per tile (theta = 1: z' = z bit for bit)
                scale_tile<kThreads>(ztile, T * V, theta);
                __syncthreads();
            }
        }


        PGASR_STAMP(dbg, 31);
        // ---- P1: softmax CDF + K draws, one thread per frame (DESIGN.md "sampler spec") ------------
        const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
        for (int t0 = 0; t0 < T; t0 += kThreads) {
            const int t = t0 + threadIdx.x;
            const bool live = t < Tb;
            const float* z = (kStream ? lg : ztile) + (size_t)(live ? t : 0) * V;
            // one code path per alphabet width: the CDF lives in 32 registers (V <= 32, the common case) or in 64
            auto sample_frame = [&](auto vp_tag) {
                constexpr int VPW = decltype(vp_tag)::value;
                float cdf[VPW];
                float mx = -INFINITY, S = 0.0f, logS = 0.0f;
                if (live) {
#pragma unroll
                    for (int v = 0; v < VPW; ++v) cdf[v] = v < V ? zv(z, v) : -INFINITY;
#pragma unroll
                    for (int v = 0; v < VPW; ++v) mx = fmaxf(mx, cdf[v]);
                    float c = 0.0f;
#pragma unroll
                    for (int v = 0; v < VPW; ++v) {
                        if (v < V) c = __fadd_rn(c, exp_spec(__fsub_rn(cdf[v], mx)));
                        cdf[v] = c;
                    }
                    S = c;
                    logS = logf(S);
                    if (togo) lz_s[t] = mx + logS;
                }
                uint4 rnd = make_uint4(0, 0, 0, 0);
                for (int k = 0; k < K; ++k) {
                    float term = 0.0f;
                    int pi = 0;
                    if (live) {
                        float u;
                        if (a.uniforms) {
                            u = __ldg(a.uniforms + ((size_t)b * K + k) * T + t);
                        } else {
                            if ((k & 3) == 0)
                                rnd = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)b, (uint32_t)(k >> 2), 0x50474153u), key);
                            const uint32_t x = (k & 3) == 0 ? rnd.x : (k & 3) == 1 ? rnd.y : (k & 3) == 2 ? rnd.z : rnd.w;
                            u = u32_to_uniform(x);
                        }
                        const float tau = __fmul_rn(u, S);
                        // (entries V.. of cdf[] repeat S, so the count over all entries differs from the spec's count
                        // over V entries only when tau == S, where both clamp to V - 1)
                        int cnt;
                        if constexpr (VPW == 32) {
                            cnt = cdf_count32(cdf, tau);
                        } else {
                            const bool hi = cdf[31] <= tau;           // the CDF is non-decreasing: pick the half, search it
                            float half[32];
#pragma unroll
                            for (int i = 0; i < 32; ++i) half[i] = hi ? cdf[32 + i] : cdf[i];
                            cnt = (hi ? 32 : 0) + cdf_count32(half, tau);
                        }
                        pi = min(cnt, V - 1);
                        term = (zv(z, pi) - mx) - logS;
                    }
                    if (t < T) {
                        samples_s[(size_t)k * Tp + t] = (uint8_t)pi;
                        if (a.samples) a.samples[((size_t)b * K + k) * T + t] = (uint8_t)pi;
                    }
                    // the warp's 32 terms in ONE instruction: 2^-19 fixed point (a term lies in [-92, 0]: the sum of 32 fits an
                    // int32; the rounding, 1e-6 per frame, is far inside the 1e-4 the log-probabilities are checked to)
                    const int ti = __reduce_add_sync(kFull, __float2int_rn(term * 524288.0f));
                    if (lane == 0) warp_acc[warp * kFusedMaxK + k] += (double)ti * (1.0 / 524288.0);   // across passes and warps in fp64: log p ~ -1000
                }
            };
            if (!kStream && a.cdf_smem) {
                // The CDF row of the frame in shared memory (33 floats: odd stride, a thread's walk along its row never
                // collides with its neighbours'), built and searched by ROLLED loops: the fully unrolled register version
                // is ~2000 straight-line instructions per thread, and with every warp streaming through them once the phase
                // was bound by instruction fetch (no_inst was half of its stall samples).  Same arithmetic, same counts.
                float* cr = cdf_s + (size_t)threadIdx.x * 33;       // (one row per thread, reused by every pass)
                float mx = -INFINITY, S = 0.0f, logS = 0.0f;
                if (live) {
#pragma unroll 2
                    for (int v = 0; v < V; ++v) mx = fmaxf(mx, z[v]);
                    // four classes at a time: the four exp chains are independent, only the running sum is sequential
                    // (a thread's chain of ~25 dependent fp32 operations per class left the issue slots idle: 290 cycles
                    // per class with four warps per scheduler, measured).  Entries V..31 repeat S.
                    float c = 0.0f;
#pragma unroll 1
                    for (int v = 0; v < 32; v += 4) {
                        float e[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) e[u] = exp_spec(__fsub_rn(z[min(v + u, V - 1)], mx));
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            c = v + u < V ? __fadd_rn(c, e[u]) : c;
                            cr[v + u] = c;
                        }
                    }
                    S = c;
                    logS = logf(S);
                    if (togo) lz_s[t] = mx + logS;
                }
                PGASR_STAMP(dbg && t0 == 0, 60);
                // four draws (one Philox block) side by side.  The loop is instantiated per source of the uniforms and per
                // "K is a multiple of four", so that its body is ONE basic block: with the run-time tests inside it the
                // compiler recomputed the frame's row address for every draw (11 instructions per z[pi]) and kept a
                // branch per draw (~90 instructions per draw, now ~70).  The search walks a BYTE offset (the count is the
                // offset / 4); the 32 log-prob terms of a warp and draw are summed by one redux in 2^-19 fixed point (a
                // term lies in [-92, 0]: the sum fits an int32) and kept by lane k of the warp until the end of the pass.
                // Shared-memory addresses are taken once, as opaque 32-bit values: the role is compiled against the CTA's
                // 128-register cap and the compiler otherwise REMATERIALISES them per draw (window base, padded row stride,
                // even the thread index) rather than hold them.  Frames beyond T (last pass) store to the unused 33rd entry
                // of the thread's CDF row with stride 0, so the stores need no branch.
                unsigned cr32 = (unsigned)__cvta_generic_to_shared(cr);
                unsigned z32 = (unsigned)__cvta_generic_to_shared(z);
                unsigned s32 = t < T ? (unsigned)__cvta_generic_to_shared(samples_s + t) : cr32 + 128u;
                unsigned sstr = t < T ? (unsigned)Tp : 0u;
                asm volatile("mov.u32 %0, %0;\n mov.u32 %1, %1;\n mov.u32 %2, %2;\n mov.u32 %3, %3;\n"
                             : "+r"(cr32), "+r"(z32), "+r"(s32), "+r"(sstr) : : "memory");   // (after the row's stores above)
                auto draw_loop = [&](auto ph_tag, auto full_tag) {
                    constexpr bool kPh = decltype(ph_tag)::value, kFullK = decltype(full_tag)::value;
                    int acc = 0;                              // lane k & 31: sum of draw k's terms over the warp's frames
                    auto flush = [&](int base) {              // across passes and warps in fp64: log p ~ -1000
                        if (base + lane < K) warp_acc[warp * kFusedMaxK + base + lane] += (double)acc * (1.0 / 524288.0);
                        acc = 0;
                    };
                    unsigned sk = s32;                        // running address of samples_s[k0][t]
#pragma unroll 1
                    for (int k0 = 0; k0 < K; k0 += 4) {
                        if (k0 == 32) flush(0);               // (K > 32: the lanes take the second 32 draws)
                        float term[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                        int pi[4] = {0, 0, 0, 0};
                        if (live) {
                            float tau[4];
                            if constexpr (kPh) {
                                const uint4 rnd = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)b, (uint32_t)(k0 >> 2), 0x50474153u), key);
                                tau[0] = __fmul_rn(u32_to_uniform(rnd.x), S);
                                tau[1] = __fmul_rn(u32_to_uniform(rnd.y), S);
                                tau[2] = __fmul_rn(u32_to_uniform(rnd.z), S);
                                tau[3] = __fmul_rn(u32_to_uniform(rnd.w), S);
                            } else {
#pragma unroll
                                for (int u = 0; u < 4; ++u) {
                                    const float un = (kFullK || k0 + u < K) ? __ldg(a.uniforms + ((size_t)b * K + k0 + u) * T + t) : 0.0f;
                                    tau[u] = __fmul_rn(un, S);
                                }
                            }
                            unsigned off[4] = {cr32, cr32, cr32, cr32};   // row address + 4 #{v < 32 : cdf[v] <= tau} (non-decreasing CDF)
                            cdf_search_step<16>(off, tau); cdf_search_step<8>(off, tau); cdf_search_step<4>(off, tau);
                            cdf_search_step<2>(off, tau);  cdf_search_step<1>(off, tau);
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                pi[u] = min((int)((off[u] - cr32) >> 2), V - 1);
                                float zv;
                                asm("ld.shared.f32 %0, [%1];\n" : "=f"(zv) : "r"(z32 + 4u * (unsigned)pi[u]));
                                term[u] = (kFullK || k0 + u < K) ? (zv - mx) - logS : 0.0f;
                            }
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int k = k0 + u;
                            if (kFullK || k < K) {                // (warp uniform)
                                asm volatile("st.shared.u8 [%0], %1;\n" ::"r"(sk), "r"(pi[u]));
                                sk += sstr;
                                const int ti = __reduce_add_sync(kFull, __float2int_rn(term[u] * 524288.0f));
                                acc += lane == (k & 31) ? ti : 0;
                            }
                        }
                    }
                    flush(K > 32 ? 32 : 0);
                };
                using std::true_type; using std::false_type;
                if (a.uniforms) {
                    if ((K & 3) == 0) draw_loop(false_type{}, true_type{}); else draw_loop(false_type{}, false_type{});
                } else {
                    if ((K & 3) == 0) draw_loop(true_type{}, true_type{}); else draw_loop(true_type{}, false_type{});
                }
            } else if (V <= 32) sample_frame(std::integral_constant<int, 32>{});
            else sample_frame(std::integral_constant<int, 64>{});
        }
        __syncthreads();
        if (!kStream && a.cdf_smem && a.samples) {         // (that path keeps the draw loop free of global stores)
            for (int i = threadIdx.x; i < K * T; i += kThreads) {
                const int k = i / T, tt = i - k * T;
                a.samples[((size_t)b * K + k) * T + tt] = samples_s[(size_t)k * Tp + tt];
            }
        }

        PGASR_STAMP(dbg, 32);
    }

    // ======== collapse ========
    for (int uu = 0; uu < nutt; ++uu) {
        const PgU X = pg_u(uu);
        const int b = X.b, Tb = X.Tb, m = X.m;
        uint8_t* const samples_s = X.samples_s; uint8_t* const hyp_s = X.hyp_s; uint8_t* const hrev_s = X.hrev_s;
        uint32_t* const peq = X.peq; uint32_t* const peq_r = X.peq_r; int16_t* const fg_s = X.fg_s;
        double* const warp_acc = X.warp_acc; float* const adv_s = X.adv_s; int* const hlen_s = X.hlen_s;
        int* const dist_s = X.dist_s; float* const misc_s = X.misc_s;
        const float* const lg = a.logits + (size_t)b * T * V;
        const int32_t* const ref = a.targets + (size_t)b * a.Lmax;
        const bool dbg = b == 0 && threadIdx.x == 0;
        (void)dbg; (void)samples_s; (void)hyp_s; (void)hrev_s; (void)peq; (void)peq_r; (void)fg_s; (void)warp_acc; (void)adv_s;
        (void)hlen_s; (void)dist_s; (void)misc_s; (void)lg; (void)ref; (void)Tb; (void)m;
        const int (&ref_r)[2] = ref_rr[uu];
        // ---- P2: collapse (one warp per sample) and the match table of the transcript ---------------
        if constexpr (kWord) {
            // word modes: the transcript as u8 ids for the word phase (0xFF: an id no hypothesis holds -- blank or
            // outside [0, V) -- its word matches nothing), and that phase's zeroed hashes and flags
            const WordRef R = word_ref_carve(wtail, uu, a.Lmax, wa.cap);
            auto map_id = [&](int c) { return (uint8_t)((c >= 0 && c < V && c != a.blank) ? c : 0xFF); };
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int j = threadIdx.x + q * kThreads;
                if (j < m) R.ref[j] = map_id(ref_r[q]);
            }
            for (int j = threadIdx.x + 2 * kThreads; j < m; j += kThreads) R.ref[j] = map_id(ref[j]);
            for (int j = threadIdx.x; j < a.Lmax + 2; j += kThreads) { R.hash[j] = 0u; R.cls[j] = 0; }
        } else {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int j = threadIdx.x + q * kThreads;
            const uint32_t c = (uint32_t)ref_r[q];
            if (j < m && c < (uint32_t)V) {
                atomicOr(&peq[c * W + (j >> 5)], 1u << (j & 31));
                const int jr = m - 1 - j;
                atomicOr(&peq_r[c * W + (jr >> 5)], 1u << (jr & 31));
            }
        }
        for (int j = threadIdx.x + 2 * kThreads; j < m; j += kThreads) {     // (Lmax > 2 * threads: never with Lmax <= 511)
            const uint32_t c = (uint32_t)ref[j];
            if (c < (uint32_t)V) {
                atomicOr(&peq[c * W + (j >> 5)], 1u << (j & 31));
                const int jr = m - 1 - j;
                atomicOr(&peq_r[c * W + (jr >> 5)], 1u << (jr & 31));
            }
        }
        }   // (character modes)
        for (int k = warp; k < K; k += kWarps) {
            const uint8_t* in = samples_s + (size_t)k * Tp;
            uint8_t* o = hyp_s + (size_t)k * Tp;
            int base = 0, carry = -1;
            for (int t0 = 0; t0 < Tb; t0 += 32) {
                const int t = t0 + lane;
                const int x = t < Tb ? (int)in[t] : -2;
                int p = __shfl_up_sync(kFull, x, 1);
                if (lane == 0) p = carry;
                const bool keep = t < Tb && x != p && x != a.blank;
                const unsigned mask = __ballot_sync(kFull, keep);
                if (keep) o[base + __popc(mask & ((1u << lane) - 1u))] = (uint8_t)x;
                base += __popc(mask);
                carry = __shfl_sync(kFull, x, 31);
            }
            if (lane == 0) hlen_s[k] = base;
            __syncwarp();
            if constexpr (!kWord) {                           // (word modes: the word phase writes the halves)
            uint8_t* orv = hrev_s + (size_t)k * Tp2;          // the edit distance meets in the middle: second half backwards
            for (int i = lane; i < base / 2; i += 32) orv[i] = o[base - 1 - i];
            }
        }
    }
    __syncthreads();

    // ======== word phase (word modes): transcripts into word classes and match tables, hypotheses into class ids ========
    if constexpr (kWord) {
        PGASR_STAMP(b0 == 0 && threadIdx.x == 0, 61);
        const unsigned lt = (1u << lane) - 1u;
        // W1, warp uu for utterance uu: split the transcript (word_split_warp: ballot over the separators, hashes by
        // shared-memory atomics), give every word whose ids a hypothesis can hold a class -- dense ids in the order of
        // first occurrence, a word equal to an earlier one takes that one's class (hash and length filter, then id by
        // id) -- and set its bit in the class's rows of the forward and the reversed match table
        if (warp < nutt) {
            const PgU X = pg_u(warp);
            const WordRef R = word_ref_carve(wtail, warp, a.Lmax, wa.cap);
            const int m = X.m;
            const int nw = word_split_warp(R.ref, m, wa.sep, R.start, R.hash, R.cls);   // (R.cls: 1 = bad word)
            if (lane == 0) R.start[0] = 0;
            __syncwarp();
            auto rlen = [&](int w) { return (w + 1 < nw ? (int)R.start[w + 1] - 1 : m) - (int)R.start[w]; };
            for (int w = lane; w < nw; w += 32) R.key[w] = ((uint64_t)rlen(w) << 32) | R.hash[w];
            __syncwarp();
            int ncls = 0;
            for (int w0 = 0; w0 < nw; w0 += 32) {
                const int w = w0 + lane;
                bool first = false;
                int rep = w, s0 = 0;
                uint64_t kw = 0u;
                if (w < nw && R.cls[w] == 0) {                // (each lane reads and writes only its own word's flag)
                    s0 = R.start[w]; kw = R.key[w];
                    const int len = (int)(kw >> 32);
                    first = true;
                    // the first equal word (a bad one never is: it holds 0xFF): equal key, then equal ids
                    for (int j = word_find_key(R.key, 0, w, kw); j < w; j = word_find_key(R.key, j + 1, w, kw)) {
                        const int sj = R.start[j];
                        bool eq = true;
                        for (int i = 0; i < len && eq; ++i) eq = R.ref[sj + i] == R.ref[s0 + i];
                        if (eq) { first = false; rep = j; break; }
                    }
                }
                const unsigned fm = __ballot_sync(kFull, first);
                const int c = ncls + __popc(fm & lt);
                if (first) { R.cstart[c] = (uint16_t)s0; R.ckey[c] = kw; }
                if (w < nw) { R.cls[w] = first ? (uint8_t)c : (uint8_t)0xFF; R.rep[w] = (uint16_t)rep; }
                ncls += __popc(fm);
            }
            __syncwarp();
            for (int w = lane; w < nw; w += 32) {             // repeated words: the class of their first occurrence
                const int j = R.rep[w];
                if (j != w) R.cls[w] = R.cls[j];
            }
            __syncwarp();
            for (int w = lane; w < nw; w += 32) {
                const uint32_t c = R.cls[w];
                if (c != 0xFFu) {
                    atomicOr(&X.peq[c * W + (w >> 5)], 1u << (w & 31));
                    const int wr = nw - 1 - w;
                    atomicOr(&X.peq_r[c * W + (wr >> 5)], 1u << (wr & 31));
                }
            }
            if (lane == 0) { reinterpret_cast<int*>(X.misc_s)[1] = nw; reinterpret_cast<int*>(X.misc_s)[2] = ncls; }
        }
        __syncthreads();
        PGASR_STAMP(b0 == 0 && threadIdx.x == 0, 62);
        // W2, one warp per sample: split the collapsed hypothesis, look every word up among the transcript's classes
        // (hash and length, then id by id; "absent" = the class count, the zero row of the tables), then write the class
        // ids over the sample's characters -- forwards into hyp_s, the second half reversed into hrev_s -- for P3
        {
            const int tw = word_hyp_slots(T);
            unsigned char* wp = wtail + (size_t)nutt * word_ref_bytes(a.Lmax, wa.cap) + (size_t)warp * word_warp_bytes(T);
            uint16_t* hstart = reinterpret_cast<uint16_t*>(wp);
            uint32_t* hhash = reinterpret_cast<uint32_t*>(wp + word_a16(2 * (size_t)tw));
            uint8_t* hid = wp + word_a16(2 * (size_t)tw) + 4 * (size_t)tw;
            for (int sidx = warp; sidx < nutt * K; sidx += kWarps) {
                const int uu = sidx / K, k = sidx - uu * K;
                const PgU X = pg_u(uu);
                const WordRef R = word_ref_carve(wtail, uu, a.Lmax, wa.cap);
                const int ncls = reinterpret_cast<const int*>(X.misc_s)[2];
                const int n = X.hlen_s[k];
                uint8_t* row = X.hyp_s + (size_t)k * Tp;
                for (int i = lane; i < tw; i += 32) hhash[i] = 0u;
                __syncwarp();
                const int nwh = word_split_warp(row, n, wa.sep, hstart, hhash, nullptr);
                if (lane == 0) hstart[0] = 0;
                __syncwarp();
                for (int w = lane; w < nwh; w += 32) {
                    const int s0 = hstart[w], len = (w + 1 < nwh ? (int)hstart[w + 1] - 1 : n) - s0;
                    const uint64_t kw = ((uint64_t)len << 32) | hhash[w];
                    int id = ncls;
                    for (int c = word_find_key(R.ckey, 0, ncls, kw); c < ncls; c = word_find_key(R.ckey, c + 1, ncls, kw)) {
                        const int cs = R.cstart[c];
                        bool eq = true;
                        for (int i = 0; i < len && eq; ++i) eq = R.ref[cs + i] == row[s0 + i];
                        if (eq) { id = c; break; }
                    }
                    hid[w] = (uint8_t)id;
                }
                __syncwarp();                                 // (every lane is done reading the characters)
                for (int i = lane; i < nwh; i += 32) row[i] = hid[i];
                const int n1 = myers_split_point(nwh);
                uint8_t* rv = X.hrev_s + (size_t)k * Tp2;
                for (int i = lane; i < nwh - n1; i += 32) rv[i] = hid[nwh - 1 - i];
                if (lane == 0) X.dist_s[k] = nwh;             // (P3 reads the word count here, then writes the distance)
                __syncwarp();
            }
        }
        __syncthreads();
    }

    PGASR_STAMP(b0 == 0 && threadIdx.x == 0, 33);
    // ======== edit distances: the utterances of the CTA side by side ========
    if (togo) {                                            // (one utterance per CTA in this mode)
        const int uu = 0;
        const PgU X = pg_u(uu);
        const int b = X.b, Tb = X.Tb, m = X.m;
        uint8_t* const samples_s = X.samples_s; uint8_t* const hyp_s = X.hyp_s; uint8_t* const hrev_s = X.hrev_s;
        uint32_t* const peq = X.peq; uint32_t* const peq_r = X.peq_r; int16_t* const fg_s = X.fg_s;
        double* const warp_acc = X.warp_acc; float* const adv_s = X.adv_s; int* const hlen_s = X.hlen_s;
        int* const dist_s = X.dist_s; float* const misc_s = X.misc_s;
        const float* const lg = a.logits + (size_t)b * T * V;
        const int32_t* const ref = a.targets + (size_t)b * a.Lmax;
        const bool dbg = b == 0 && threadIdx.x == 0;
        (void)dbg; (void)samples_s; (void)hyp_s; (void)hrev_s; (void)peq; (void)peq_r; (void)fg_s; (void)warp_acc; (void)adv_s;
        (void)hlen_s; (void)dist_s; (void)misc_s; (void)lg; (void)ref; (void)Tb; (void)m;
        // ---- P3 (reward-to-go): one thread per sample, the whole last column; then one warp per sample turns it into the
        // per-position rewards (output) and, in place, into the reward-to-go of every frame ----------------------------
        {
            if ((int)threadIdx.x < K) {
                const int k = threadIdx.x;
                dist_s[k] = myers_row<W, true, int16_t>(hyp_s + (size_t)k * Tp, hlen_s[k], peq, V, m, col_s + (size_t)k * Tc);
            }
            __syncthreads();
            for (int k = warp; k < K; k += kWarps) {
                int16_t* c = col_s + (size_t)k * Tc;
                const int n = hlen_s[k];
                const int cn = c[n];
                if (a.r_pos) {                                 // r_i = -(c[i+1] - c[i]), zero beyond the hypothesis
                    int8_t* rp = a.r_pos + ((size_t)b * K + k) * T;
                    for (int i = lane; i < T; i += 32) rp[i] = i < n ? (int8_t)(c[i] - c[i + 1]) : (int8_t)0;
                }
                __syncwarp();
                // G_t = c[pos(t)] - c[n], pos(t) = symbols emitted at frames < t; frames from the end towards the start so
                // that slot t can take G_t (every later read is at pos(t') <= t' < t)
                const uint8_t* in = samples_s + (size_t)k * Tp;
                const int nch = (T + 31) / 32;
                // emitted symbols before each chunk: one forward pass of ballots
                int before = 0;
                for (int ch = 0; ch < nch; ++ch) {
                    const int t = ch * 32 + lane;
                    const int x = t < Tb ? (int)in[t] : -2;
                    const int pv = t > 0 && t - 1 < Tb ? (int)in[t - 1] : -1;
                    const bool keep = t < Tb && x != pv && x != a.blank;
                    const unsigned mask = __ballot_sync(kFull, keep);
                    if (lane == 0) warp_acc_i[warp * 64 + (ch & 63)] = before;   // (T <= 2048: at most 64 chunks)
                    before += __popc(mask);
                }
                __syncwarp();
                for (int ch = nch - 1; ch >= 0; --ch) {
                    const int t = ch * 32 + lane;
                    const int x = t < Tb ? (int)in[t] : -2;
                    const int pv = t > 0 && t - 1 < Tb ? (int)in[t - 1] : -1;
                    const bool keep = t < Tb && x != pv && x != a.blank;
                    const unsigned mask = __ballot_sync(kFull, keep);
                    const int pos = warp_acc_i[warp * 64 + (ch & 63)] + __popc(mask & ((1u << lane) - 1u));
                    const int g = t < Tb ? (int)c[pos] - cn : 0;
                    __syncwarp();
                    if (t < T) {
                        c[t] = (int16_t)g;
                        if (a.to_go) a.to_go[((size_t)b * K + k) * T + t] = (int16_t)g;
                    }
                    __syncwarp();
                }
            }
            __syncthreads();
        }
    } else
    // ---- P3: edit distance, P lanes per sample ---------------------------------------------------
    // (all K samples in the lanes of as few warps as possible: a Myers step is a chain of dependent integer
    // instructions, and lanes of one warp share them; one sample per warp was measured 3.6x slower.  The words of a
    // sample are spread over P lanes that run one block apart, see myers_half)
    if constexpr (W >= 4) {
        // per utterance: forward halves on nw warps, backward halves on the next nw (myers_core.cuh, "Meeting in the
        // middle"); the utterances of the CTA next to each other when the warps suffice
        constexpr int P = 4;                              // lanes per sample
        const int nw = (K * P + 31) / 32;
        const bool bidir = 2 * nw <= kWarps;              // (K = 64 in the 256-thread variant: forward only, all of h)
        const int wpu = (bidir ? 2 : 1) * nw;             // warps per utterance
        const int ucon = nutt * wpu <= kWarps ? nutt : 1; // utterances side by side
        for (int u0 = 0; u0 < nutt; u0 += ucon) {
            uint32_t VPh[W / P], VNh[W / P];
            int k = 0, p = 0, n = 0, n1 = 0;
            const int uw = warp / wpu;                    // which of the concurrent utterances this warp serves
            const bool mine = uw < ucon;
            const int wl = warp - uw * wpu;               // warp within the utterance's group
            const PgU X = pg_u(u0 + (mine ? uw : 0));
            if (mine) {                                   // whole warps: the lanes shuffle with a full mask
                const bool fwd = wl < nw;
                const int tid = (wl - (fwd ? 0 : nw)) * 32 + lane;
                k = tid / P; p = tid % P;
                const int kc = min(k, K - 1);
                n = k < K ? (kWord ? X.dist_s : X.hlen_s)[kc] : 0;
                n1 = bidir ? myers_split_point(n) : n;
                const int nsym = fwd ? n1 : n - n1;
                const int nmax = __reduce_max_sync(kFull, nsym);
                myers_half<W, P, false>(fwd ? X.hyp_s + (size_t)kc * Tp : X.hrev_s + (size_t)kc * Tp2, nsym, fwd ? X.peq : X.peq_r,
                                        kWord ? reinterpret_cast<const int*>(X.misc_s)[2] : V, p, nmax, VPh, VNh);
                if (!fwd) myers_store_column<W, P>(VPh, VNh, n - n1, p, X.fg_s + (size_t)k * (W * 32 + 2));
            }
            __syncthreads();
            if (mine && wl < nw) {
                const int mq = kWord ? reinterpret_cast<const int*>(X.misc_s)[1] : X.m;   // (word modes: n_w)
                int d;
                if (bidir) {
                    d = myers_meet<W, P>(VPh, VNh, n1, mq, p, X.fg_s + (size_t)k * (W * 32 + 2));
                } else {                                  // dp[n, m] = n + sum_{j<m} (VP_j - VN_j)
                    d = 0;
#pragma unroll
                    for (int w = 0; w < W / P; ++w) {
                        const int lo = (p * (W / P) + w) * 32;
                        const uint32_t msk = mq >= lo + 32 ? 0xffffffffu : (mq > lo ? (1u << (mq - lo)) - 1u : 0u);
                        d += __popc(VPh[w] & msk) - __popc(VNh[w] & msk);
                    }
#pragma unroll
                    for (int o = 1; o < P; o <<= 1) d += __shfl_xor_sync(kFull, d, o);
                    d += n;
                }
                if (k < K && p == 0) X.dist_s[k] = d;
            }
        }
    } else {                                              // two words: one thread per sample is as fast (measured)
        if ((int)threadIdx.x < nutt * K) {
            const PgU X = pg_u((int)threadIdx.x / K);
            const int k = (int)threadIdx.x % K;
            if constexpr (kWord) {
                const int* wi = reinterpret_cast<const int*>(X.misc_s);
                X.dist_s[k] = myers_row<W, false>(X.hyp_s + (size_t)k * Tp, X.dist_s[k], X.peq, wi[2], wi[1], static_cast<int32_t*>(nullptr));
            } else
            X.dist_s[k] = myers_row<W, false>(X.hyp_s + (size_t)k * Tp, X.hlen_s[k], X.peq, V, X.m, static_cast<int32_t*>(nullptr));
        }
    }
    __syncthreads();

    // ======== rewards, baseline, advantages, loss terms: warp uu for utterance uu ========
    if (warp < nutt) {
        const int uu = warp;
        const PgU X = pg_u(uu);
        const int b = X.b, Tb = X.Tb, m = X.m;
        uint8_t* const samples_s = X.samples_s; uint8_t* const hyp_s = X.hyp_s; uint8_t* const hrev_s = X.hrev_s;
        uint32_t* const peq = X.peq; uint32_t* const peq_r = X.peq_r; int16_t* const fg_s = X.fg_s;
        double* const warp_acc = X.warp_acc; float* const adv_s = X.adv_s; int* const hlen_s = X.hlen_s;
        int* const dist_s = X.dist_s; float* const misc_s = X.misc_s;
        const float* const lg = a.logits + (size_t)b * T * V;
        const int32_t* const ref = a.targets + (size_t)b * a.Lmax;
        const bool dbg = b == 0 && threadIdx.x == 0;
        (void)dbg; (void)samples_s; (void)hyp_s; (void)hrev_s; (void)peq; (void)peq_r; (void)fg_s; (void)warp_acc; (void)adv_s;
        (void)hlen_s; (void)dist_s; (void)misc_s; (void)lg; (void)ref; (void)Tb; (void)m;
        PGASR_STAMP(dbg, 34);
        // ---- P4: rewards, baseline, advantages, loss term (warp 0) -----------------------------------
        {
            // rewards are fp32 by contract (bit exact with the oracle); baseline, advantage and the loss term are fp64:
            // an fp32 rounding of A (1e-7 relative) times log p ~ -1000 would already show in the scalar loss
            double sumR = 0.0;
            for (int k = lane; k < K; k += 32) {
                float R = -(float)dist_s[k];
                if (a.reward_mode == PGASR_REWARD_NEG_CER) R = __fdiv_rn(R, (float)m);
                if constexpr (kWord) {                        // -ED_w / n_w, the WER ratio
                    if (a.reward_mode == PGASR_REWARD_NEG_WER) R = __fdiv_rn(R, (float)reinterpret_cast<const int*>(misc_s)[1]);
                }
                if (togo) R = (float)(m - dist_s[k]);         // G_0 = c[0] - c[n]: what the whole hypothesis earned
                adv_s[k] = R;
                sumR += (double)R;
            }
            sumR = warp_sum(sumR);
            double term = 0.0;
            float sumA = 0.0f;
            for (int k = lane; k < K; k += 32) {
                const float R = adv_s[k];
                double base = 0.0;
                if (a.baseline_mode == PGASR_BASELINE_MEAN) base = sumR / (double)K;
                else if (a.baseline_mode == PGASR_BASELINE_LOO) base = K > 1 ? (sumR - (double)R) / (double)(K - 1) : 0.0;
                else if (a.baseline_mode == PGASR_BASELINE_VALUE) base = (double)a.baseline_value;
                const double Ad = (double)R - base;
                const float A = (float)Ad;
                double lp = 0.0;
                for (int w = 0; w < kWarps; ++w) lp += warp_acc[w * kFusedMaxK + k];
                term += -Ad * lp;
                sumA += A;
                adv_s[k] = A;
                const size_t o = (size_t)b * K + k;
                if (a.rewards) a.rewards[o] = R;
                if (a.logp) a.logp[o] = (float)lp;
                if (a.hyp_len) a.hyp_len[o] = hlen_s[k];
                if (a.dist) a.dist[o] = dist_s[k];
            }
            term = warp_sum(term);
            sumA = warp_sum(sumA);
            if (lane == 0 && !togo) {                         // (reward-to-go: advantages are per frame, the loss term comes from P5)
                a.loss_terms[b] = (float)term;
                misc_s[0] = sumA;
            }
        }
    }
    __syncthreads();

    // ======== gradient tiles and their way into dlogits, the utterance sampled last first (its logits are still in
    // the tile buffer; an earlier one's are reloaded when the dense term needs them) ========
    for (int uu = nutt - 1; uu >= 0; --uu) {
        const PgU X = pg_u(uu);
        const int b = X.b, Tb = X.Tb, m = X.m;
        uint8_t* const samples_s = X.samples_s; uint8_t* const hyp_s = X.hyp_s; uint8_t* const hrev_s = X.hrev_s;
        uint32_t* const peq = X.peq; uint32_t* const peq_r = X.peq_r; int16_t* const fg_s = X.fg_s;
        double* const warp_acc = X.warp_acc; float* const adv_s = X.adv_s; int* const hlen_s = X.hlen_s;
        int* const dist_s = X.dist_s; float* const misc_s = X.misc_s;
        const float* const lg = a.logits + (size_t)b * T * V;
        const int32_t* const ref = a.targets + (size_t)b * a.Lmax;
        const bool dbg = b == 0 && threadIdx.x == 0;
        (void)dbg; (void)samples_s; (void)hyp_s; (void)hrev_s; (void)peq; (void)peq_r; (void)fg_s; (void)warp_acc; (void)adv_s;
        (void)hlen_s; (void)dist_s; (void)misc_s; (void)lg; (void)ref; (void)Tb; (void)m;
        PGASR_STAMP(dbg, 35);
        const bool dense = a.baseline_mode != PGASR_BASELINE_MEAN;   // sum_k A_k == 0 under the per-utterance mean
        // exploration: the entropy term (or its output) needs the dense softmax under every baseline
        const bool ent = kExp && (px.x.ent_c != 0.0f || px.x.entropy != nullptr);
        if (!kStream && uu != nutt - 1) {
            if (dense || ent) {                            // (the tile holds the previous utterance's gradient)
                if (a.bulk_tile) {
                    if (threadIdx.x == 0) bulk_load_tile(ztile, lg, (unsigned)((size_t)T * V * 4), s_mbar);
                    mbar_wait(s_mbar, nload++ & 1u);
                } else {
                    for (int i = threadIdx.x; i < T * V; i += kThreads) ztile[i] = __ldg(lg + i);
                }
                if constexpr (kExp) {
                    if (theta != 1.0f) {
                        __syncthreads();
                        scale_tile<kThreads>(ztile, T * V, theta);
                    }
                }
            }
            __syncthreads();
        }
        // ---- P5: REINFORCE gradient tile, in place of the logits tile ---------------------------------
        // (exploration: times theta, the chain factor of z' = theta z)
        const float coef = kExp ? __fmul_rn(a.w_pg / ((float)a.B * (float)K), theta) : a.w_pg / ((float)a.B * (float)K);
        const float ent_c = kExp ? __fmul_rn(px.x.ent_c, theta) : 0.0f;
        double hsum = 0.0;                                     // exploration: this thread's frames' H_bt
        (void)ent_c; (void)hsum;
        // exploration: the gradient row of a frame from its z' row (in place): theta (coef sum_k A_k p' [dense] +
        // (beta / B) p' (log p' + H_t)) -- the sample terms follow; returns H_t
        auto explore_row = [&](float* row, float lz, float dcoef) {
            float H = 0.0f;
            for (int v = 0; v < V; ++v) {
                const float lp = row[v] - lz;                  // log p' = z' - m' - ln S, never log(p')
                H -= ent_plogp(__expf(lp), lp);
            }
            for (int v = 0; v < V; ++v) {
                const float lp = row[v] - lz, p = __expf(lp);
                row[v] = ent_grad(p, dcoef + (ent ? ent_c * (lp + H) : 0.0f));
            }
            return H;
        };
        (void)explore_row;
        // exploration: H_b = sum of the frames' H_t in a fixed order (threads -> warps -> warp 0..), the entropy output,
        // and - beta K / w_pg H_b folded into the utterance's loss term (the loss then carries -beta / B sum_b H_b).  The
        // loss term must be final before this CTA draws its done ticket.
        auto explore_finish = [&]() {
            hsum = warp_sum(hsum);
            if (lane == 0) warp_acc[32 + warp] = hsum;     // (P4 has consumed the log-prob partial sums)
            __syncthreads();
            if (threadIdx.x == 0) {
                double H = 0.0;
                for (int w = 0; w < kWarps; ++w) H += warp_acc[32 + w];
                if (px.x.entropy) px.x.entropy[b] = (float)H;
                if (px.x.ent_lt != 0.0f) a.loss_terms[b] = (float)((double)a.loss_terms[b] - (double)px.x.ent_lt * H);
            }
        };
        (void)explore_finish;
        const float dense_c = coef * misc_s[0];
        float* dlog_u = a.dlogits + (size_t)b * T * V;
        const bool final_u = uu == 0;                          // the last utterance this CTA finishes: it draws the done ticket
        if constexpr (kStream) {
            // one thread per frame: the K sample ids into registers, then for every class the advantage mass that fell
            // on it; the row is added to (or, without a CTC term, stored as) dlogits directly
            if (threadIdx.x == 0) {
                if (a.do_ctc) {
                    const unsigned* flag = a.ctrl + 4 + b;
                    while (ld_acquire(flag) == 0u) __nanosleep(40);
                }
                if (final_u && !ent) draw_done_ticket(a, s_last);
            }
            __syncthreads();
            PGASR_STAMP(dbg, 37);
            for (int t = threadIdx.x; t < T; t += kThreads) {
                float* out = dlog_u + (size_t)t * V;
                if (t >= Tb) {
                    if (!a.do_ctc)
                        for (int v = 0; v < V; ++v) out[v] = 0.0f;
                    continue;
                }
                float mx = 0.0f, sc = 0.0f, lz = 0.0f, H = 0.0f;
                const float* zr = lg + (size_t)t * V;
                if (dense || ent) {
                    mx = -INFINITY;
                    float ssum = 0.0f;
                    for (int v = 0; v < V; ++v) mx = fmaxf(mx, zv(zr, v));
                    for (int v = 0; v < V; ++v) ssum += __expf(zv(zr, v) - mx);
                    sc = dense_c / ssum;
                    if (ent) {                                 // H_t = -sum_v p' log p', log p' = z' - m' - ln S
                        lz = mx + logf(ssum);
                        for (int v = 0; v < V; ++v) {
                            const float lp = zv(zr, v) - lz;
                            H -= ent_plogp(__expf(lp), lp);
                        }
                        hsum += (double)H;
                    }
                }
                for (int v = 0; v < V; ++v) {
                    float g;
                    if (ent) {
                        const float lp = zv(zr, v) - lz;
                        g = ent_grad(__expf(lp), (dense ? dense_c : 0.0f) + ent_c * (lp + H));
                    } else {
                        g = dense ? __expf(zv(zr, v) - mx) * sc : 0.0f;
                    }
                    for (int k = 0; k < K; ++k)              // same order of subtractions as the tile mode: k ascending
                        if (samples_s[(size_t)k * Tp + t] == v) g -= coef * adv_s[k];
                    out[v] = a.do_ctc ? __ldcg(out + v) + g : g;
                }
            }
            if constexpr (kExp) {
                if (ent) {                                     // (the ticket after the loss term is final)
                    explore_finish();
                    if (threadIdx.x == 0 && final_u) draw_done_ticket(a, s_last);
                }
            }
            PGASR_STAMP(dbg, 38);
        } else {
        if (togo) {
            // per-frame advantages A_kt = G_kt - b_kt (baseline over the K samples of the frame), the loss term
            // -sum_kt A_kt log p_t(pi_kt) and the gradient row (1/BK) (p_tv sum_k A_kt - sum_k A_kt [pi_kt = v])
            double lt = 0.0;
            for (int t = threadIdx.x; t < T; t += kThreads) {
                float* row = ztile + (size_t)t * V;
                if (t < Tb) {
                    const float lz = lz_s[t];
                    int sumGi = 0;
                    for (int k = 0; k < K; ++k) sumGi += (int)col_s[(size_t)k * Tc + t];
                    const float sumG = (float)sumGi;
                    auto adv_of = [&](int k) {
                        const float G = (float)col_s[(size_t)k * Tc + t];
                        float base = 0.0f;
                        if (a.baseline_mode == PGASR_BASELINE_MEAN) base = sumG / (float)K;
                        else if (a.baseline_mode == PGASR_BASELINE_LOO) base = K > 1 ? (sumG - G) / (float)(K - 1) : 0.0f;
                        else if (a.baseline_mode == PGASR_BASELINE_VALUE) base = a.baseline_value;
                        return G - base;
                    };
                    float sumA = 0.0f;
                    for (int k = 0; k < K; ++k) {
                        const float A = adv_of(k);
                        lt += -(double)A * (double)(row[samples_s[(size_t)k * Tp + t]] - lz);
                        sumA += A;
                    }
                    if (ent) {
                        hsum += (double)explore_row(row, lz, dense ? coef * sumA : 0.0f);
                    } else if (dense) {
                        const float sc = coef * sumA;
                        for (int v = 0; v < V; ++v) row[v] = __expf(row[v] - lz) * sc;
                    } else {
                        for (int v = 0; v < V; ++v) row[v] = 0.0f;
                    }
                    for (int k = 0; k < K; ++k) row[samples_s[(size_t)k * Tp + t]] -= coef * adv_of(k);
                } else {
                    for (int v = 0; v < V; ++v) row[v] = 0.0f;
                }
            }
            lt = warp_sum(lt);
            __syncthreads();                                   // (warp_acc: the log-prob partial sums are consumed)
            if (lane == 0) warp_acc[warp] = lt;
            __syncthreads();
            if (threadIdx.x == 0) {
                double tot = 0.0;
                for (int w = 0; w < kWarps; ++w) tot += warp_acc[w];
                a.loss_terms[b] = (float)tot;
            }
        } else
        for (int t = threadIdx.x; t < T; t += kThreads) {
            float* row = ztile + (size_t)t * V;
            if (t < Tb) {
                if (ent) {
                    float mx = -INFINITY, s = 0.0f;
                    for (int v = 0; v < V; ++v) mx = fmaxf(mx, row[v]);
                    for (int v = 0; v < V; ++v) s += __expf(row[v] - mx);
                    hsum += (double)explore_row(row, mx + logf(s), dense ? dense_c : 0.0f);
                } else if (dense) {
                    float mx = -INFINITY, s = 0.0f;
                    for (int v = 0; v < V; ++v) mx = fmaxf(mx, row[v]);
                    for (int v = 0; v < V; ++v) s += __expf(row[v] - mx);
                    const float sc = dense_c / s;
                    for (int v = 0; v < V; ++v) row[v] = __expf(row[v] - mx) * sc;
                } else {
                    for (int v = 0; v < V; ++v) row[v] = 0.0f;
                }
                for (int k = 0; k < K; ++k) row[samples_s[(size_t)k * Tp + t]] -= coef * adv_s[k];
            } else {
                for (int v = 0; v < V; ++v) row[v] = 0.0f;
            }
        }
        __syncthreads();
        if constexpr (kExp) {
            if (ent) explore_finish();                     // (thread 0 draws the done ticket below, after this)
        }

        PGASR_STAMP(dbg, 36);
        // ---- P6: add the tile onto the CTC rows (or store it when there is no CTC term) ---------------
        if (threadIdx.x == 0) {
            if (a.do_ctc) {
                const unsigned* flag = a.ctrl + 4 + b;
#ifdef PGASR_TIMING
                const unsigned long long f0 = gtime();
#endif
                while (ld_acquire(flag) == 0u) __nanosleep(40);
#ifdef PGASR_TIMING
                atomicAdd(&g_role_ns[1][3], gtime() - f0);
#endif
            }
            if (final_u) draw_done_ticket(a, s_last);
        }
        __syncthreads();
        PGASR_STAMP(dbg, 37);
        if (((reinterpret_cast<uintptr_t>(dlog_u) | ((size_t)T * V * 4)) & 15) == 0) {   // (dlogits: any float*)
            float4* d4 = reinterpret_cast<float4*>(dlog_u);
            const float4* t4 = reinterpret_cast<const float4*>(ztile);
            const int n4 = T * V / 4;
            // In the CTA that drew the last ticket the last warp reduces the loss (three dependent L2 round trips) while
            // the other warps share the pass among themselves, instead of after it.
            const bool last = final_u && *s_last != 0u;
            const int nt = last ? kThreads - 32 : kThreads;
            if (last && warp == kWarps - 1) {
                loss_reduce_and_rearm(a);
            } else if (a.do_ctc) {
                // eight L2 reads in flight per thread (one at a time, every pass waited out the full L2 latency)
                for (int i0 = threadIdx.x; i0 < n4; i0 += 8 * nt) {
                    float4 c[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int i = i0 + u * nt;
                        c[u] = i < n4 ? __ldcg(d4 + i) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int i = i0 + u * nt;
                        if (i < n4) {
                            const float4 g = t4[i];
                            d4[i] = make_float4(g.x + c[u].x, g.y + c[u].y, g.z + c[u].z, g.w + c[u].w);
                        }
                    }
                }
            } else {
                for (int i = threadIdx.x; i < n4; i += nt) d4[i] = t4[i];
            }
        } else {
            if (final_u && *s_last != 0u && warp == kWarps - 1) loss_reduce_and_rearm(a);    // (then it joins the pass)
            for (int i = threadIdx.x; i < T * V; i += kThreads)
                dlog_u[i] = a.do_ctc ? __ldcg(dlog_u + i) + ztile[i] : ztile[i];
        }
        PGASR_STAMP(dbg, 38);
        }   // tile mode
        __syncthreads();                                   // (the next utterance rewrites the tile)
    }
}


template <int SPL, int kThreads, bool kGT, bool kStream, bool kBW = false>
__global__ void __launch_bounds__(kThreads, 1) pg_ctc_fused_kernel(const FusedArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned s_ticket, s_last;
#ifdef PGASR_TIMING
    __shared__ long long s_clk[2];                          // clock64 at CTA start and after the grid-dependency wait
    if (threadIdx.x == 0) s_clk[0] = clock64();
#endif
    __shared__ __align__(8) unsigned long long s_mbar;      // completion of the bulk tile load (a.bulk_tile)
    if (threadIdx.x == 0 && a.bulk_tile) {
        mbar_init(&s_mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
#ifdef PGASR_TIMING
    const unsigned long long t_start = gtime();
#endif
    if (threadIdx.x == 0) s_ticket = atomicAdd(a.ctrl, 1u);
    __syncthreads();
    // Programmatic dependent launch: everything above (CTA start, role ticket on this step's own control block)
    // overlaps the tail of the previous kernel in the stream; nothing below may touch global memory before that kernel
    // has completed and flushed.  The next launch may start as soon as every CTA of this grid got here.
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
#ifdef PGASR_TIMING
    const unsigned long long t_go = gtime();
    if (threadIdx.x == 0) s_clk[1] = clock64();
    if (threadIdx.x == 0 && s_ticket == 0) { g_dbg[4] = s_clk[0]; g_dbg[5] = s_clk[1]; }
#endif
    const unsigned ticket = s_ticket;
    const unsigned n_ctc = a.do_ctc ? (unsigned)a.B : 0u;
    if (ticket < n_ctc) fused_ctc_role<SPL, kThreads, kGT, kBW>(a, (int)ticket, smem_raw, &s_last, &s_mbar);
    else {
        // a PG CTA serves one utterance, or two (a.pg_pair: utterances 2j and 2j + 1)
        const int j = (int)(ticket - n_ctc);
        const int b0 = a.pg_pair ? 2 * j : j;
        fused_pg_role<SPL / 2, kThreads, kStream>(a, b0, a.pg_pair ? min(2, a.B - b0) : 1, smem_raw, &s_last, &s_mbar);
    }

#ifdef PGASR_TIMING
    if (threadIdx.x == 0 && ticket < 2048) { g_cta_ns[ticket][0] = t_start; g_cta_ns[ticket][1] = gtime(); }
#endif
    // ---- the CTA that drew the last second ticket (draw_done_ticket, inside the roles) reduces the loss in a fixed
    // order and re-arms the control block; the rows of dlogits are published by the kernel boundary ----
    // (a PG CTA with its tile in shared memory has done that already, next to its read-modify-write pass)
    __syncthreads();
    if (s_last && threadIdx.x < 32 && (ticket < n_ctc || kStream)) loss_reduce_and_rearm(a);
#ifdef PGASR_TIMING
    if (threadIdx.x == 0 && ticket == 0) g_dbg[8] = clock64();
    if (threadIdx.x == 0 && ticket < 2048) g_cta_ns[ticket][2] = gtime();
    if (threadIdx.x == 0) {
        const int role = ticket < n_ctc ? 0 : 1;
        atomicAdd(&g_role_ns[role][0], 1ull);
        atomicAdd(&g_role_ns[role][1], t_go - t_start);
        atomicAdd(&g_role_ns[role][2], gtime() - t_go);
    }
#endif
}

// word-level rewards (tile mode: the PG role keeps the logits tile in shared memory): the kernel above with the word
// phase in its PG role (fused_pg_role<..., true>); same ticket protocol, no timing stamps
template <int SPL, int kThreads, bool kGT, bool kBW>
__global__ void __launch_bounds__(kThreads, 1) pg_ctc_fused_word_kernel(const FusedArgs a, const WordArgs wa) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned s_ticket, s_last;
    __shared__ __align__(8) unsigned long long s_mbar;
    if (threadIdx.x == 0 && a.bulk_tile) {
        mbar_init(&s_mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (threadIdx.x == 0) s_ticket = atomicAdd(a.ctrl, 1u);
    __syncthreads();
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    const unsigned ticket = s_ticket;
    const unsigned n_ctc = a.do_ctc ? (unsigned)a.B : 0u;
    if (ticket < n_ctc) fused_ctc_role<SPL, kThreads, kGT, kBW>(a, (int)ticket, smem_raw, &s_last, &s_mbar);
    else {
        const int j = (int)(ticket - n_ctc);
        const int b0 = a.pg_pair ? 2 * j : j;
        fused_pg_role<SPL / 2, kThreads, false, true>(a, b0, a.pg_pair ? min(2, a.B - b0) : 1, smem_raw, &s_last, &s_mbar,
                                                      wa);
    }
    __syncthreads();
    if (s_last && threadIdx.x < 32 && ticket < n_ctc) loss_reduce_and_rearm(a);
}

// exploration (temperature / entropy bonus, character or word modes): the kernels above with the exploration variant of
// the PG role (fused_pg_role<..., kExp = true>); same ticket protocol, no timing stamps
template <int SPL, int kThreads, bool kGT, bool kStream, bool kBW, bool kWord>
__global__ void __launch_bounds__(kThreads, 1) pg_ctc_fused_explore_kernel(const FusedArgs a, const WordArgs wa,
                                                                           const ExploreArgs x) {
    static_assert(!(kWord && kStream), "the streaming PG role has no word phase");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned s_ticket, s_last;
    __shared__ __align__(8) unsigned long long s_mbar;
    if (threadIdx.x == 0 && a.bulk_tile) {
        mbar_init(&s_mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (threadIdx.x == 0) s_ticket = atomicAdd(a.ctrl, 1u);
    __syncthreads();
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    const unsigned ticket = s_ticket;
    const unsigned n_ctc = a.do_ctc ? (unsigned)a.B : 0u;
    if (ticket < n_ctc) fused_ctc_role<SPL, kThreads, kGT, kBW>(a, (int)ticket, smem_raw, &s_last, &s_mbar);
    else {
        const int j = (int)(ticket - n_ctc);
        const int b0 = a.pg_pair ? 2 * j : j;
        const int nutt = a.pg_pair ? min(2, a.B - b0) : 1;
        if constexpr (kWord)
            fused_pg_role<SPL / 2, kThreads, false, true, true>(a, b0, nutt, smem_raw, &s_last, &s_mbar, wa, x);
        else
            fused_pg_role<SPL / 2, kThreads, kStream, false, true>(a, b0, nutt, smem_raw, &s_last, &s_mbar, x);
    }
    __syncthreads();
    if (s_last && threadIdx.x < 32 && (ticket < n_ctc || kStream)) loss_reduce_and_rearm(a);
}

// the dynamic shared-memory opt-in of `kern`: sticky PER DEVICE, raised only when a larger tile comes on the device the
// launch goes to (smem_set: one per kernel)
template <typename Kern>
static int fused_smem_optin(Kern kern, size_t (&smem_set)[64], size_t smem) {
    int dev = 0;
    PGASR_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || smem > smem_set[dev]) {
        PGASR_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (dev >= 0 && dev < 64) smem_set[dev] = smem;
    }
    return PGASR_OK;
}

template <int SPL, int kThreads, bool kGT, bool kStream, bool kBW, bool kWord>
static int launch_fused_explore(FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word, const ExploreArgs& x,
                                cudaLaunchConfig_t& cfg) {
    static thread_local size_t smem_set[64] = {0};
    const auto kern = pg_ctc_fused_explore_kernel<SPL, kThreads, kGT, kStream, kBW, kWord>;
    const int rc = fused_smem_optin(kern, smem_set, smem);
    if (rc) return rc;
    const WordArgs wa = word ? *word : WordArgs{-1, 0};
    PGASR_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, a, wa, x));
    ++g_launches;
    return PGASR_OK;
}

template <int SPL, int kThreads, bool kGT, bool kStream, bool kBW = false>
static int launch_fused(FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word = nullptr,
                        const ExploreArgs* explore = nullptr) {
    static thread_local size_t smem_set[64] = {0};
    static thread_local size_t smem_set_w[64] = {0};
    if constexpr (!kStream) {
        if (word && !explore) {
            const int rc = fused_smem_optin(pg_ctc_fused_word_kernel<SPL, kThreads, kGT, kBW>, smem_set_w, smem);
            if (rc) return rc;
        }
    }
    if (!word && !explore) {
        const int rc = fused_smem_optin(pg_ctc_fused_kernel<SPL, kThreads, kGT, kStream, kBW>, smem_set, smem);
        if (rc) return rc;
    }
    const int grid = (a.do_ctc ? a.B : 0) + (a.do_pg ? (a.pg_pair ? (a.B + 1) / 2 : a.B) : 0);
    static const bool no_pdl = getenv("PGASR_NO_PDL") != nullptr;     // (A/B measurements)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (no_pdl || a.no_pdl) ? 0 : 1;
    if (explore) {
        if constexpr (!kStream) {
            if (word) return launch_fused_explore<SPL, kThreads, kGT, kStream, kBW, true>(a, smem, st, word, *explore, cfg);
        }
        if (word) return PGASR_ERR_UNSUPPORTED;
        return launch_fused_explore<SPL, kThreads, kGT, kStream, kBW, false>(a, smem, st, word, *explore, cfg);
    }
    if constexpr (!kStream) {
        if (word) {
            PGASR_CUDA_TRY(cudaLaunchKernelEx(&cfg, pg_ctc_fused_word_kernel<SPL, kThreads, kGT, kBW>, a, *word));
            ++g_launches;
            return PGASR_OK;
        }
    }
    if (word) return PGASR_ERR_UNSUPPORTED;
    PGASR_CUDA_TRY(cudaLaunchKernelEx(&cfg, pg_ctc_fused_kernel<SPL, kThreads, kGT, kStream, kBW>, a));
    ++g_launches;
    return PGASR_OK;
}

// one translation unit per SPL instantiates its modes (0: tiles in shared memory, 1: the CTC role streams,
// 2: both roles stream, 3: tiles in shared memory with block workers -- up to 8 states per lane only) so that the
// variants compile in parallel
// word (non-NULL): the word-mode kernel, modes 0, 1 and 3 (the PG role keeps its tile in shared memory)
// explore (non-NULL): the exploration variant of either
template <int SPL, int kThreads>
int launch_fused_modes(int mode, FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word,
                       const ExploreArgs* explore) {
    if constexpr (SPL <= 8) {
        if (mode == 3) return launch_fused<SPL, kThreads, false, false, true>(a, smem, st, word, explore);
    }
    switch (mode) {
        case 0: return launch_fused<SPL, kThreads, false, false>(a, smem, st, word, explore);
        case 1: return launch_fused<SPL, kThreads, true, false>(a, smem, st, word, explore);
        default: return launch_fused<SPL, kThreads, true, true>(a, smem, st, word, explore);
    }
}

}  // namespace pgasr
