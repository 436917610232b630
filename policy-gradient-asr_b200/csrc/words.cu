// Word edit distance (DESIGN.md "word reward spec"; upstream metrics.py:23-31 evaluate: WER = edit_dist over
// s.split(" ")): the rows of pgasr_edit_distance_u8 split into words at the separator id, then the Levenshtein
// distance over the word sequences.  The stand-alone kernel of the step's chain path (shapes whose samples do not fit
// an SM); the single-launch step has its own word phase (fused_impl.cuh).
//
// One CTA per reference: warp 0 splits the transcript, every thread gives one of its words its class (the index of
// the first equal word), the match table is built over the classes.  Then one warp per hypothesis row splits the row,
// its lanes look their words up among the transcript's classes (length and hash first, then id by id), and lane 0
// runs the bit-parallel recurrence (myers_core.cuh) over the word classes.
#include "myers_core.cuh"
#include "words_core.cuh"

namespace pgasr {

struct WordEdSmem { size_t ref, rstart, rhash, rcls, peq, fixed, per_warp; };   // (rcls: bad flag, then class: 2 arrays)
__host__ __device__ inline WordEdSmem word_ed_smem(int W, int ref_stride, int hyp_stride) {
    WordEdSmem s;
    const size_t nw = (size_t)ref_stride + 2;
    s.ref = word_a16((size_t)ref_stride);                   // ids as u8 (an id outside [0, 256) makes its word bad)
    s.rstart = word_a16(4 * nw);
    s.rhash = word_a16(4 * nw);
    s.rcls = 2 * word_a16(4 * nw);
    s.peq = (size_t)(nw + 1) * W * 4;
    s.fixed = s.ref + s.rstart + s.rhash + s.rcls + s.peq;
    s.per_warp = 3 * word_a16(4 * ((size_t)hyp_stride + 2));      // word starts, hashes, classes (int32 each)
    return s;
}

template <int W>
__global__ void word_ed_u8_kernel(const uint8_t* __restrict__ hyps, const int32_t* __restrict__ hyp_len, int N,
                                  int hyp_stride, const int32_t* __restrict__ refs, const int32_t* __restrict__ ref_len,
                                  int rows_per_ref, int ref_stride, int sep, int32_t* __restrict__ dist,
                                  int32_t* __restrict__ ref_words) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    const WordEdSmem L = word_ed_smem(W, ref_stride, hyp_stride);
    unsigned char* p = sm_raw;
    uint8_t* rtok = p;                                  p += L.ref;
    int32_t* rstart = reinterpret_cast<int32_t*>(p);    p += L.rstart;
    uint32_t* rhash = reinterpret_cast<uint32_t*>(p);   p += L.rhash;
    int32_t* rcls = reinterpret_cast<int32_t*>(p);      p += L.rcls / 2;   // -1: bad word
    int32_t* rclass = reinterpret_cast<int32_t*>(p);    p += L.rcls / 2;   // the first word equal to it
    uint32_t* peq = reinterpret_cast<uint32_t*>(p);     p += L.peq;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int g = blockIdx.x;
    int m = ref_len ? ref_len[g] : ref_stride;
    m = min(max(m, 0), ref_stride);
    const int32_t* ref = refs + (size_t)g * ref_stride;
    // the transcript as u8: a word holding an id outside [0, 256) equals no word of a hypothesis row ("bad": it gets no
    // class, its column never matches)
    for (int j = threadIdx.x; j < m; j += blockDim.x) rtok[j] = (uint8_t)ref[j];
    for (int j = threadIdx.x; j < ref_stride + 2; j += blockDim.x) { rhash[j] = 0u; rcls[j] = 0; }
    __syncthreads();
    // warp 0: split the transcript (ids equal to sep are the separators; sep may be >= 255: then there are none in the
    // hypotheses, but the transcript still splits at its own)
    __shared__ int s_nw;
    if (warp == 0) {
        int wbase = 0, open = 0;
        for (int t0 = 0; t0 < m; t0 += 32) {
            const int t = t0 + lane;
            const bool live = t < m;
            const int32_t c = live ? ref[t] : 0;
            const bool is_sep = live && c == sep;
            const unsigned smk = __ballot_sync(kFull, is_sep);
            const int wi = wbase + __popc(smk & lt);
            const unsigned below = smk & lt;
            const int st = below ? t0 + (31 - __clz(below)) + 1 : open;
            if (is_sep) rstart[wi + 1] = t + 1;
            else if (live) {
                atomicAdd(rhash + wi, word_mix((uint32_t)c & 0xFFu, (uint32_t)(t - st)));
                if (c < 0 || c > 255) rcls[wi] = -1;       // (bad word)
            }
            if (smk) open = t0 + (31 - __clz(smk)) + 1;
            wbase += __popc(smk);
        }
        if (lane == 0) { rstart[0] = 0; s_nw = wbase + 1; }
    }
    __syncthreads();
    const int nwr = s_nw;
    auto rlen = [&](int w) { return (w + 1 < nwr ? rstart[w + 1] - 1 : m) - rstart[w]; };
    // class of every transcript word: the first word equal to it (a bad word is its own class and matches nothing)
    for (int i = threadIdx.x; i < (nwr + 1) * W; i += blockDim.x) peq[i] = 0u;
    for (int w = threadIdx.x; w < nwr; w += blockDim.x) {
        int c = w;
        if (rcls[w] >= 0) {
            const int s = rstart[w], len = rlen(w);
            const uint32_t h = rhash[w];
            for (int j = 0; j < w; ++j) {
                if (rhash[j] != h || rlen(j) != len || rcls[j] < 0) continue;
                const int sj = rstart[j];
                bool eq = true;
                for (int i = 0; i < len && eq; ++i) eq = rtok[sj + i] == rtok[s + i];
                if (eq) { c = j; break; }
            }
        }
        rclass[w] = c;
    }
    __syncthreads();
    for (int w = threadIdx.x; w < nwr; w += blockDim.x)
        if (rcls[w] >= 0) atomicOr(&peq[rclass[w] * W + (w >> 5)], 1u << (w & 31));
    if (ref_words && threadIdx.x == 0) ref_words[g] = nwr;
    __syncthreads();

    // one warp per hypothesis row
    int32_t* hstart = reinterpret_cast<int32_t*>(p + (size_t)warp * L.per_warp);
    uint32_t* hhash = reinterpret_cast<uint32_t*>(p + (size_t)warp * L.per_warp + L.per_warp / 3);
    int32_t* hid = reinterpret_cast<int32_t*>(p + (size_t)warp * L.per_warp + 2 * (L.per_warp / 3));
    for (int k = warp; k < rows_per_ref; k += nwarps) {
        const int row = g * rows_per_ref + k;
        if (row >= N) break;
        int n = hyp_len[row];
        n = min(max(n, 0), hyp_stride);
        const uint8_t* h = hyps + (size_t)row * hyp_stride;
        for (int i = lane; i < hyp_stride + 2; i += 32) hhash[i] = 0u;
        __syncwarp();
        int wbase = 0, open = 0;
        for (int t0 = 0; t0 < n; t0 += 32) {
            const int t = t0 + lane;
            const bool live = t < n;
            const uint32_t c = live ? h[t] : 0u;
            const bool is_sep = live && (int)c == sep;
            const unsigned smk = __ballot_sync(kFull, is_sep);
            const int wi = wbase + __popc(smk & lt);
            const unsigned below = smk & lt;
            const int st = below ? t0 + (31 - __clz(below)) + 1 : open;
            if (is_sep) hstart[wi + 1] = t + 1;
            else if (live) atomicAdd(hhash + wi, word_mix(c, (uint32_t)(t - st)));
            if (smk) open = t0 + (31 - __clz(smk)) + 1;
            wbase += __popc(smk);
        }
        if (lane == 0) hstart[0] = 0;
        const int nwh = wbase + 1;
        __syncwarp();
        for (int w = lane; w < nwh; w += 32) {
            const int s = hstart[w], len = (w + 1 < nwh ? hstart[w + 1] - 1 : n) - s;
            const uint32_t hh = hhash[w];
            int id = nwr;                                  // absent: the all-zero row of the match table
            for (int j = 0; j < nwr; ++j) {
                if (rclass[j] != j || rcls[j] < 0 || rhash[j] != hh || rlen(j) != len) continue;
                const int sj = rstart[j];
                bool eq = true;
                for (int i = 0; i < len && eq; ++i) eq = rtok[sj + i] == h[s + i];
                if (eq) { id = j; break; }
            }
            hid[w] = id;
        }
        __syncwarp();
        if (lane == 0) {
            MyersState<W> S;
            uint32_t sel[W];
#pragma unroll
            for (int w = 0; w < W; ++w) { S.VP[w] = 0xffffffffu; S.VN[w] = 0u; sel[w] = 0u; }
            for (int i = 0; i < nwh; ++i) {
                uint32_t eq[W];
                myers_load_eq<W>(peq, (uint32_t)hid[i], eq);
                myers_step<W, false>(S, eq, sel);
            }
            int d = nwh;                                   // dp[n, m] = n + sum_{j<m} (VP_j - VN_j)
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const int lo = w * 32;
                const uint32_t msk = nwr >= lo + 32 ? 0xffffffffu : (nwr > lo ? (1u << (nwr - lo)) - 1u : 0u);
                d += __popc(S.VP[w] & msk) - __popc(S.VN[w] & msk);
            }
            dist[row] = d;
        }
        __syncwarp();
    }
}

template <int W>
static int launch_word_ed(const uint8_t* hyps, const int32_t* hyp_len, int N, int hyp_stride, const int32_t* refs,
                          const int32_t* ref_len, int rows_per_ref, int ref_stride, int sep, int32_t* dist,
                          int32_t* ref_words, cudaStream_t st) {
    const WordEdSmem L = word_ed_smem(W, ref_stride, hyp_stride);
    constexpr size_t kLimit = 200 * 1024;
    if (L.fixed + L.per_warp > kLimit) return PGASR_ERR_UNSUPPORTED;
    int warps = (int)((kLimit - L.fixed) / L.per_warp);
    warps = warps > 8 ? 8 : warps;
    const size_t smem = L.fixed + (size_t)warps * L.per_warp;
    if (smem > 48 * 1024)
        PGASR_CUDA_TRY(cudaFuncSetAttribute(word_ed_u8_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int groups = (N + rows_per_ref - 1) / rows_per_ref;
    word_ed_u8_kernel<W><<<groups, warps * 32, smem, st>>>(hyps, hyp_len, N, hyp_stride, refs, ref_len, rows_per_ref,
                                                          ref_stride, sep, dist, ref_words);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}

}  // namespace pgasr

extern "C" int pgasr_word_edit_distance_u8(const uint8_t* hyps, const int32_t* hyp_len, int N, int hyp_stride,
                                           const int32_t* refs, const int32_t* ref_len, int rows_per_ref, int ref_stride,
                                           int sep, int32_t* dist, int32_t* ref_words, void* stream) {
    using namespace pgasr;
    if (!hyps || !hyp_len || !refs || !dist || N < 0 || hyp_stride <= 0 || ref_stride <= 0 || rows_per_ref <= 0 ||
        rows_per_ref > 1024 || sep < 0)
        return PGASR_ERR_INVALID_ARG;
    if (ref_stride > 511) return PGASR_ERR_UNSUPPORTED;
    if (N == 0) return PGASR_OK;
    cudaStream_t st = as_stream(stream);
    // n_w <= ref_len + 1 <= 512 words: W 32-bit words of the bit vectors
#define PGASR_WORD_ED(Wv) \
    return launch_word_ed<Wv>(hyps, hyp_len, N, hyp_stride, refs, ref_len, rows_per_ref, ref_stride, sep, dist, ref_words, st)
    if (ref_stride + 1 <= 32) PGASR_WORD_ED(1);
    if (ref_stride + 1 <= 64) PGASR_WORD_ED(2);
    if (ref_stride + 1 <= 128) PGASR_WORD_ED(4);
    if (ref_stride + 1 <= 256) PGASR_WORD_ED(8);
    PGASR_WORD_ED(16);
#undef PGASR_WORD_ED
}
