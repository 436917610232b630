// CTC prefix beam search, batched: one CTA per utterance (SURVEY.md 8f.2; upstream CTCdecoder.py:41-116, the
// decoder policy_grad.reward (policy_grad.py:6) and predict() (model.py:324) call with beam_size=5).
//
// Upstream keeps the beam as a dict {prefix tuple: (p_blank, p_non_blank)} in log space, proposes every
// (prefix, symbol) pair per frame, merges proposals that spell the same prefix, sorts and trims (:110-113).  Here a
// prefix is a node of a per-utterance trie in global memory (parent, symbol, hash-consed through an open-addressing
// table so that a prefix re-entering the beam gets its old node back), and the only merge that can happen inside
// one frame -- an extension (q, s) that spells a prefix p already on the beam -- is resolved through links kept
// with the beam: par[p] = beam slot of p's parent string q, mask[q] = symbols s for which q+s is on the beam.
//   stay candidate of beam member i  : n_p_b  = lse(p_b + y_blank, p_nb + y_blank)                     (:78-81)
//                                      n_p_nb = lse(p_nb + y_last  [repeat merge, :103-106],
//                                                   extension of its parent by `last` [:88-98])
//   extension candidate (i, s)       : n_p_nb = s != last_i ? lse(p_b + y_s, p_nb + y_s) : p_b + y_s   (:91-98)
// Candidates are numbered in upstream's dict insertion order for blank == 0 (members first, then extensions by
// symbol, then member), so "largest score, then smallest index" reproduces its stable descending sort.
// Arithmetic is fp64 log space like upstream's (math.log / math.exp on Python floats).
#include <math.h>

#include "pgasr_common.cuh"

namespace pgasr {

constexpr int kBeamThreads = 128;
constexpr int kBeamMax = 128;
constexpr int kBeamMaxV = 64;            // classes of the one-word symbol masks (ctc_beam_kernel)
constexpr int kBeamWideWords = kMaxWideV / 64;   // mask words per slot of ctc_beam_wide_kernel (kBeamMaxV < V <= 256)
constexpr size_t kBeamMaxSmem = 226 * 1024;  // dynamic shared memory a CTA may take (227 KB less the static part)

__device__ __forceinline__ double lse2(double a, double b) {
    if (a == -INFINITY) return b;
    if (b == -INFINITY) return a;
    const double m = fmax(a, b);
    return m + log(exp(a - m) + exp(b - m));
}

struct BeamSet {            // one generation of the beam, in shared memory
    double* pb; double* pnb;
    int* node; int* pnode; int* last; int* par;
    unsigned long long* mask;   // NW words per slot: bit s of slot i = (s >> 6, s & 63)
};

template <int NW>
__device__ __forceinline__ BeamSet beam_carve(unsigned char*& p, int beam) {
    BeamSet b;
    b.pb = reinterpret_cast<double*>(p);                p += sizeof(double) * beam;
    b.pnb = reinterpret_cast<double*>(p);               p += sizeof(double) * beam;
    b.mask = reinterpret_cast<unsigned long long*>(p);  p += sizeof(unsigned long long) * NW * beam;
    b.node = reinterpret_cast<int*>(p);                 p += sizeof(int) * beam;
    b.pnode = reinterpret_cast<int*>(p);                p += sizeof(int) * beam;
    b.last = reinterpret_cast<int*>(p);                 p += sizeof(int) * beam;
    b.par = reinterpret_cast<int*>(p);                  p += sizeof(int) * beam;
    return b;
}

// at V = 256 (4 mask words) this is 2188 beam + 2112 bytes: beams up to 104 fit kBeamMaxSmem
static size_t beam_smem_bytes(int V, int beam) {
    const int nw = V > kBeamMaxV ? kBeamWideWords : 1;
    const size_t set = (size_t)beam * (2 * 8 + 8 * nw + 4 * 4);
    return 2 * set + sizeof(double) * (size_t)V + sizeof(double) * (size_t)beam * (V + 1) + sizeof(int) * (size_t)beam + 64;
}

// is s on slot i's children mask
template <int NW>
__device__ __forceinline__ bool beam_has_child(const BeamSet& b, int i, int s) {
    if constexpr (NW == 1) return (b.mask[i] >> s) & 1ull;
    else return (b.mask[i * NW + (s >> 6)] >> (s & 63)) & 1ull;
}

// (n_p_b, n_p_nb) of candidate c; see the header comment
template <int NW>
__device__ __forceinline__ void beam_candidate(const BeamSet& b, int nb, int beam, int V, int blank, const double* lp,
                                               int c, double& npb, double& npnb) {
    npb = npnb = -INFINITY;
    if (c < beam) {
        const int i = c;
        if (i >= nb) return;
        const double yb = lp[blank];
        npb = lse2(b.pb[i] + yb, b.pnb[i] + yb);
        const int last = b.last[i];
        if (last >= 0) {
            const double y = lp[last];
            npnb = b.pnb[i] + y;                                   // repeat merge: the prefix stays as it is
            const int j = b.par[i];
            if (j >= 0) {                                          // its parent string extended by `last`
                const double ext = last != b.last[j] ? lse2(b.pb[j] + y, b.pnb[j] + y) : b.pb[j] + y;
                npnb = lse2(npnb, ext);
            }
        }
    } else {
        const int e = c - beam, s = e / beam, i = e - s * beam;
        if (i >= nb || s == blank || s >= V || beam_has_child<NW>(b, i, s)) return;
        const double y = lp[s];
        npnb = s != b.last[i] ? lse2(b.pb[i] + y, b.pnb[i] + y) : b.pb[i] + y;
    }
}

__device__ __forceinline__ unsigned long long beam_hash(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}

// node id of prefix(parent) + s: the existing node, or a new one
__device__ int beam_child(int parent, int s, unsigned long long* hkeys, int* hvals, int H, int* node_parent,
                          int* node_char, int* node_count, int maxn) {
    const unsigned long long key = (((unsigned long long)(unsigned)parent << 8) | (unsigned)s) + 1ull;
    unsigned slot = (unsigned)beam_hash(key) & (unsigned)(H - 1);
    for (;;) {
        const unsigned long long prev = atomicCAS(hkeys + slot, 0ull, key);
        if (prev == 0ull) {
            const int id = atomicAdd(node_count, 1);
            if (id < maxn) { node_parent[id] = parent; node_char[id] = s; }
            hvals[slot] = id;
            return id;
        }
        if (prev == key) return hvals[slot];
        slot = (slot + 1) & (unsigned)(H - 1);
    }
}

// one utterance; NW 64-bit words per children mask (the two kernels below)
template <int NW>
__device__ __forceinline__ void beam_utterance(
    const double* __restrict__ probs, const int32_t* __restrict__ in_len, int T, int V, int beam, int blank,
    int32_t* __restrict__ labels, int32_t* __restrict__ label_len, double* __restrict__ nll,
    int* node_parent_all, int* node_char_all, unsigned long long* hkeys_all, int* hvals_all, int maxn, int H) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_count, s_m, s_win;
    __shared__ double s_wscore[kBeamThreads / 32];
    __shared__ int s_widx[kBeamThreads / 32];
    const int u = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned char* p = smem;
    BeamSet cur = beam_carve<NW>(p, beam), nxt = beam_carve<NW>(p, beam);
    double* lp = reinterpret_cast<double*>(p);          p += sizeof(double) * V;
    double* score = reinterpret_cast<double*>(p);       p += sizeof(double) * (size_t)beam * (V + 1);
    int* sel = reinterpret_cast<int*>(p);
    const int C = beam * (V + 1);
    int* node_parent = node_parent_all + (size_t)u * maxn;
    int* node_char = node_char_all + (size_t)u * maxn;
    unsigned long long* hkeys = hkeys_all + (size_t)u * H;
    int* hvals = hvals_all + (size_t)u * H;
    int Tu = in_len ? in_len[u] : T;
    Tu = min(max(Tu, 0), T);

    if (tid == 0) {
        cur.pb[0] = 0.0; cur.pnb[0] = -INFINITY; cur.node[0] = 0; cur.pnode[0] = -1; cur.last[0] = -1; cur.par[0] = -1;
#pragma unroll
        for (int w = 0; w < NW; ++w) cur.mask[w] = 0ull;
        node_parent[0] = -1; node_char[0] = -1;
        s_count = 1;
    }
    int nb = 1;
    __syncthreads();

    for (int t = 0; t < Tu; ++t) {
        const double* row = probs + ((size_t)u * T + t) * V;
        for (int v = tid; v < V; v += kBeamThreads) lp[v] = log(row[v]);
        __syncthreads();
        // ---- scores of all candidates ---------------------------------------------------------------
        double best = -INFINITY;
        int best_c = 0x7fffffff;
        for (int c = tid; c < C; c += kBeamThreads) {
            double a, b2;
            beam_candidate<NW>(cur, nb, beam, V, blank, lp, c, a, b2);
            const double sc = lse2(a, b2);
            score[c] = sc;
            if (sc > best) { best = sc; best_c = c; }
        }
        if (tid == 0) s_m = 0;
        __syncthreads();
        // ---- the `beam` best, one at a time: largest score, then smallest index ---------------------------
        for (int it = 0; it < beam; ++it) {
            double ws = best;
            int wc = best_c;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double os = __shfl_xor_sync(kFull, ws, o);
                const int oc = __shfl_xor_sync(kFull, wc, o);
                if (os > ws || (os == ws && oc < wc)) { ws = os; wc = oc; }
            }
            if (lane == 0) { s_wscore[warp] = ws; s_widx[warp] = wc; }
            __syncthreads();
            if (tid == 0) {
                double bs = s_wscore[0];
                int bc = s_widx[0];
                for (int w = 1; w < kBeamThreads / 32; ++w)
                    if (s_wscore[w] > bs || (s_wscore[w] == bs && s_widx[w] < bc)) { bs = s_wscore[w]; bc = s_widx[w]; }
                if (bs == -INFINITY) bc = -1;
                s_win = bc;
                if (bc >= 0) { sel[it] = bc; s_m = it + 1; }
            }
            __syncthreads();
            const int win = s_win;
            if (win < 0) break;
            if ((win % kBeamThreads) == tid) {                     // the owner drops it and rescans its candidates
                score[win] = -INFINITY;
                best = -INFINITY;
                best_c = 0x7fffffff;
                for (int c = tid; c < C; c += kBeamThreads)
                    if (score[c] > best) { best = score[c]; best_c = c; }
            }
        }
        __syncthreads();
        const int m = s_m;
        if (m == 0) break;                                         // no path has non-zero probability
        // ---- the new beam, already in descending order ---------------------------------------------------
        for (int a = tid; a < m; a += kBeamThreads) {
            const int c = sel[a];
            double npb, npnb;
            beam_candidate<NW>(cur, nb, beam, V, blank, lp, c, npb, npnb);
            nxt.pb[a] = npb;
            nxt.pnb[a] = npnb;
#pragma unroll
            for (int w = 0; w < NW; ++w) nxt.mask[a * NW + w] = 0ull;
            if (c < beam) {
                nxt.node[a] = cur.node[c]; nxt.pnode[a] = cur.pnode[c]; nxt.last[a] = cur.last[c];
            } else {
                const int e = c - beam, s = e / beam, i = e - s * beam;
                nxt.node[a] = beam_child(cur.node[i], s, hkeys, hvals, H, node_parent, node_char, &s_count, maxn);
                nxt.pnode[a] = cur.node[i];
                nxt.last[a] = s;
            }
        }
        __syncthreads();
        for (int a = tid; a < m; a += kBeamThreads) {              // links: parent slot, children masks
            const int pn = nxt.pnode[a];
            int par = -1;
            if (pn >= 0)
                for (int b2 = 0; b2 < m; ++b2)
                    if (nxt.node[b2] == pn) { par = b2; break; }
            nxt.par[a] = par;
            if (par >= 0) {
                const int s = nxt.last[a];
                if constexpr (NW == 1) atomicOr(nxt.mask + par, 1ull << s);
                else atomicOr(nxt.mask + par * NW + (s >> 6), 1ull << (s & 63));
            }
        }
        __syncthreads();
        BeamSet tmp = cur; cur = nxt; nxt = tmp;
        nb = m;
    }

    if (tid == 0) {
        const double ll = lse2(cur.pb[0], cur.pnb[0]);
        nll[u] = -ll;
        int n = 0;
        for (int x = cur.node[0]; x > 0; x = node_parent[x]) ++n;
        label_len[u] = n;
        int k = n;
        for (int x = cur.node[0]; x > 0; x = node_parent[x]) labels[(size_t)u * T + --k] = node_char[x];
        for (int k2 = n; k2 < T; ++k2) labels[(size_t)u * T + k2] = 0;
    }
}

#define PGASR_BEAM_KERNEL(name, nw)                                                                                   \
    __global__ void __launch_bounds__(kBeamThreads) name(                                                             \
        const double* __restrict__ probs, const int32_t* __restrict__ in_len, int T, int V, int beam, int blank,      \
        int32_t* __restrict__ labels, int32_t* __restrict__ label_len, double* __restrict__ nll,                      \
        int* node_parent_all, int* node_char_all, unsigned long long* hkeys_all, int* hvals_all, int maxn, int H) {   \
        beam_utterance<nw>(probs, in_len, T, V, beam, blank, labels, label_len, nll, node_parent_all, node_char_all,  \
                           hkeys_all, hvals_all, maxn, H);                                                            \
    }
PGASR_BEAM_KERNEL(ctc_beam_kernel, 1)                   // V <= 64
PGASR_BEAM_KERNEL(ctc_beam_wide_kernel, kBeamWideWords) // 64 < V <= 256
#undef PGASR_BEAM_KERNEL

// a shape the kernels take: V <= 256, beam <= 128, and the candidate table beam (V + 1) fits shared memory
static bool beam_supported(int V, int beam) {
    return V <= kMaxWideV && beam <= kBeamMax && beam_smem_bytes(V, beam) <= kBeamMaxSmem;
}

struct BeamWs { size_t parent, chr, keys, vals, total; int maxn, H; };

static BeamWs beam_ws(int N, int T, int beam) {
    BeamWs w;
    w.maxn = 1 + T * beam;
    int H = 1024;
    while (H < 2 * w.maxn) H <<= 1;
    w.H = H;
    auto al = [](size_t x) { return (x + 255) / 256 * 256; };
    w.keys = al((size_t)N * H * sizeof(unsigned long long));          // first: the part that must start at zero
    w.vals = al((size_t)N * H * sizeof(int));
    w.parent = al((size_t)N * w.maxn * sizeof(int));
    w.chr = al((size_t)N * w.maxn * sizeof(int));
    w.total = w.keys + w.vals + w.parent + w.chr;
    return w;
}

}  // namespace pgasr

extern "C" size_t pgasr_ctc_beam_search_workspace_bytes(int N, int T, int V, int beam) {
    using namespace pgasr;
    if (N <= 0 || T <= 0 || V <= 0 || beam <= 0 || !beam_supported(V, beam)) return 0;
    return beam_ws(N, T, beam).total;
}

extern "C" int pgasr_ctc_beam_search(const double* probs, const int32_t* in_len, int N, int T, int V, int beam,
                                     int blank, int32_t* labels, int32_t* label_len, double* nll, void* workspace,
                                     size_t workspace_bytes, void* stream) {
    using namespace pgasr;
    if (!probs || !labels || !label_len || !nll || !workspace || N <= 0 || T <= 0 || V <= 0 || beam <= 0 || blank < 0 ||
        blank >= V)
        return PGASR_ERR_INVALID_ARG;
    if (!beam_supported(V, beam)) return PGASR_ERR_UNSUPPORTED;
    const BeamWs w = beam_ws(N, T, beam);
    if (workspace_bytes < w.total) return PGASR_ERR_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    char* p = reinterpret_cast<char*>(workspace);
    unsigned long long* hkeys = reinterpret_cast<unsigned long long*>(p);   p += w.keys;
    int* hvals = reinterpret_cast<int*>(p);                                  p += w.vals;
    int* node_parent = reinterpret_cast<int*>(p);                            p += w.parent;
    int* node_char = reinterpret_cast<int*>(p);
    PGASR_CUDA_TRY(cudaMemsetAsync(hkeys, 0, w.keys, st));
    const size_t smem = beam_smem_bytes(V, beam);
    const auto kern = V > kBeamMaxV ? ctc_beam_wide_kernel : ctc_beam_kernel;
    PGASR_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<N, kBeamThreads, smem, st>>>(probs, in_len, T, V, beam, blank, labels, label_len, nll, node_parent, node_char,
                                        hkeys, hvals, w.maxn, w.H);
    PGASR_LAUNCH_CHECK();
    return PGASR_OK;
}
