// Word-level rewards (DESIGN.md "word reward spec"): what the single-launch step (fused_impl.cuh, word phase) and
// fused.cu (its shared-memory sizing) share.  Words are the id sequences between separators, split as Python's
// str.split(" "): count(sep) + 1 words, empty words kept.
#pragma once
#include "pgasr_common.cuh"

namespace pgasr {

// Upper bound of the distinct words of a transcript of <= Lmax ids that a collapsed hypothesis can match (words made
// of ids in [0, V) other than blank and the separator): one empty word, at most V - 2 one-id words (2 ids each with
// their separator), the rest at least 3 ids each -- 2a + 3b <= Lmax.  192 for Lmax = 511, V = 64: class ids fit u8
// with the "absent" class after them.
__host__ __device__ inline int word_class_cap(int Lmax, int V) {
    const int A = V > 2 ? V - 2 : 0;
    const int a = A < Lmax / 2 ? A : Lmax / 2;
    const int b = (Lmax - 2 * a) / 3;
    const int c = 1 + a + b;
    return c < Lmax + 1 ? c : Lmax + 1;
}

// Scratch of the word phase, carved from the PG role's tail region (the CDF rows of P1, dead by then): per utterance
// the transcript and its words, per warp the words of the hypothesis it is splitting.
__host__ __device__ inline size_t word_a16(size_t x) { return (x + 15) & ~(size_t)15; }
__host__ __device__ inline size_t word_ref_bytes(int Lmax, int cap) {
    const size_t nw = (size_t)Lmax + 2;
    return word_a16((size_t)Lmax + 1) + 2 * word_a16(2 * nw) + word_a16(4 * nw) + word_a16(8 * nw) + word_a16(nw) +
           word_a16(8 * (size_t)cap) + word_a16(2 * (size_t)cap);
}
// words of a collapsed hypothesis of <= T ids: two separators in a row need a blank frame between them, so
// count(sep) <= (T + 1) / 2
__host__ __device__ inline int word_hyp_slots(int T) { return ((T + 1) / 2 + 2 + 15) & ~15; }
__host__ __device__ inline size_t word_warp_bytes(int T) {
    const size_t tw = (size_t)word_hyp_slots(T);
    return word_a16(2 * tw) + 4 * tw + word_a16(tw);
}
__host__ __device__ inline size_t word_tail_bytes(int T, int Lmax, int cap, int nutt, int warps) {
    return (size_t)nutt * word_ref_bytes(Lmax, cap) + (size_t)warps * word_warp_bytes(T);
}

struct WordRef {
    uint8_t* ref;                  // [Lmax + 1] the transcript as ids; 0xFF for an id no hypothesis can hold (blank, >= V)
    uint16_t* start; uint16_t* rep; uint32_t* hash; uint64_t* key; uint8_t* cls;   // per word: first id, first equal word,
                                                                                  // hash, (length << 32 | hash), class
    uint64_t* ckey; uint16_t* cstart;                                             // per class: its first word's key, first id
};
__device__ __forceinline__ WordRef word_ref_carve(unsigned char* base, int uu, int Lmax, int cap) {
    unsigned char* p = base + (size_t)uu * word_ref_bytes(Lmax, cap);
    const size_t nw = (size_t)Lmax + 2;
    WordRef r;
    r.ref = p;                                        p += word_a16((size_t)Lmax + 1);
    r.start = reinterpret_cast<uint16_t*>(p);         p += word_a16(2 * nw);
    r.rep = reinterpret_cast<uint16_t*>(p);           p += word_a16(2 * nw);
    r.hash = reinterpret_cast<uint32_t*>(p);          p += word_a16(4 * nw);
    r.key = reinterpret_cast<uint64_t*>(p);           p += word_a16(8 * nw);
    r.cls = p;                                        p += word_a16(nw);
    r.ckey = reinterpret_cast<uint64_t*>(p);          p += word_a16(8 * (size_t)cap);
    r.cstart = reinterpret_cast<uint16_t*>(p);
    return r;
}

// hash of a word = sum over its ids of word_mix(id, position in the word) mod 2^32: order independent, so the lanes
// of a warp add their ids' terms with shared-memory atomics while they split the sequence.  Only a prefilter: equal
// (length, hash) is always confirmed id by id.
__device__ __forceinline__ uint32_t word_mix(uint32_t c, uint32_t i) {
    uint32_t x = (c + 1u) * 0x9E3779B1u + i * 0x85EBCA77u;
    x ^= x >> 15;
    x *= 0x2C1B3C6Du;
    x ^= x >> 12;
    return x;
}

// One warp splits ids[0, n) at `sep` in chunks of 32: start[w] (w >= 1) = first id of word w, hash[w] += the terms of
// its ids (hash[] zeroed by the caller), bad (optional) set for words holding 0xFF.  Returns the number of words.
// The caller sets start[0] = 0.  The terms of a word's ids in one chunk are summed by a segmented shuffle scan first,
// so that a word costs one shared-memory atomic per chunk (32 lanes adding to one address serialise).
__device__ __forceinline__ int word_split_warp(const uint8_t* ids, int n, int sep, uint16_t* start, uint32_t* hash,
                                               uint8_t* bad) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    int wbase = 0, open = 0;                          // words closed so far, first id of the open word
    for (int t0 = 0; t0 < n; t0 += 32) {
        const int t = t0 + lane;
        const bool live = t < n;
        const uint32_t c = live ? ids[t] : 0u;
        const bool is_sep = live && (int)c == sep;
        const unsigned sm = __ballot_sync(kFull, is_sep);
        const int wi = wbase + __popc(sm & lt);
        const unsigned below = sm & lt;
        const int st = below ? t0 + (31 - __clz(below)) + 1 : open;
        uint32_t v = live && !is_sep ? word_mix(c, (uint32_t)(t - st)) : 0u;
        const int seg0 = below ? 32 - __clz(below) : 0;  // first lane of this lane's word in the chunk
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(kFull, v, o);
            if (lane - o >= seg0) v += u;
        }
        if (is_sep) {
            start[wi + 1] = (uint16_t)(t + 1);
        } else if (live) {
            if (lane == 31 || t + 1 >= n || ((sm >> (lane + 1)) & 1u)) atomicAdd(hash + wi, v);   // (last id of the word here)
            if (bad && c == 0xFFu) bad[wi] = 1;
        }
        if (sm) open = t0 + (31 - __clz(sm)) + 1;
        wbase += __popc(sm);
    }
    return wbase + 1;
}

// First i in [i0, i1) with keys[i] == k, else i1: every key loaded unconditionally (independent loads, pipelined),
// not a loop that waits for each compare before the next load.
__device__ __forceinline__ int word_find_key(const uint64_t* keys, int i0, int i1, uint64_t k) {
    int f = i1;
#pragma unroll 4
    for (int i = i0; i < i1; ++i) f = (f == i1 && keys[i] == k) ? i : f;
    return f;
}

}  // namespace pgasr
