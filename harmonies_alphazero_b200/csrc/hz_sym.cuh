// hz_sym.cuh — the game's symmetry group on the packed state and on action rows (include/harmonies_b200.h
// "Game symmetries"): element g = (pile part c = g >> 2) << 2 | (board part b = g & 3).  Tables: hz_tables.inc.
#pragma once
#include "hz_core.cuh"

namespace hz {

// 0! .. 5!
__device__ __forceinline__ int sym_fact(int m) { return m <= 1 ? 1 : m == 2 ? 2 : m == 3 ? 6 : m == 4 ? 24 : 120; }

// packed pile permutation (pi[i] at bits 3i) of element g for m piles, or its inverse
__device__ __forceinline__ uint32_t sym_pile_perm(int g, int m, bool inverse) {
    m = m < 5 ? m : 5;
    const int idx = sym_pile_off(m) + (g >> 2) % sym_fact(m);
    return inverse ? __ldg(&SYM_PILE_INV_G[idx]) : __ldg(&SYM_PILE_PERM_G[idx]);
}

// sigma(a) for board part b, m piles and the packed pile permutation pp of sigma (the inverse tables give sigma^-1)
__device__ __forceinline__ int sym_action(int a, int b, int m, uint32_t pp, const uint8_t (*hex)[23]) {
    if (a < 5) return a < m ? (int)((pp >> (3 * a)) & 7u) : a;
    const int r = a - 5, t = r / 23, h = r - 23 * t;
    return 5 + 23 * t + __ldg(&hex[b][h]);
}

// Frame of a leaf row: rand(sk ^ HZ_SYMMETRY_SALT, canon_hash(words, HZ_KEY_EXACT)) scaled to 0..G-1.
__device__ __forceinline__ int sym_frame_of_key(uint64_t exact_key, uint64_t sk, int G) {
    const uint64_t z = rand64(sk ^ HZ_SYMMETRY_SALT, exact_key);
    return (int)(((z >> 32) * (uint64_t)G) >> 32);
}
// w: the 32 words (any memory space the caller can read uniformly).
__device__ __forceinline__ int sym_frame(const uint32_t* w, uint64_t sk, int G) {
    return sym_frame_of_key(exact_key_of_words(w), sk, G);
}

// Pile words 18..20 of T_g (the hand in the high half of word 20 stays): new position j < m holds old pile pi^-1[j].
__device__ __forceinline__ void sym_pile_words(uint32_t& w18, uint32_t& w19, uint32_t& w20, uint32_t w22, int g) {
    int m = (int)((w22 >> 16) & 0xFFu);
    m = m < 5 ? m : 5;
    const uint32_t inv = sym_pile_perm(g, m, true);
    const uint32_t p[5] = {w18 & 0xFFFFu, w18 >> 16, w19 & 0xFFFFu, w19 >> 16, w20 & 0xFFFFu};
    uint32_t q[5];
#pragma unroll
    for (int j = 0; j < 5; j++) {
        const int s = j < m ? (int)((inv >> (3 * j)) & 7u) : j;
        q[j] = s == 0 ? p[0] : s == 1 ? p[1] : s == 2 ? p[2] : s == 3 ? p[3] : p[4];   // selects: no local memory
    }
    w18 = q[0] | (q[1] << 16);
    w19 = q[2] | (q[3] << 16);
    w20 = q[4] | (w20 & 0xFFFF0000u);
}

// Warp-cooperative T_g for a record a warp already holds (the search's staged leaf): lane i holds word i and receives
// word i of T_g(record).  A plane word is permuted by one ballot (lane i < 23 contributes bit tau_b^-1(i)).  g warp-uniform.
__device__ __forceinline__ uint32_t warp_sym_word(uint32_t w, int g, int lane) {
    constexpr unsigned FULL_MASK = 0xFFFFFFFFu;
    const int src = lane < HZ_NUM_HEXES ? __ldg(&SYM_HEX_INV_G[g & 3][lane]) : 0;
    uint32_t out = w;
#pragma unroll
    for (int k = 0; k < 18; k++) {
        const uint32_t wk = __shfl_sync(FULL_MASK, w, k);
        const uint32_t nw = __ballot_sync(FULL_MASK, lane < HZ_NUM_HEXES && ((wk >> src) & 1u));
        if (lane == k) out = nw;
    }
    uint32_t w18 = __shfl_sync(FULL_MASK, w, HZ_W_PILES01), w19 = __shfl_sync(FULL_MASK, w, HZ_W_PILES23);
    uint32_t w20 = __shfl_sync(FULL_MASK, w, HZ_W_PILE4H);
    const uint32_t w22 = __shfl_sync(FULL_MASK, w, HZ_W_BAG1META);
    if (lane >= HZ_W_PILES01 && lane <= HZ_W_PILE4H) {
        sym_pile_words(w18, w19, w20, w22, g);
        out = lane == HZ_W_PILES01 ? w18 : lane == HZ_W_PILES23 ? w19 : w20;
    }
    return out;
}

}  // namespace hz
