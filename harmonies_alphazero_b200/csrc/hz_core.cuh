// hz_core.cuh — device-side Harmonies engine on the 128-byte packed state
// (layout: include/harmonies_b200.h).  One thread owns one state in registers; every
// function is branch-light bit-board arithmetic over 23-bit hex masks.
//
// Reference behaviour reproduced (file:line into the reference):
//   legal moves      harmonies_engine.py:145-208
//   apply_move       harmonies_engine.py:210-298
//   end of turn      harmonies_engine.py:301-329, draws :120-137
//   scoring          harmonies_engine.py:357-523
//   canonical key    harmonies_engine.py:81-113 (+ MCTS.py:14,177,185 for HZ_KEY_REFERENCE)
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/harmonies_b200.h"
#include "hz_common.cuh"   // HZ_BOUND

namespace hz {

constexpr uint32_t VALID = 0x7FFFFFu;  // 23 hexes
constexpr int SW = 28;                 // live words of a state (28..31 are reserved zeros)

struct State {
    uint32_t w[SW];
};

// ---- neighbour tables ------------------------------------------------------------------
// NBR[i] = mask of hexes adjacent to hex i (constants.py:35 + harmonies_engine.py:31-43),
// derived offline from the axial coordinates; checked against the reference in the tests.
__constant__ uint32_t NBR[23] = {
    0x00000Cu, 0x000064u, 0x0000CBu, 0x000185u, 0x000220u, 0x000652u, 0x000CA6u, 0x00194Cu,
    0x003088u, 0x004430u, 0x00CA60u, 0x0194C0u, 0x032980u, 0x061100u, 0x088600u, 0x194C00u,
    0x329800u, 0x253000u, 0x022000u, 0x50C000u, 0x698000u, 0x130000u, 0x180000u};
// (y*7+x) cell of hex i in the 5x7 plane (process_game_state.py:9-12,36-37)
__constant__ uint8_t HEX_CELL[23] = {28, 15, 22, 29, 2, 9, 16, 23, 30, 3, 10, 17,
                                     24, 31, 4,  11, 18, 25, 32, 5, 12, 19, 6};
// fp32 bit patterns of float(c / INITIAL_BAG[t]) are produced with a double division, as
// the reference does (process_game_state.py:122-130)
__constant__ int INIT_BAG[6] = {23, 19, 21, 23, 15, 19};

// Shared-memory neighbour-expansion LUT: nbr(m) = L[0][m&255] | L[1][(m>>8)&255] | L[2][m>>16]
struct NbrLut {
    uint32_t t[3][256];
};
// The table is a compile-time constant in global memory (generated from the geometry by
// gen_tables.py).  Kernels that score a lot copy it to shared memory with coalesced loads
// (6 per thread at 128 threads); kernels that score rarely (the search tree: only children
// that end the game) read it in place through L1 via global_nbr_lut().
#include "hz_tables.inc"
__device__ __forceinline__ void build_nbr_lut(NbrLut* lut) {
    uint32_t* dst = &lut->t[0][0];
    for (int e = threadIdx.x; e < 768; e += blockDim.x) dst[e] = NBR_LUT_G[e];
}
__device__ __forceinline__ const NbrLut* global_nbr_lut() { return reinterpret_cast<const NbrLut*>(NBR_LUT_G); }
__device__ __forceinline__ uint32_t nbr(const NbrLut* lut, uint32_t m) {
    return lut->t[0][m & 255] | lut->t[1][(m >> 8) & 255] | lut->t[2][(m >> 16) & 127];
}
// The same expansion as ~20 shift/logic ops and no memory access.  With a full warp the three
// random LUT reads cost ~6 shared-memory wavefronts (bank conflicts); scoring uses this form in
// its straight-line part and the LUT inside the sparse, few-lane flood loops so that neither the
// LSU pipe nor the ALU pipe is the only one loaded (profiles/README.md, k_score).
__device__ __forceinline__ uint32_t nbr_alu(uint32_t m) {
    return pull_E(m) | pull_W(m) | pull_S(m) | pull_N(m) | pull_NE(m) | pull_SW(m);
}

// ---- rng ---------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t rand64(uint64_t key, uint64_t ctr) {
    return mix64(key ^ mix64(ctr + 0x9E3779B97F4A7C15ull));
}
// The inner mix depends on the counter only, and counters are small (move numbers < 200, draw
// events*8+k < 400): a per-block shared table of the first RTAB_N inner values halves the cost
// of every random number in the fused playout.  The values are a compile-time table (RAND_TAB_G, gen_tables.py); a block
// copies them to shared memory with coalesced 16-byte loads (4 per thread at 64 threads) instead of computing 512 mix64.
constexpr int RTAB_N = 512;
static_assert(sizeof(RAND_TAB_G) == RTAB_N * sizeof(uint64_t), "hz_tables.inc: RAND_TAB_G has RTAB_N entries");
__device__ __forceinline__ void build_rand_table(uint64_t* rtab) {   // rtab: 16-byte aligned
    const uint4* src = reinterpret_cast<const uint4*>(RAND_TAB_G);
    uint4* dst = reinterpret_cast<uint4*>(rtab);
    for (int e = threadIdx.x; e < RTAB_N / 2; e += blockDim.x) dst[e] = src[e];
}
// The table is handed around as its 32-bit shared-window address (0: no table, compute): through a generic pointer the
// compiler rebuilds the window address (S2R SR_CgaCtaId + LEA) in front of every lookup.
struct RandTab {
    uint32_t saddr;
    __device__ __forceinline__ RandTab(decltype(nullptr) = nullptr) : saddr(0) {}
    __device__ __forceinline__ explicit RandTab(uint32_t a) : saddr(a) {}
};
__device__ __forceinline__ RandTab rand_table_handle(const uint64_t* rtab) {   // rtab: the __shared__ array built above
    uint32_t a = (uint32_t)__cvta_generic_to_shared(rtab);
    asm volatile("" : "+r"(a));          // one register for the whole kernel, not rematerialised
    __builtin_assume(a != 0);
    return RandTab(a);
}
// rand64(key, ctr) with the inner mix read from the table; the caller guarantees a table and ctr < RTAB_N
__device__ __forceinline__ uint64_t rand64_tab(RandTab rtab, uint64_t key, uint32_t ctr) {
    uint32_t lo, hi;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(rtab.saddr + ctr * 8u));
    return mix64(key ^ ((uint64_t)lo | ((uint64_t)hi << 32)));
}
__device__ __forceinline__ uint64_t rand64_t(RandTab rtab, uint64_t key, uint64_t ctr) {
    if (rtab.saddr != 0 && ctr < (uint64_t)RTAB_N) return rand64_tab(rtab, key, (uint32_t)ctr);
    return mix64(key ^ mix64(ctr + 0x9E3779B97F4A7C15ull));
}

// ---- state access -------------------------------------------------------------------------
__device__ __forceinline__ void load_state(State& s, const void* base, int64_t idx) {
    const uint4* p = reinterpret_cast<const uint4*>(base) + idx * 8;
#pragma unroll
    for (int k = 0; k < 7; k++) {
        uint4 v = p[k];
        s.w[4 * k] = v.x; s.w[4 * k + 1] = v.y; s.w[4 * k + 2] = v.z; s.w[4 * k + 3] = v.w;
    }
}
// Warp-cooperative record load for the streaming kernels (k_legal, k_hash): the warp's 32 records (4 KB) arrive as 8 fully
// coalesced LDG.128 — 512 contiguous bytes = 4 lines per instruction, where the thread-per-record load above touches 32 lines
// per instruction and is bound by L1 tag lookups, not by HBM — and reach their threads through a swizzled shared-memory
// tile: chunk c of record r sits at [r][c ^ (r & 7)], which makes both the row-major store and the per-record read
// conflict-free.  All 32 lanes must call it (lanes past n get zeros); `tile` = 256 uint4 per warp.  NCH < 8: only the first
// NCH 16-byte chunks of every record are fetched (the rest of s.w is zero) — a kernel that never looks at words >= 24
// leaves the record's fourth 32-byte sector in DRAM.
template <int NCH = 8>
__device__ __forceinline__ void load_state_warp(State& s, const void* base, int64_t g_warp0, int64_t n, uint4* tile) {
    const int lane = threadIdx.x & 31;
    const uint4* p = reinterpret_cast<const uint4*>(base) + g_warp0 * 8;
    const int64_t lim = (n - g_warp0) * 8;                             // 16-byte chunks that exist
    uint4 v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = ((k * 32 + lane) < lim && (lane & 7) < NCH) ? __ldg(p + k * 32 + lane) : make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int rec = 4 * k + (lane >> 3), c = lane & 7;
        if (c < NCH) tile[rec * 8 + (c ^ (rec & 7))] = v[k];
    }
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 7; c++) {
        const uint4 x = c < NCH ? tile[lane * 8 + (c ^ (lane & 7))] : make_uint4(0, 0, 0, 0);
        s.w[4 * c] = x.x; s.w[4 * c + 1] = x.y; s.w[4 * c + 2] = x.z; s.w[4 * c + 3] = x.w;
    }
}
__device__ __forceinline__ void store_state(const State& s, void* base, int64_t idx) {
    uint4* p = reinterpret_cast<uint4*>(base) + idx * 8;
#pragma unroll
    for (int k = 0; k < 7; k++) p[k] = make_uint4(s.w[4 * k], s.w[4 * k + 1], s.w[4 * k + 2], s.w[4 * k + 3]);
    p[7] = make_uint4(0, 0, 0, 0);
}

__device__ __forceinline__ uint32_t meta(const State& s) { return s.w[HZ_W_BAG1META] >> 24; }
__device__ __forceinline__ int player_of(const State& s) { return (s.w[HZ_W_BAG1META] >> 24) & 1; }
__device__ __forceinline__ int phase_of(const State& s) { return (s.w[HZ_W_BAG1META] >> 25) & 7; }
__device__ __forceinline__ int ending_of(const State& s) { return (s.w[HZ_W_BAG1META] >> 28) & 1; }
__device__ __forceinline__ int winner_code(const State& s) { return (s.w[HZ_W_BAG1META] >> 29) & 3; }
__device__ __forceinline__ int n_piles_of(const State& s) { return (s.w[HZ_W_BAG1META] >> 16) & 0xFF; }
__device__ __forceinline__ uint32_t hand_of(const State& s) { return s.w[HZ_W_PILE4H] >> 16; }
__device__ __forceinline__ bool is_over(const State& s) { return ending_of(s) && winner_code(s) != 0; }
__device__ __forceinline__ int outcome_of(const State& s) {   // harmonies_engine.py:335-342
    int wc = winner_code(s);
    return (!ending_of(s)) ? 0 : wc == 1 ? 1 : wc == 2 ? -1 : 0;
}
__device__ __forceinline__ uint64_t key_of(const State& s) {
    return (uint64_t)s.w[HZ_W_KEYLO] | ((uint64_t)s.w[HZ_W_KEYHI] << 32);
}

// one player's board: 9 planes, bp[level*3+bit]
struct Board {
    uint32_t p[9];
};
__device__ __forceinline__ Board board_of(const State& s, int player) {
    Board b;
#pragma unroll
    for (int k = 0; k < 9; k++) b.p[k] = player ? s.w[9 + k] : s.w[k];
    return b;
}
__device__ __forceinline__ void set_board(State& s, int player, const Board& b) {
#pragma unroll
    for (int k = 0; k < 9; k++) {
        if (player) s.w[9 + k] = b.p[k]; else s.w[k] = b.p[k];
    }
}

// derived masks of one board
struct Tops {
    uint32_t occ0, occ1, occ2;  // height >= 1, 2, 3
    uint32_t t0, t1, t2;        // bits of the top tile's code
};
__device__ __forceinline__ Tops tops_of(const Board& b) {
    Tops t;
    t.occ0 = b.p[0] | b.p[1] | b.p[2];
    t.occ1 = b.p[3] | b.p[4] | b.p[5];
    t.occ2 = b.p[6] | b.p[7] | b.p[8];
    t.t0 = b.p[6] | (b.p[3] & ~t.occ2) | (b.p[0] & ~t.occ1);
    t.t1 = b.p[7] | (b.p[4] & ~t.occ2) | (b.p[1] & ~t.occ1);
    t.t2 = b.p[8] | (b.p[5] & ~t.occ2) | (b.p[2] & ~t.occ1);
    return t;
}
// tile codes: water 1, plant 2, wood 3, stone 4, building 5, field 6
__device__ __forceinline__ uint32_t top_water(const Tops& t) { return t.t0 & ~t.t1 & ~t.t2; }
__device__ __forceinline__ uint32_t top_plant(const Tops& t) { return ~t.t0 & t.t1 & ~t.t2; }
__device__ __forceinline__ uint32_t top_wood(const Tops& t) { return t.t0 & t.t1 & ~t.t2; }
__device__ __forceinline__ uint32_t top_stone(const Tops& t) { return ~t.t0 & ~t.t1 & t.t2; }
__device__ __forceinline__ uint32_t top_building(const Tops& t) { return t.t0 & ~t.t1 & t.t2; }
__device__ __forceinline__ uint32_t top_field(const Tops& t) { return ~t.t0 & t.t1 & t.t2; }

// ---- legal moves (harmonies_engine.py:145-208) ---------------------------------------------
// per-type 23-bit masks of legal hexes for the mover; types not in hand give 0.
struct Legal {
    uint32_t m[6];
    int n_piles;  // choose phase: number of selectable piles (else 0)
};
// REL ("mover-relative", only the fused playout's -DHZ_PLAYOUT_CHECKED comparison path; the default is playout_step<P> below): words 0..8 always hold the board of the player to
// move and 9..17 the other one; the halves are swapped whenever the player changes, so board
// access needs no per-word select on the player bit.  swap_boards() converts both ways.
__device__ __forceinline__ void swap_boards(State& s) {
#pragma unroll
    for (int k = 0; k < 9; k++) { uint32_t x = s.w[k]; s.w[k] = s.w[9 + k]; s.w[9 + k] = x; }
}
template <bool REL = false>
__device__ __forceinline__ Legal legal_of(const State& s) {
    Legal L;
#pragma unroll
    for (int t = 0; t < 6; t++) L.m[t] = 0;
    L.n_piles = 0;
    int ph = phase_of(s);
    if (ph == HZ_PHASE_CHOOSE) {
        L.n_piles = n_piles_of(s);                                   // :158
    } else if (ph <= HZ_PHASE_PLACE3) {
        uint32_t hand = hand_of(s);
        Tops t = tops_of(board_of(s, REL ? 0 : player_of(s)));
        uint32_t empty = ~t.occ0 & VALID;                            // :173
        uint32_t on_plant = top_wood(t) & ~t.occ2;                   // :183  (h <= 2)
        uint32_t on_stone = top_stone(t) & ~t.occ2;                  // :186  (h < 3)
        uint32_t on_build = (top_wood(t) | top_stone(t) | top_building(t)) & ~t.occ1;  // :190-192
        L.m[0] = (hand & 0x003) ? empty : 0;
        L.m[1] = (hand & 0x00C) ? (empty | on_plant) : 0;
        L.m[2] = (hand & 0x030) ? empty : 0;
        L.m[3] = (hand & 0x0C0) ? (empty | on_stone) : 0;
        L.m[4] = (hand & 0x300) ? (empty | on_build) : 0;
        L.m[5] = (hand & 0xC00) ? empty : 0;
    }
    return L;
}
__device__ __forceinline__ int legal_count(const Legal& L) {
    return L.n_piles + __popc(L.m[0]) + __popc(L.m[1]) + __popc(L.m[2]) + __popc(L.m[3]) +
           __popc(L.m[4]) + __popc(L.m[5]);
}
// 143-bit action mask, bit a = 5 + 23*t + hex (process_game_state.py:156-177)
__device__ __forceinline__ void legal_words(const Legal& L, uint32_t out[5]) {
    uint64_t lo = ((1u << L.n_piles) - 1u);           // bits 0..4
    lo |= (uint64_t)L.m[0] << 5;                      // 5..27
    lo |= (uint64_t)L.m[1] << 28;                     // 28..50
    uint64_t mid = (uint64_t)L.m[2] >> 13;            // bit 51.. -> word pair 1 (bits 64..127)
    lo |= (uint64_t)L.m[2] << 51;
    mid |= (uint64_t)L.m[3] << 10;                    // 74 - 64
    mid |= (uint64_t)L.m[4] << 33;                    // 97 - 64
    mid |= (uint64_t)L.m[5] << 56;                    // 120 - 64
    uint32_t hi = L.m[5] >> 8;                        // bits 128..142
    out[0] = (uint32_t)lo; out[1] = (uint32_t)(lo >> 32);
    out[2] = (uint32_t)mid; out[3] = (uint32_t)(mid >> 32);
    out[4] = hi;
}
// position of the k-th (0-based) set bit of a 23-bit mask m; k < popc(m)
__device__ __forceinline__ int nth_set_bit(uint32_t m, int k) {
    // the byte by cumulative counts (the trick of draw_tile): bytes 1 and 2 of e hold the set bits of bytes 0 and 0..1, and
    // bit 7 of each byte of d says k reached that count (all counts and k are < 128: no borrow between bytes)
    const uint32_t e = (uint32_t)__popc(m & 0xFFu) * 0x100u + (uint32_t)__popc(m & 0xFFFFu) * 0x10000u;
    const uint32_t d = (((uint32_t)k * 0x01010100u) | 0x80808000u) - e;
    const uint32_t j = __popc(d & 0x00808000u);
    k -= (int)__byte_perm(e, 0u, j);                                   // byte j of e: the set bits below byte j (byte 0 is 0)
    int pos = 8 * (int)j, c;
    m >>= pos;
    c = __popc(m & 0xFu);    if (k >= c) { k -= c; pos += 4;  m >>= 4; }
    // in the last nibble the same way: byte i of pre = set bits of the nibble's bits 0..i (the multiply by 0x204081 moves
    // bit i to bit 8i without carries), and the k-th set bit is at the number of those counts <= k
    const uint32_t pre = (((m & 0xFu) * 0x204081u) & 0x01010101u) * 0x01010101u;
    return pos + __popc(((((uint32_t)k * 0x01010101u) | 0x80808080u) - pre) & 0x80808080u);
}
// k-th legal action in ascending action-index order; k < legal_count(L)
__device__ __forceinline__ int kth_action(const Legal& L, int k) {
    if (k < L.n_piles) return k;                      // choose phase (all type masks are zero)
    // placement: pick the type whose cumulative count covers k with selects, then ONE bit search
    // shared by all lanes (a per-type branch leaves ~5 of 32 lanes active in each search)
    k -= L.n_piles;
    int c0 = __popc(L.m[0]), c1 = c0 + __popc(L.m[1]), c2 = c1 + __popc(L.m[2]);
    int c3 = c2 + __popc(L.m[3]), c4 = c3 + __popc(L.m[4]);
    int t = (k >= c0) + (k >= c1) + (k >= c2) + (k >= c3) + (k >= c4);
    uint32_t m = t == 0 ? L.m[0] : t == 1 ? L.m[1] : t == 2 ? L.m[2] : t == 3 ? L.m[3] : t == 4 ? L.m[4] : L.m[5];
    int below = t == 0 ? 0 : t == 1 ? c0 : t == 2 ? c1 : t == 3 ? c2 : t == 4 ? c3 : c4;
    return 5 + 23 * t + nth_set_bit(m, k - below);
}
// the uniform-random playout policy (see hz_random_actions in harmonies_b200.h)
__device__ __forceinline__ int random_action(const State& s, const Legal& L, RandTab rtab = nullptr) {
    int n = legal_count(L);
    if (n == 0) return -1;
    uint64_t r = rand64_t(rtab, key_of(s) ^ HZ_PLAYOUT_SALT, (uint64_t)s.w[HZ_W_MOVES]);
    int k = (int)(((r >> 32) * (uint64_t)n) >> 32);
    return kth_action(L, k);
}

// ---- scoring (harmonies_engine.py:357-523) --------------------------------------------------
__device__ __forceinline__ uint32_t flood(const NbrLut* lut, uint32_t seed, uint32_t within) {
    uint32_t f = seed, nf;
    while ((nf = (f | nbr(lut, f)) & within) != f) f = nf;
    return f;
}
__device__ __forceinline__ int water_points(int len) {              // :18-27
    return len <= 1 ? 0 : len == 2 ? 2 : len <= 5 ? 3 * len - 4 : 15 + (len - 6) * 4;
}
// Water components of >= 5 hexes are rare (a few percent of boards) but one of them costs a lane
// ~20 flood iterations while the other 31 wait.  A caller whose block reconverges after scoring
// passes a WaterQueue: such components are pushed there instead, and resolve_water() gives each
// queued component a whole warp, one BFS source per lane.
template <int CAP, int OWNERS>
struct WaterQueue {
    uint32_t comp[CAP];
    uint16_t owner[CAP];
    int extra[OWNERS];      // points of the resolved components, per owner slot
    int count;
};
template <int CAP, int OWNERS>
__device__ __forceinline__ void water_queue_init(WaterQueue<CAP, OWNERS>* q) {   // then __syncthreads()
    for (int e = threadIdx.x; e < OWNERS; e += blockDim.x) q->extra[e] = 0;
    if (threadIdx.x == 0) q->count = 0;
}
struct NoWaterQueue {};
__device__ __forceinline__ bool water_push(NoWaterQueue*, uint32_t, int) { return false; }
template <int CAP, int OWNERS>
__device__ __forceinline__ bool water_push(WaterQueue<CAP, OWNERS>* q, uint32_t comp, int owner) {
    int slot = atomicAdd(&q->count, 1);
    if (slot >= CAP) return false;                                    // full: the caller scores it in place
    HZ_BOUND(slot, CAP, 401);
    HZ_BOUND(owner, OWNERS, 402);
    q->comp[slot] = comp;
    q->owner[slot] = (uint16_t)owner;
    return true;
}
template <typename Q = NoWaterQueue>
__device__ __forceinline__ void score_board(const NbrLut* lut, const Board& b, int terms[5], Q* wq = nullptr,
                                            int owner = 0) {
    Tops t = tops_of(b);
    uint32_t h1 = t.occ0 & ~t.occ1, h2 = t.occ1 & ~t.occ2, h3 = t.occ2;
    // grass :369-385
    uint32_t tp = top_plant(t);
    uint32_t l0_wood = b.p[0] & b.p[1] & ~b.p[2], l1_wood = b.p[3] & b.p[4] & ~b.p[5];
    terms[0] = __popc(tp & h1) + 3 * __popc(tp & h2 & l0_wood) + 7 * __popc(tp & h3 & l0_wood & l1_wood);
    // One neighbour expansion per top type serves every term: n_X = hexes adjacent to an X-top.
    uint32_t tw = top_water(t), twd = top_wood(t), ts = top_stone(t), tbl = top_building(t), tf = top_field(t);
    uint32_t n_w = nbr_alu(tw), n_p = nbr_alu(tp), n_wd = nbr_alu(twd), n_s = nbr_alu(ts);
    uint32_t n_b = nbr_alu(tbl), n_f = nbr_alu(tf);
    // mountains :392-413
    uint32_t adj = ts & n_s;
    terms[1] = __popc(adj & h1) + 3 * __popc(adj & h2) + 7 * __popc(adj & h3);
    // buildings :454-469 — >= 3 distinct top types among the neighbours, for all hexes at once:
    // bit-sliced count of the six adjacency masks (two full adders), no per-hex loop
    uint32_t s1 = n_w ^ n_p ^ n_wd, c1 = (n_w & n_p) | (n_wd & (n_w ^ n_p));
    uint32_t s2 = n_s ^ n_b ^ n_f, c2 = (n_s & n_b) | (n_f & (n_s ^ n_b));
    uint32_t atleast3 = (c1 & c2) | ((c1 | c2) & (s1 | s2));
    terms[3] = 5 * __popc(tbl & h2 & atleast3);
    // fields :424-443 — 5 points per component of size >= 2.  Isolated hexes are dropped up front;
    // the component count of what is left comes from the Euler characteristic of the hex cells,
    // components - holes = V - E + T (hexes, adjacent pairs, mutually adjacent triples), each term a
    // popcount of masked shifts, so the common case has no data-dependent loop.  A hole needs a
    // ring of >= 6 field hexes: only then the enclosed regions of the complement are counted.
    uint32_t rem = tf & n_f;
    uint32_t fe = rem & pull_E(rem);
    int comps = __popc(rem) - __popc(fe) - __popc(rem & pull_S(rem)) - __popc(rem & pull_NE(rem))
              + __popc(fe & pull_S(rem)) + __popc(fe & pull_NE(rem));
    if (__popc(rem) >= 6) {
        uint32_t c = VALID & ~rem;
        uint32_t enclosed = c & ~flood(lut, c & BOUNDARY_HEXES, c);
        while (enclosed) {
            uint32_t hole = flood(lut, enclosed & (0u - enclosed), enclosed);
            enclosed &= ~hole;
            comps++;
        }
    }
    terms[2] = 5 * comps;
    // water :480-518 — per component of size >= 2: (BFS diameter + 1) -> table.  Size-2 components
    // (by far the most common) are found without a loop: both hexes have exactly one water
    // neighbour (bit-sliced count over the six directions) and are adjacent to each other.
    int sc = 0;
    rem = tw & n_w;
    uint32_t we = pull_E(rem), ws = pull_S(rem), wne = pull_NE(rem), deg1;
    {
        uint32_t one = we, more = 0, p;
        p = pull_W(rem);  more |= one & p; one ^= p;
        more |= one & ws;  one ^= ws;
        p = pull_N(rem);  more |= one & p; one ^= p;
        more |= one & wne; one ^= wne;
        p = pull_SW(rem); more |= one & p; one ^= p;
        deg1 = rem & one & ~more;
        uint32_t pairs = deg1 & nbr(lut, deg1);
        sc = __popc(pairs);                                           // length 2 -> 2 points per pair
        rem &= ~pairs;
    }
    while (rem) {                                                     // components of size >= 3
        uint32_t comp = flood(lut, rem & (0u - rem), rem);
        rem &= ~comp;
        int size = __popc(comp), diameter;
        if (size <= 4) {
            // closed forms from the edge count: 3 hexes are a triangle (diameter 1) or a path (2);
            // 4 hexes have diameter 3 only as a path (3 edges, two ends), every other shape on this
            // lattice (claw, triangle + tail, rhombus) has diameter 2
            int edges = __popc(comp & we) + __popc(comp & ws) + __popc(comp & wne);
            diameter = size == 3 ? 4 - edges : (edges == 3 && __popc(comp & deg1) == 2) ? 3 : 2;
        } else {
            if (water_push(wq, comp, owner)) continue;
            diameter = 0;
            uint32_t src = comp;
            while (src) {
                uint32_t f = src & (0u - src), nf;
                src ^= f;
                int d = 0;
                while ((nf = (f | nbr(lut, f)) & comp) != f) { f = nf; d++; }
                diameter = max(diameter, d);
            }
        }
        sc += water_points(diameter + 1);
    }
    terms[4] = sc;
}
// all threads of the block, between two __syncthreads(): q->extra[owner] += points of each queued component
template <int CAP, int OWNERS>
__device__ __forceinline__ void resolve_water(const NbrLut* lut, WaterQueue<CAP, OWNERS>* q) {
    // FOUR components per warp: a group of 8 lanes takes one component, lane j of the group the BFS from its j-th, (j+8)-th ...
    // hex.  (One component per warp with one source per lane left 24-27 lanes idle: these components have 5-8 hexes.)
    const int n = min(q->count, CAP), lane = threadIdx.x & 31, sub = lane >> 3, j0 = lane & 7;
    const int nw = blockDim.x >> 5;
    for (int base = (threadIdx.x >> 5) * 4; base < n; base += nw * 4) {
        const int e = base + sub;
        const uint32_t comp = e < n ? q->comp[e] : 0u;
        const int size = __popc(comp);
        int d = 0;
        for (int j = j0; j < size; j += 8) {
            uint32_t f = 1u << __fns(comp, 0, j + 1), nf;
            int dd = 0;
            while ((nf = (f | nbr(lut, f)) & comp) != f) { f = nf; dd++; }
            d = max(d, dd);
        }
        d = max(d, __shfl_xor_sync(0xFFFFFFFFu, d, 1));
        d = max(d, __shfl_xor_sync(0xFFFFFFFFu, d, 2));
        d = max(d, __shfl_xor_sync(0xFFFFFFFFu, d, 4));
        if (e < n && j0 == 0) atomicAdd(&q->extra[q->owner[e]], water_points(d + 1));
    }
}
__device__ __forceinline__ int score_player(const NbrLut* lut, const State& s, int p) {
    int t[5];
    score_board(lut, board_of(s, p), t);
    return t[0] + t[1] + t[2] + t[3] + t[4];
}

// ---- draws (harmonies_engine.py:120-137) -----------------------------------------------------
// bag as 6 bytes of a 64-bit word (TILE_TYPES order)
__device__ __forceinline__ uint64_t bag_of(const State& s) {
    return (uint64_t)s.w[HZ_W_BAG0] | ((uint64_t)(s.w[HZ_W_BAG1META] & 0xFFFFu) << 32);
}
__device__ __forceinline__ void set_bag(State& s, uint64_t bag) {
    s.w[HZ_W_BAG0] = (uint32_t)bag;
    s.w[HZ_W_BAG1META] = (s.w[HZ_W_BAG1META] & 0xFFFF0000u) | (uint32_t)(bag >> 32);
}
__device__ __forceinline__ int bag_total(uint64_t bag) {
    uint32_t lo = (uint32_t)bag, hi = (uint32_t)(bag >> 32);
    uint32_t s = (lo & 0x00FF00FFu) + ((lo >> 8) & 0x00FF00FFu) + (hi & 0xFFu) + ((hi >> 8) & 0xFFu);
    return (s & 0xFFFFu) + (s >> 16);
}
// draws min(3,total) tiles; returns the pile's multiset code (0 if the bag was empty)
__device__ __forceinline__ uint32_t shl_clamped(uint32_t v, uint32_t n) {   // v << n, 0 for n >= 32 (PTX shl.b32 clamps)
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
    return r;
}
// draw j (0..2) of a pile from a bag of 0 < `total` <= 127 tiles, the bag as two 32-bit halves (types 0..3 | 4,5): the
// cumulative counts and the decrement stay 32-bit operations.  Returns the tile's increment of the pile code.
__device__ __forceinline__ uint32_t draw_tile(uint32_t& lo, uint32_t& hi, uint32_t total, uint64_t z, int j) {
    uint32_t x = (uint32_t)(z >> (21 * j)) & 0x1FFFFFu;
    uint32_t r = (x * total) >> 21;                                  // 21+7 bits < 32
    uint32_t clo = lo * 0x01010101u;                                 // byte k = sum of bytes 0..k (totals <= 255: no carries)
    uint32_t c4 = (clo >> 24) + (hi & 0xFFu);
    // types 0..3 whose cumulative count is <= r, four at once: bit 7 of each byte of the difference is set exactly there
    // (total <= 127, so r and the counts are < 128 and no byte borrows; __vcmpleu4 is emulated on sm_100a)
    uint32_t rr = (r * 0x01010101u) | 0x80808080u;
    int t = __popc((rr - clo) & 0x80808080u) + (c4 <= r ? 1 : 0);
    lo -= shl_clamped(1u, 8u * (uint32_t)t);                         // t >= 4: shifted out
    hi -= shl_clamped(1u, 8u * (uint32_t)t - 32u);                   // t < 4: the count wraps to >= 32, shifted out
    return 1u << (2 * t);
}
__device__ __forceinline__ uint32_t draw_pile(uint64_t& bag, uint64_t z) {
    uint32_t lo = (uint32_t)bag, hi = (uint32_t)(bag >> 32), code = 0;
    int total = bag_total(bag);
    if (total > 127) {
        // A game's bag never holds more than 120 tiles, but a record may carry up to 255 of each type (pack_fields): past
        // draw_tile's range, three draws by the plain cumulative loop of the specification (x * total < 2^21 * 1530 < 2^32).
#pragma unroll
        for (int j = 0; j < 3; j++, total--) {
            const uint32_t r = (((uint32_t)(z >> (21 * j)) & 0x1FFFFFu) * (uint32_t)total) >> 21;
            int t = 0;
            uint32_t cum = (uint32_t)bag & 0xFFu;                    // count of types 0..t
            while (t < 5 && cum <= r) cum += (uint32_t)(bag >> (8 * ++t)) & 0xFFu;
            bag -= 1ull << (8 * t);
            code += 1u << (2 * t);
        }
        return code;
    }
#pragma unroll
    for (int j = 0; j < 3; j++) {
        if (total > 0) {
            code += draw_tile(lo, hi, (uint32_t)total, z, j);
            total--;
        }
    }
    bag = (uint64_t)lo | ((uint64_t)hi << 32);
    return code;
}
// draw_pile from a bag of 3 <= total <= 127 tiles: always three draws, no branch
__device__ __forceinline__ uint32_t draw_pile3(uint32_t& lo, uint32_t& hi, uint32_t total, uint64_t z) {
    uint32_t code = draw_tile(lo, hi, total, z, 0);                  // (three statements: each draw sees the bag the last left)
    code += draw_tile(lo, hi, total - 1u, z, 1);
    return code + draw_tile(lo, hi, total - 2u, z, 2);
}
__device__ __forceinline__ bool pile_available(uint64_t bag, uint32_t code) {
    bool ok = true;
#pragma unroll
    for (int t = 0; t < 6; t++) ok &= ((code >> (2 * t)) & 3u) <= ((uint32_t)(bag >> (8 * t)) & 0xFFu);
    return ok;
}
__device__ __forceinline__ uint64_t bag_minus(uint64_t bag, uint32_t code) {
#pragma unroll
    for (int t = 0; t < 6; t++) bag -= (uint64_t)((code >> (2 * t)) & 3u) << (8 * t);
    return bag;
}

// piles as 5 registers
struct Piles {
    uint32_t p[5];
};
__device__ __forceinline__ Piles piles_of(const State& s) {
    Piles P;
    P.p[0] = s.w[HZ_W_PILES01] & 0xFFFFu; P.p[1] = s.w[HZ_W_PILES01] >> 16;
    P.p[2] = s.w[HZ_W_PILES23] & 0xFFFFu; P.p[3] = s.w[HZ_W_PILES23] >> 16;
    P.p[4] = s.w[HZ_W_PILE4H] & 0xFFFFu;
    return P;
}
__device__ __forceinline__ void set_piles(State& s, const Piles& P, uint32_t hand, int n_piles) {
    s.w[HZ_W_PILES01] = P.p[0] | (P.p[1] << 16);
    s.w[HZ_W_PILES23] = P.p[2] | (P.p[3] << 16);
    s.w[HZ_W_PILE4H] = P.p[4] | (hand << 16);
    s.w[HZ_W_BAG1META] = (s.w[HZ_W_BAG1META] & 0xFF00FFFFu) | ((uint32_t)n_piles << 16);
}
__device__ __forceinline__ void set_meta(State& s, uint32_t m) {
    s.w[HZ_W_BAG1META] = (s.w[HZ_W_BAG1META] & 0x00FFFFFFu) | (m << 24);
}

// ---- apply_move (harmonies_engine.py:210-329) -------------------------------------------------
// dkey/devent: draw stream used if this move ends a turn; explicit_code != HZ_NO_DRAW
// replaces the first pile drawn (trace replay); bump_event: advance the state's own event
// counter (engine streams) or leave it (in-tree draws keyed by (simulation, action)).
// Returns an HZ_MOVE_* status; the state is modified only on HZ_MOVE_OK.
// DEFER_SCORE: at the end of the game only mark phase game_over (winner still None) and let
// the caller run finalize_scores() later — the fused playout does that once per warp after
// all of its games have ended, so the scoring loops run with all lanes converged.
__device__ __forceinline__ void store_final_scores(State& s, int s0, int s1) {
    s.w[HZ_W_SCORES] = ((uint32_t)s0 & 0xFFFFu) | (((uint32_t)s1 & 0xFFFFu) << 16);
    uint32_t wc = s0 > s1 ? 1u : s1 > s0 ? 2u : 3u;                       // :348-354
    s.w[HZ_W_BAG1META] = (s.w[HZ_W_BAG1META] & ~(3u << 29)) | (wc << 29);
}
__device__ __forceinline__ void finalize_scores(State& s, const NbrLut* lut) {
    int s0 = score_player(lut, s, 0), s1 = score_player(lut, s, 1);       // :344-346
    store_final_scores(s, s0, s1);
}
// both players' scores with large water components pushed to the block's queue (owner slots
// 2*threadIdx.x + player); the caller adds q->extra[...] after resolve_water()
template <int CAP, int OWNERS>
__device__ __forceinline__ void partial_scores(const State& s, const NbrLut* lut, WaterQueue<CAP, OWNERS>* q, int& s0, int& s1) {
    int t[5];
    score_board(lut, board_of(s, 0), t, q, (int)threadIdx.x * 2);
    s0 = t[0] + t[1] + t[2] + t[3] + t[4];
    score_board(lut, board_of(s, 1), t, q, (int)threadIdx.x * 2 + 1);
    s1 = t[0] + t[1] + t[2] + t[3] + t[4];
}
// ---- _replenish_piles (:132-137) + _end_turn_actions (:301-329) -------------------------------------
// Tops the piles up to five from the bag (first pile = explicit_code when use_explicit: trace replay),
// draw k of event `devent` of stream `dkey` being rand(dkey, devent*8 + k).  Returns whether the bag
// was empty BEFORE replenishing (:307).
__device__ __forceinline__ bool replenish_piles(State& s, uint32_t hand, bool use_explicit, uint32_t explicit_code, uint64_t dkey,
                                                uint32_t devent, RandTab rtab, int& np_out) {
    int np = n_piles_of(s);
    uint64_t bag = bag_of(s);
    bool bag_empty_before = bag_total(bag) == 0;                      // :307
    Piles P = piles_of(s);
    for (int k = 0; np < 5; k++) {                                    // _replenish_piles :132-137
        uint32_t pc;
        if (k == 0 && use_explicit) { pc = explicit_code; bag = bag_minus(bag, pc); }
        else pc = draw_pile(bag, rand64_t(rtab, dkey, (uint64_t)devent * 8 + (uint64_t)k));
        if (pc == 0) break;                                           // :135-136
#pragma unroll
        for (int j = 0; j < 5; j++) P.p[j] = (j == np) ? pc : P.p[j];
        np++;
    }
    set_bag(s, bag);
    set_piles(s, P, hand, np);   // the reference does not clear a (non-standard) leftover hand at end of turn
    np_out = np;
    return bag_empty_before;
}
// `pl` has just finished a turn; occ_after = occupancy mask of pl's board.  (The reference's
// _end_turn_actions, also called directly by its GUI: GUI/main.py:364-365.)
template <bool DEFER_SCORE = false, bool REL = false>
__device__ __forceinline__ int end_turn(State& s, int pl, uint32_t occ_after, uint32_t hand, bool use_explicit, uint32_t explicit_code,
                                        uint64_t dkey, uint32_t devent, bool bump_event, const NbrLut* lut, RandTab rtab) {
    bool player_trigger = (23 - __popc(occ_after)) <= 2;              // :304-305
    int np;
    bool bag_empty_before = replenish_piles(s, hand, use_explicit, explicit_code, dkey, devent, rtab, np);
    if (bump_event) s.w[HZ_W_EVENT]++;
    bool triggered = player_trigger || (bag_empty_before && np == 0);  // :309-311
    bool ending = ending_of(s);
    uint32_t m = meta(s) & 1u;                                        // keep player
    if (triggered && !ending && pl == 0) {                            // :314-318
        m = 1u | (HZ_PHASE_CHOOSE << 1) | (1u << 4);
        if (REL) swap_boards(s);
    } else if ((triggered && !ending) || ending) {                    // :319-326
        set_meta(s, m | (HZ_PHASE_OVER << 1) | (1u << 4));            // :320,324 (winner still None)
        if (!DEFER_SCORE) finalize_scores(s, lut);                    // :321-322,325-326
        return HZ_MOVE_OK;
    } else {                                                          // :327-329
        m = (m ^ 1u) | (HZ_PHASE_CHOOSE << 1);
        if (REL) swap_boards(s);
    }
    set_meta(s, m);
    return HZ_MOVE_OK;
}

template <bool DEFER_SCORE = false, bool REL = false>
__device__ __forceinline__ int apply_move(State& s, int a, uint32_t explicit_code, uint64_t dkey,
                                          uint32_t devent, bool bump_event, const NbrLut* lut,
                                          RandTab rtab = nullptr) {
    int ph = phase_of(s);
    if (ph == HZ_PHASE_CHOOSE) {
        int np = n_piles_of(s);
        if (a < 0 || a >= np) return HZ_MOVE_BAD_PILE;               // :217-220
        Piles P = piles_of(s);
        uint32_t hand = P.p[0];
#pragma unroll
        for (int j = 1; j < 5; j++) hand = (a == j) ? P.p[j] : hand;
#pragma unroll
        for (int j = 0; j < 4; j++) P.p[j] = (j >= a) ? P.p[j + 1] : P.p[j];   // pop(i), :221
        P.p[4] = 0;
        set_piles(s, P, hand, np - 1);
        set_meta(s, (meta(s) & ~0xEu) | (HZ_PHASE_PLACE1 << 1));      // :223
        s.w[HZ_W_MOVES]++;
        return HZ_MOVE_OK;
    }
    if (ph > HZ_PHASE_PLACE3) return HZ_MOVE_BAD_PHASE;              // :296
    if (a < 5) return HZ_MOVE_BAD_FORMAT;                            // :227-236
    if (a >= HZ_ACTION_SIZE) return HZ_MOVE_BAD_COORD;               // :241-242
    int tile = (a - 5) / 23, hex = (a - 5) - 23 * tile;
    uint32_t hand = hand_of(s);
    if (((hand >> (2 * tile)) & 3u) == 0) return HZ_MOVE_NOT_IN_HAND;   // :244-248
    int pl = player_of(s);
    Board b = board_of(s, REL ? 0 : pl);
    Tops t = tops_of(b);
    uint32_t bit = 1u << hex;
    uint32_t ok = ~t.occ0;                                            // :255-257
    ok |= (tile == 1) ? (top_wood(t) & ~t.occ2) : 0u;                 // :263
    ok |= (tile == 3) ? (top_stone(t) & ~t.occ2) : 0u;                // :265
    ok |= (tile == 4) ? ((top_wood(t) | top_stone(t) | top_building(t)) & ~t.occ1) : 0u;  // :267-271
    if (!(ok & bit)) return HZ_MOVE_ILLEGAL_STACK;                    // :281
    bool ends_turn = ph == HZ_PHASE_PLACE3;
    int np = n_piles_of(s);
    uint64_t bag = bag_of(s);
    bool use_explicit = ends_turn && explicit_code != HZ_NO_DRAW && np < 5;
    if (use_explicit && !pile_available(bag, explicit_code)) return HZ_MOVE_BAD_DRAW;

    // place the tile on level h of the hex (:257,275)
    uint32_t code = (uint32_t)tile + 1u;
    uint32_t at0 = bit & ~t.occ0, at1 = bit & t.occ0 & ~t.occ1, at2 = bit & t.occ1;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        uint32_t on = (code >> k) & 1u ? 0xFFFFFFFFu : 0u;
        b.p[k] |= at0 & on; b.p[3 + k] |= at1 & on; b.p[6 + k] |= at2 & on;
    }
    set_board(s, REL ? 0 : pl, b);
    hand -= 1u << (2 * tile);                                         // hand.remove, :250
    s.w[HZ_W_PILE4H] = (s.w[HZ_W_PILE4H] & 0xFFFFu) | (hand << 16);
    s.w[HZ_W_MOVES]++;
    if (!ends_turn) {
        set_meta(s, meta(s) + 2u);                                    // phase+1, :287-290
        return HZ_MOVE_OK;
    }

    // ---- _end_turn_actions (:301-329)
    return end_turn<DEFER_SCORE, REL>(s, pl, t.occ0 | bit, hand, use_explicit, explicit_code, dkey, devent, bump_event, lut, rtab);
}

// ---- one step of the uniform-random playout (fused kernel only) -------------------------------------
// The choose (:217-223): pile a becomes the hand, the piles behind it move up.
__device__ __forceinline__ uint32_t take_pile(Piles& pl, int a) {
    uint32_t hand = pl.p[0];
#pragma unroll
    for (int j = 1; j < 5; j++) hand = (a == j) ? pl.p[j] : hand;
#pragma unroll
    for (int j = 0; j < 4; j++) pl.p[j] = (j >= a) ? pl.p[j + 1] : pl.p[j];
    pl.p[4] = 0;
    return hand;
}
// A placement (:145-208 for the legal set, :250-275 for the move) on the mover's planes b[0..8] with policy draw rh:
// the tile goes on its hex and leaves the hand.  Returns the hex's bit, or 0 when no hex is legal; b and hand are then
// unchanged.  No branch: playout_round() runs six of these in a row.
__device__ __forceinline__ uint32_t place_random(uint32_t* b, uint32_t& hand, uint32_t rh) {
    struct { uint32_t occ0, occ1, occ2; } t = {b[0] | b[1] | b[2], b[3] | b[4] | b[5], b[6] | b[7] | b[8]};
    const uint32_t empty = ~t.occ0 & VALID;                            // :173
    // Stacking only ever looks at tops below level 3: where occ2 is clear the top tile is the level-1 tile if there is one,
    // else the level-0 tile, so the code bits of the top need two levels (tops_of() merges all three), and a height-1 top
    // is the level-0 code itself.
    const uint32_t T0 = b[3] | (b[0] & ~t.occ1), T1 = b[4] | (b[1] & ~t.occ1), T2 = b[5] | (b[2] & ~t.occ1);
    const uint32_t x1 = T0 & T1 & ~T2 & ~t.occ2, x3 = ~T0 & ~T1 & T2 & ~t.occ2;                 // wood / stone top, h <= 2: :183, :186
    const uint32_t x4 = ((b[0] & b[1] & ~b[2]) | (~b[1] & b[2])) & ~t.occ1;                     // wood, stone or building at h == 1: :190-192
    // Type t's legal set is m_t = empty | x_t (x_0 = x_2 = x_5 = 0) if the hand holds t, else empty.  x1, x3 and x4 lie
    // inside occ0 because records are gap-free (level l + 1 is occupied only where level l is; the stacking masks above
    // assume it too), so popc(m_t) = h_t * (popc(empty) + popc(x_t)): four popcounts, and the counts are summed as bytes
    // by multiplications.  Byte t of clo is the count of types 0..t, cum4 and n those of types 0..4 and 0..5 (n <= 138).
    const uint32_t pe = __popc(empty);
    const uint32_t hf = (hand | (hand >> 1)) & 0x555u;                    // bit 2t: the hand holds type t
    const uint32_t f03 = ((hf & 0x55u) * 0x41041u) & 0x01010101u;         // byte t: h_t, t = 0..3
    const uint32_t f45 = ((hf >> 8) * 0x41u) & 0x0101u;                   // byte t - 4: h_t, t = 4, 5
    const uint32_t clo = ((f03 * 0xFFu) & (pe * 0x01010101u + (uint32_t)__popc(x1) * 0x100u + (uint32_t)__popc(x3) * 0x1000000u)) * 0x01010101u;
    const uint32_t c45 = (f45 * 0xFFu) & (pe * 0x0101u + (uint32_t)__popc(x4));
    const uint32_t cum4 = (clo >> 24) + (c45 & 0xFFu), n = cum4 + (c45 >> 8);
    const uint32_t k = __umulhi(rh, n);
    // the type whose cumulative count covers k: the number of counts <= k, four of them at once as bytes (they are <= 92;
    // k is capped at 127 so that bit 7 of each byte of the difference says count <= k, with no borrow between bytes)
    const uint32_t d = ((min(k, 127u) * 0x01010101u) | 0x80808080u) - clo;
    const uint32_t tile = __popc(d & 0x80808080u) + (k >= cum4 ? 1u : 0u);
    // the types before it: byte `tile` of (cum4, cum3 | cum2, cum1, cum0, 0)
    const uint32_t below = __byte_perm(clo << 8, __byte_perm(clo, cum4, 0x43u), tile);
    // the type's legal set: empty plus its stacking set, picked by the flags (tile == 1, 3, 4) as byte `tile` of three
    // constants (tile <= 5); the sets are disjoint from empty and one flag at most is set, so multiply-adds do the or-ing
    const uint32_t m = empty + x1 * __byte_perm(0x100u, 0u, tile) + x3 * __byte_perm(0x1000000u, 0u, tile) +
                       x4 * __byte_perm(0u, 1u, tile);
    const uint32_t any = n != 0;                                      // shifts, not selects: a select here becomes a branch
    const uint32_t bit = any << nth_set_bit(m, (int)(k - below));
    // place the tile on level h of the hex (:257,275): the hex's bit goes into the planes of the code's set bits.  The hex
    // is free at level h (it is not in occ2: x1 and x3 exclude it, x4 excludes occ1), so adding the bit is or-ing it, and
    // the multiply-adds run on the FMA pipe
    const uint32_t code = tile + 1u;
    const uint32_t at[3] = {bit & empty, bit & t.occ0 & ~t.occ1, bit & t.occ1};
#pragma unroll
    for (int q = 0; q < 3; q++) {
        const uint32_t cq = (code >> q) & 1u;
        b[q] += at[0] * cq; b[3 + q] += at[1] * cq; b[6 + q] += at[2] * cq;
    }
    hand -= any << (2 * tile);                                        // hand.remove, :250
    return bit;
}
// legal_of + random_action + apply_move for a state whose mover is player P (a template parameter: the kernel branches on the
// player once per step, so the mover's planes are words 9P..9P+8 statically — no per-word select on the player bit and no
// swapping of the two boards when the player changes), for a move that is legal BY CONSTRUCTION: the action is
// drawn from the legal set computed here, so apply_move's validation (harmonies_engine.py:217-281) cannot fail and is not
// repeated, tile and hex are not re-derived from the action index, and the planes are updated in place (apply_move works
// on a copy because it must leave the state untouched on an error: that copy was 36 register moves per placement).
// Same draws, same result as the three calls (tests: fused playout == unfused kernels == oracle).  false: no legal move.
template <int P, bool DEFER_SCORE>
__device__ __forceinline__ bool playout_step(State& s, const NbrLut* lut, RandTab rtab) {
    const int ph = phase_of(s);
    const uint64_t r = rand64_t(rtab, key_of(s) ^ HZ_PLAYOUT_SALT, (uint64_t)s.w[HZ_W_MOVES]);
    const uint32_t rh = (uint32_t)(r >> 32);
    if (ph == HZ_PHASE_CHOOSE) {                                      // :158, :217-223
        const int np = n_piles_of(s);
        if (np == 0) return false;
        Piles pl = piles_of(s);
        const uint32_t hand = take_pile(pl, (int)__umulhi(rh, (uint32_t)np));
        set_piles(s, pl, hand, np - 1);
        set_meta(s, (meta(s) & ~0xEu) | (HZ_PHASE_PLACE1 << 1));
        s.w[HZ_W_MOVES]++;
        return true;
    }
    if (ph > HZ_PHASE_PLACE3) return false;
    uint32_t hand = hand_of(s);
    if (!place_random(&s.w[9 * P], hand, rh)) return false;
    s.w[HZ_W_PILE4H] = (s.w[HZ_W_PILE4H] & 0xFFFFu) | (hand << 16);
    s.w[HZ_W_MOVES]++;
    if (ph != HZ_PHASE_PLACE3) {
        set_meta(s, meta(s) + 2u);                                    // phase+1, :287-290
        return true;
    }
    const uint32_t occ_after = s.w[9 * P] | s.w[9 * P + 1] | s.w[9 * P + 2];
    end_turn<DEFER_SCORE, false>(s, P, occ_after, hand, false, HZ_NO_DRAW, key_of(s), s.w[HZ_W_EVENT], true, lut, rtab);
    return true;
}

// ---- one whole round of the uniform-random playout (fused kernel only) -------------------------------------------
// A round is player 0's turn and then player 1's: choose a pile, place three tiles, top the piles up — 8 actions.  From
// (player 0, CHOOSE, not ending, 5 piles) all ten random numbers of the round are known up front (8 policy draws at
// moves+0..7, the two top-ups' pile draws at events ev, ev+1), and the round is three chains that do not wait on each
// other: piles, hands and bag; player 0's placements on board 0; player 1's on board 1, which needs only player 1's
// hand from the first chain.  playout_round() is one straight-line body over registers that the compiler can interleave,
// and writes the record once; playout_step runs them one after the other with a branch on phase and player per action.
// The straight line covers the regular round: every placement has a legal hex and each top-up draws three tiles from a
// bag of 3..127 (draw_pile3's range; a game's bag never holds more than 120).  Anything else returns false with s
// untouched, and the caller plays the round with playout_step.
// Same draws, same result as eight playout_step<P, true> calls; the final scoring is left to the caller as there.
__device__ __forceinline__ bool round_ready(const State& s) {
    // the rand table covers every counter of the round (moves+7, (ev+1)*8 < RTAB_N)
    return (meta(s) & 0x1Fu) == (0u | (HZ_PHASE_CHOOSE << 1)) && n_piles_of(s) == 5 &&
           s.w[HZ_W_MOVES] <= (uint32_t)RTAB_N - 8u && s.w[HZ_W_EVENT] <= (uint32_t)RTAB_N / 8u - 2u;
}
// precondition: round_ready(s), rtab a table
__device__ __forceinline__ bool playout_round(State& s, RandTab rtab) {
    const uint64_t key = key_of(s), pkey = key ^ HZ_PLAYOUT_SALT;
    const uint32_t mv = s.w[HZ_W_MOVES], ev = s.w[HZ_W_EVENT];
    uint32_t rh[8];
#pragma unroll
    for (int i = 0; i < 8; i++) rh[i] = (uint32_t)(rand64_tab(rtab, pkey, mv + (uint32_t)i) >> 32);
    const uint64_t z0 = rand64_tab(rtab, key, ev * 8u), z1 = rand64_tab(rtab, key, (ev + 1u) * 8u);
    // piles, hands and bag: both chooses of 5 piles, both top-ups of one pile (:132-137, :217-223)
    Piles pl = piles_of(s);
    uint32_t lo = s.w[HZ_W_BAG0], hi = s.w[HZ_W_BAG1META] & 0xFFFFu;
    const uint32_t total = (uint32_t)bag_total((uint64_t)lo | ((uint64_t)hi << 32));
    uint32_t hand0 = take_pile(pl, (int)__umulhi(rh[0], 5u));
    pl.p[4] = draw_pile3(lo, hi, total, z0);
    uint32_t hand1 = take_pile(pl, (int)__umulhi(rh[4], 5u));
    pl.p[4] = draw_pile3(lo, hi, total - 3u, z1);
    // the two boards' placements, interleaved
    uint32_t b0[9], b1[9];
#pragma unroll
    for (int q = 0; q < 9; q++) { b0[q] = s.w[q]; b1[q] = s.w[9 + q]; }
    bool ok = total - 6u <= 127u - 6u;                               // 6 <= total <= 127
#pragma unroll
    for (int i = 1; i <= 3; i++) {
        ok &= place_random(b0, hand0, rh[i]) != 0u;
        ok &= place_random(b1, hand1, rh[4 + i]) != 0u;
    }
    if (!ok) return false;
#pragma unroll
    for (int q = 0; q < 9; q++) { s.w[q] = b0[q]; s.w[9 + q] = b1[q]; }
    s.w[HZ_W_BAG0] = lo;
    s.w[HZ_W_BAG1META] = (s.w[HZ_W_BAG1META] & 0xFFFF0000u) | hi;
    set_piles(s, pl, hand1, 5);       // player 0's leftover hand was replaced by player 1's choose
    // end of both turns (:301-329): 2 or fewer empty hexes after either turn ends the game after player 1's; else player 0
    // chooses next.  The bag is not empty before either top-up and both leave 5 piles, so only the boards can trigger.
    const bool trig0 = 23 - __popc(b0[0] | b0[1] | b0[2]) <= 2, trig1 = 23 - __popc(b1[0] | b1[1] | b1[2]) <= 2;
    set_meta(s, (trig0 || trig1) ? 1u | (HZ_PHASE_OVER << 1) | (1u << 4) : 0u | (HZ_PHASE_CHOOSE << 1));
    s.w[HZ_W_MOVES] = mv + 8u;
    s.w[HZ_W_EVENT] = ev + 2u;
    return true;
}

// ---- the game loop of the fused playout kernels (k_playout, k_tree_rollout_eval) ------------------------------------
// Plays s with hz_playout's semantics until the game is over, no move is legal, or max_steps actions were applied, and
// returns the number of actions applied.  The final scoring is deferred: a game that ended here is left at phase game_over
// with winner None, and the caller scores it with the lanes of the block converged (partial_scores + resolve_water).
// lut and rtab: the block's shared neighbour LUT and rand table.
__device__ __forceinline__ uint32_t play_random(State& s, int max_steps, const NbrLut* lut, RandTab rtab) {
    uint32_t k = 0;
#ifdef HZ_PLAYOUT_CHECKED   // A/B: the three general calls on a mover-relative state (validation + board copy in apply_move)
    if (player_of(s)) swap_boards(s);
    while ((int)k < max_steps && phase_of(s) != HZ_PHASE_OVER) {
        int a = random_action(s, legal_of<true>(s), rtab);
        if (a < 0) break;  // stuck position (no legal move, not over): harmonies_engine.py:205-208
        if (apply_move<true, true>(s, a, HZ_NO_DRAW, key_of(s), s.w[HZ_W_EVENT], true, lut, rtab) != HZ_MOVE_OK) break;
        k++;
    }
    if (player_of(s)) swap_boards(s);
#else
    // Whole rounds (playout_round: eight actions, both players' placements interleaved) wherever a round starts and fits
    // in max_steps, single steps elsewhere: mid-turn starts, the tail of a max_steps slice and irregular rounds.
    // HZ_PLAYOUT_STEPWISE: steps only (A/B).  A step branches on the player once: fresh games move in lockstep (same
    // player, same phase in every lane until games end), and inside a branch the mover's planes are fixed registers.
    while ((int)k < max_steps && phase_of(s) != HZ_PHASE_OVER) {
#ifndef HZ_PLAYOUT_STEPWISE
        if ((int)k <= max_steps - 8 && round_ready(s) && playout_round(s, rtab)) {
            k += 8;
            continue;
        }
#endif
        const bool ok = player_of(s) ? playout_step<1, true>(s, lut, rtab) : playout_step<0, true>(s, lut, rtab);
        if (!ok) break;  // stuck position (no legal move, not over): harmonies_engine.py:205-208
        k++;
    }
#endif
    return k;
}

// ---- canonical keys ----------------------------------------------------------------------------
// Leftmost-embedding normal form of one board under the reference's hash aliasing
// (HZ_KEY_REFERENCE in harmonies_b200.h).  Alias pairs {1,6},{2,7},{3,8} (shift 5) and
// {4,5},{9,10},{14,15},{19,20} (shift 1); a stack moves to its lower partner iff every
// earlier stack embeds strictly below that partner.
__device__ __forceinline__ void alias_normalise(Board& b) {
    uint32_t occ = b.p[0] | b.p[1] | b.p[2];
    // adjacent pairs: hi occupied, lo empty
    uint32_t m1 = occ & ~(occ << 1) & ((1u << 5) | (1u << 10) | (1u << 15) | (1u << 20));
    bool o1 = occ & 2u, o2 = occ & 4u, o3 = occ & 8u, o4 = occ & 16u, o5 = occ & 32u;
    bool o6 = occ & 64u, o7 = occ & 128u, o8 = occ & 256u;
    bool clear25 = !(o2 | o3 | o4 | o5);
    bool mv6 = o6 && !o1 && clear25;
    bool mv7 = o7 && clear25 && (o6 ? mv6 : true);
    bool mv8 = o8 && !(o3 | o4 | o5) && (o7 ? mv7 : (o6 ? mv6 : true));
    uint32_t m5 = (mv6 ? 64u : 0u) | (mv7 ? 128u : 0u) | (mv8 ? 256u : 0u);
    uint32_t keep = ~(m1 | m5);
#pragma unroll
    for (int k = 0; k < 9; k++) b.p[k] = (b.p[k] & keep) | ((b.p[k] & m1) >> 1) | ((b.p[k] & m5) >> 5);
}
__device__ __forceinline__ uint64_t hash_step(uint64_t h, uint32_t x) {
    h = (h ^ x) * 0x9FB21C651E98DF25ull;
    return h ^ (h >> 32);
}
// key words: 23 words of canonical identity (mode-normalised)
__device__ __forceinline__ void key_words(const State& s, int mode, uint32_t k[HZ_CANON_WORDS]) {
    if (mode == HZ_KEY_REFERENCE) {
        Board b0 = board_of(s, 0), b1 = board_of(s, 1);
        alias_normalise(b0); alias_normalise(b1);
#pragma unroll
        for (int i = 0; i < 9; i++) { k[i] = b0.p[i]; k[9 + i] = b1.p[i]; }
    } else {
#pragma unroll
        for (int i = 0; i < 18; i++) k[i] = s.w[i];
    }
    k[18] = s.w[18]; k[19] = s.w[19]; k[20] = s.w[20]; k[21] = s.w[21];
    k[22] = s.w[22] & 0x0FFFFFFFu;
}
__device__ __forceinline__ uint64_t hash_key_words(const uint32_t k[HZ_CANON_WORDS]) {
    uint64_t h = 0x9E3779B97F4A7C15ull;
#pragma unroll
    for (int i = 0; i < HZ_CANON_WORDS; i++) h = hash_step(h, k[i]);
    return mix64(h);
}
__device__ __forceinline__ uint64_t canon_hash(const State& s, int mode) {
    uint32_t k[HZ_CANON_WORDS];
    key_words(s, mode, k);
    return hash_key_words(k);
}

// ---- state tensors (process_game_state.py:15-137): per-channel hex masks + global features ----
__constant__ uint8_t CELL_HEX[35] = {31, 31, 4, 9, 14, 19, 22, 31, 31, 5, 10, 15, 20, 31, 31, 1, 6, 11,
                                     16, 21, 31, 31, 2, 7, 12, 17, 31, 31, 0, 3, 8, 13, 18, 31, 31};

template <typename T> __device__ __forceinline__ T cvt(float v);
template <> __device__ __forceinline__ float cvt<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 cvt<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// channel mask c (<38) of a state given its words; bit i = value at hex i is non-zero
__device__ __forceinline__ uint32_t channel_mask(const uint32_t* w, int c) {
    if (c < 36) {
        int p = c / 18, r = c - 18 * p, t = r / 3, l = r - 3 * t;
        const uint32_t* pl = w + p * 9 + l * 3;
        uint32_t code = (uint32_t)t + 1u;
        uint32_t a = pl[0], b = pl[1], d = pl[2];
        return ((code & 1u) ? a : ~a) & ((code & 2u) ? b : ~b) & ((code & 4u) ? d : ~d) & VALID;  // :43-67
    }
    uint32_t m = w[HZ_W_BAG1META] >> 24;
    if (c == 36) return (m & 1u) ? VALID : 0u;                       // :70-71
    uint32_t ph = (m >> 1) & 7u;
    return (ph >= 1 && ph <= 3) ? VALID : 0u;                        // :74-81 (phase 0 and game_over -> 0)
}
// the 38 channel bits of the cell at hex hx (0 for the padding cells, hx >= 23): a cell holds at most 3+3 tiles, so
// each (player p, level l) sets the bit p*18 + (code-1)*3 + l of its tile code instead of probing 38 masks; bit 36 is
// player 1, bit 37 phase 1-3
__device__ __forceinline__ uint64_t cell_bits(const uint32_t* w, int hx) {
    if (hx >= 23) return 0;
    uint64_t bits = 0;
#pragma unroll
    for (int pl = 0; pl < 6; pl++) {
        uint32_t code = ((w[pl * 3] >> hx) & 1u) | (((w[pl * 3 + 1] >> hx) & 1u) << 1) | (((w[pl * 3 + 2] >> hx) & 1u) << 2);
        int p = pl / 3, l = pl - 3 * p;
        if (code) bits |= 1ull << (p * 18 + ((int)code - 1) * 3 + l);
    }
    uint32_t m = w[HZ_W_BAG1META] >> 24, ph = (m >> 1) & 7u;
    if (m & 1u) bits |= 1ull << 36;
    if (ph >= 1 && ph <= 3) bits |= 1ull << 37;
    return bits;
}
// fp32(k / 3.0) for k = 0..3 by selects (a local array would live in local memory); 1 for k > 3
__device__ __forceinline__ float third(uint32_t k) {
    return k == 0 ? 0.0f : k == 1 ? (float)(1.0 / 3.0) : k == 2 ? (float)(2.0 / 3.0) : 1.0f;
}
// the value of the phase plane (channel 37) where it is set, i.e. in phases 1-3: the reference's phase / 3.0
__device__ __forceinline__ float phase_value(const uint32_t* w) { return third((w[HZ_W_BAG1META] >> 25) & 7u); }
// the one-hot table of the vector stores: VEC = 16 / sizeof(T) bits -> 16 bytes of T 0.0 / 1.0 (16 entries for fp32,
// 256 for bf16), built by the whole block (not unrolled: with a blockDim.x stride that would cost a trip-count division)
template <typename T>
__device__ __forceinline__ void build_onehot_lut(uint4* lut) {
    constexpr int VEC = 16 / (int)sizeof(T);
#pragma unroll 1
    for (int i = threadIdx.x; i < (1 << VEC); i += blockDim.x) {
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; j++)
            o[j] = VEC == 4 ? (((i >> j) & 1) ? 0x3F800000u : 0u)
                            : (((i >> (2 * j)) & 1) ? 0x3F80u : 0u) | (((i >> (2 * j + 1)) & 1) ? 0x3F800000u : 0u);
        lut[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}
__device__ __forceinline__ float global_feature(const uint32_t* w, int g) {
    if (g < 30) {                                                    // :98-107
        int i = g / 6, t = g - 6 * i;
        uint32_t np = (w[HZ_W_BAG1META] >> 16) & 0xFFu;
        uint32_t word = w[HZ_W_PILES01 + (i >> 1)];
        uint32_t code = (i & 1) ? (word >> 16) : (word & 0xFFFFu);
        return (uint32_t)i < np ? third((code >> (2 * t)) & 3u) : 0.0f;
    }
    if (g < 36) return third(((w[HZ_W_PILE4H] >> 16) >> (2 * (g - 30))) & 3u);   // :112-118
    int t = g - 36;                                                  // :122-130
    uint32_t cnt = t < 4 ? (w[HZ_W_BAG0] >> (8 * t)) & 0xFFu : (w[HZ_W_BAG1META] >> (8 * (t - 4))) & 0xFFu;
    // The reference divides in double and stores to fp32.  A correctly rounded fp32 division of
    // the two small integers gives the same bits: c/init is exact or has a binary period of at
    // most 22 bits (init <= 23), so its 53-bit rounding can never land on an fp32 midpoint.
    return __fdiv_rn((float)cnt, (float)INIT_BAG[t]);
}

// ---- warp-level state encoding: one warp per record, one scalar store per element ------------
// LAYOUT: HZ_LAYOUT_NCHW, HZ_LAYOUT_NHWC, or HZ_LAYOUT_NHWC40 (channel stride 40, channels 38
// and 39 written as zero: the stem convolution then needs no cuDNN input-padding kernel)
template <int LAYOUT> struct RowElems { static constexpr int value = LAYOUT == HZ_LAYOUT_NHWC40 ? 1400 : 1330; };   // (T16K never takes the generic path)
template <typename T, int LAYOUT>
__device__ __forceinline__ void warp_encode(const uint32_t* w, uint32_t* smask, T* board, T* glob, int lane) {
    for (int c = lane; c < 40; c += 32) smask[c] = c < 38 ? channel_mask(w, c) : 0u;
    __syncwarp();
    float phase_val = phase_value(w);
    for (int e = lane; e < RowElems<LAYOUT>::value; e += 32) {
        int c, cell;
        if (LAYOUT == HZ_LAYOUT_NHWC40) { cell = e / 40; c = e - 40 * cell; }
        else if (LAYOUT == HZ_LAYOUT_NHWC) { cell = e / 38; c = e - 38 * cell; }
        else { c = e / 35; cell = e - 35 * c; }
        uint32_t bit = (smask[c] >> CELL_HEX[cell]) & 1u;
        board[e] = cvt<T>(bit ? (c == 37 ? phase_val : 1.0f) : 0.0f);
    }
    for (int g = lane; g < 42; g += 32) glob[g] = cvt<T>(global_feature(w, g));
    __syncwarp();
}


// ---- new game (harmonies_engine.py:66-79) ---------------------------------------------------------
__device__ __forceinline__ void init_state(State& s, uint64_t key, RandTab rtab = nullptr) {
#pragma unroll
    for (int i = 0; i < SW; i++) s.w[i] = 0;
    uint64_t bag = 23ull | (19ull << 8) | (21ull << 16) | (23ull << 24) | (15ull << 32) | (19ull << 40);
    Piles P;
#pragma unroll
    for (int k = 0; k < 5; k++) P.p[k] = draw_pile(bag, rand64_t(rtab, key, (uint64_t)k));   // event 0
    s.w[HZ_W_KEYLO] = (uint32_t)key; s.w[HZ_W_KEYHI] = (uint32_t)(key >> 32);
    s.w[HZ_W_EVENT] = 1;
    set_bag(s, bag);
    set_piles(s, P, 0, 5);
}

}  // namespace hz
