// hz_engine.cu — batched engine kernels (sm_100a) behind the C ABI of
// include/harmonies_b200.h: new games, legal masks, move application, scoring, state
// encoding, canonical keys, outcomes, random-playout policy and the fused playout.
//
// Mapping: one thread per game, state held in registers (7 x LDG.128 in, 8 x STG.128 out),
// hex-parallel work done as 23-bit bit-board arithmetic; the neighbour expansion LUT lives in
// 3 KB of shared memory per block.  hz_encode is write-bound (5.5 KB out per 128 B in) and one
// launch of k_encode: a warp renders a group of records as a bit stream and stores 16-byte vectors
// through a lookup table, and encodes the records outside whole aligned groups one by one with
// scalar stores (warp_encode); hz_greedy_actions is warp-per-game with one lane per legal move.
#include "hz_common.cuh"
#include "hz_core.cuh"

namespace hz {

constexpr int TPB = 128;

__global__ void __launch_bounds__(TPB) k_init(void* states, int64_t n, const uint64_t* keys,
                                              uint64_t seed, uint64_t first_id) {
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (g >= n) return;
    State s;
    init_state(s, keys ? keys[g] : rand64(seed, first_id + (uint64_t)g));
    store_state(s, states, g);
}

__global__ void __launch_bounds__(TPB) k_legal(const void* states, int64_t n, uint32_t* mask) {
    __shared__ __align__(16) uint4 tile[TPB / 32][256];
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    State s;
    load_state_warp<6>(s, states, g - (threadIdx.x & 31), n, tile[threadIdx.x >> 5]);   // legal moves read words 0..22 only
    uint32_t out[5];
    legal_words(legal_of(s), out);
    // the warp's 32 x 5 mask words leave as five coalesced 128-byte stores, through the same tile (stride 5: conflict-free)
    uint32_t* tw = reinterpret_cast<uint32_t*>(tile[threadIdx.x >> 5]);
    const int lane = threadIdx.x & 31;
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 5; k++) tw[lane * 5 + k] = out[k];
    __syncwarp();
    const int64_t g0 = g - lane, lim = (n - g0) * 5;
#pragma unroll
    for (int k = 0; k < 5; k++)
        if (k * 32 + lane < lim) mask[g0 * 5 + k * 32 + lane] = tw[k * 32 + lane];
}

__global__ void __launch_bounds__(TPB) k_apply(void* states, int64_t n, const int16_t* actions,
                                               const uint16_t* draws, uint8_t* status) {
    __shared__ NbrLut lut;
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    State s;
    if (g < n) load_state(s, states, g);      // issue the record loads first: the LUT copy overlaps them
    build_nbr_lut(&lut);
    __syncthreads();
    if (g >= n) return;
    uint32_t ex = draws ? (uint32_t)draws[g] : (uint32_t)HZ_NO_DRAW;
    int st = apply_move(s, (int)actions[g], ex, key_of(s), s.w[HZ_W_EVENT], true, &lut);
    if (st == HZ_MOVE_OK) store_state(s, states, g);
    if (status) status[g] = (uint8_t)st;
}

// ---- the reference's private turn helpers, for callers that drive them directly (GUI/main.py:364-365,
// harness code): _end_turn_actions (:301-329), _replenish_piles (:132-137), _draw_tiles (:120-130)
__global__ void __launch_bounds__(TPB) k_end_turn(void* states, int64_t n, const uint16_t* draws, uint8_t* status) {
    __shared__ NbrLut lut;
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    State s;
    if (g < n) load_state(s, states, g);
    build_nbr_lut(&lut);
    __syncthreads();
    if (g >= n) return;
    uint32_t ex = draws ? (uint32_t)draws[g] : (uint32_t)HZ_NO_DRAW;
    bool use_explicit = ex != HZ_NO_DRAW && n_piles_of(s) < 5;
    int st = HZ_MOVE_OK;
    if (use_explicit && !pile_available(bag_of(s), ex)) st = HZ_MOVE_BAD_DRAW;
    else {
        int pl = player_of(s);
        Tops t = tops_of(board_of(s, pl));
        st = end_turn<false, false>(s, pl, t.occ0, hand_of(s), use_explicit, ex, key_of(s), s.w[HZ_W_EVENT], true, &lut, nullptr);
        store_state(s, states, g);
    }
    if (status) status[g] = (uint8_t)st;
}

__global__ void __launch_bounds__(TPB) k_replenish(void* states, int64_t n) {
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (g >= n) return;
    State s;
    load_state(s, states, g);
    int np;
    replenish_piles(s, hand_of(s), false, 0u, key_of(s), s.w[HZ_W_EVENT], nullptr, np);
    s.w[HZ_W_EVENT]++;
    store_state(s, states, g);
}

// draws min(count, bag total) tiles one by one, uniformly without replacement from the bag multiset
// (random.sample over the flattened bag, :122-129), with the arithmetic of draw_pile; tiles[g][0..14] =
// tile types in draw order, tiles[g][15] = how many were drawn.  One draw event of the state's stream.
__global__ void __launch_bounds__(TPB) k_draw_tiles(void* states, int64_t n, int count, uint8_t* tiles) {
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (g >= n) return;
    State s;
    load_state(s, states, g);
    uint64_t bag = bag_of(s), key = key_of(s);
    int total = bag_total(bag), drawn = 0;
    for (int grp = 0; grp < 5 && drawn < count && total > 0; grp++) {
        uint64_t z = rand64(key, (uint64_t)s.w[HZ_W_EVENT] * 8 + (uint64_t)grp);
        for (int j = 0; j < 3 && drawn < count && total > 0; j++) {
            uint32_t x = (uint32_t)(z >> (21 * j)) & 0x1FFFFFu;
            uint32_t r = (x * (uint32_t)total) >> 21;
            int t = 0;
            uint32_t cum = 0;
            for (; t < 5; t++) {
                cum += (uint32_t)(bag >> (8 * t)) & 0xFFu;
                if (cum > r) break;
            }
            bag -= 1ull << (8 * t);
            total--;
            tiles[g * 16 + drawn++] = (uint8_t)t;
        }
    }
    tiles[g * 16 + 15] = (uint8_t)drawn;
    set_bag(s, bag);
    s.w[HZ_W_EVENT]++;
    store_state(s, states, g);
}

__global__ void __launch_bounds__(TPB) k_score(const void* states, int64_t n, int16_t* scores,
                                               int16_t* terms) {
    __shared__ NbrLut lut;
    __shared__ WaterQueue<2 * TPB, 2 * TPB> wq;
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    // only the 18 board words are needed: 92 -> 80 B of traffic per position; the loads are
    // issued before the LUT copy so that the two overlap
    uint32_t w[20];
    if (g < n) {
        const uint4* p = reinterpret_cast<const uint4*>(states) + g * 8;
#pragma unroll
        for (int k = 0; k < 5; k++) {
            uint4 v = p[k];
            w[4 * k] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
        }
    }
    build_nbr_lut(&lut);
    water_queue_init(&wq);
    __syncthreads();
    int t[2][5];
    if (g < n) {
#pragma unroll
        for (int pl = 0; pl < 2; pl++) {
            Board b;
#pragma unroll
            for (int k = 0; k < 9; k++) b.p[k] = w[pl * 9 + k];
            score_board(&lut, b, t[pl], &wq, (int)threadIdx.x * 2 + pl);
        }
    }
    __syncthreads();
    resolve_water(&lut, &wq);          // the rare large water components, one warp each
    __syncthreads();
    if (g >= n) return;
#pragma unroll
    for (int pl = 0; pl < 2; pl++) {
        t[pl][4] += wq.extra[threadIdx.x * 2 + pl];
        if (terms) {
#pragma unroll
            for (int k = 0; k < 5; k++) terms[(g * 2 + pl) * 5 + k] = (int16_t)t[pl][k];
        }
        if (scores) scores[g * 2 + pl] = (int16_t)(t[pl][0] + t[pl][1] + t[pl][2] + t[pl][3] + t[pl][4]);
    }
}

// (the warp-staged load of k_legal was measured here too: 32.8 us against 29.7 us per 1 M records — the hash has enough
// arithmetic per record to hide the direct loads, and the staging adds a barrier in front of it)
__global__ void __launch_bounds__(TPB) k_hash(const void* states, int64_t n, int mode, uint64_t* out) {
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (g >= n) return;
    State s;
    load_state(s, states, g);
    out[g] = canon_hash(s, mode);
}

__global__ void __launch_bounds__(TPB) k_outcome(const void* states, int64_t n, uint8_t* over, int8_t* outcome) {
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (g >= n) return;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(states) + g * 32;
    State s;
    s.w[HZ_W_BAG1META] = w[HZ_W_BAG1META];
    if (over) over[g] = is_over(s) ? 1 : 0;
    if (outcome) outcome[g] = (int8_t)(is_over(s) ? outcome_of(s) : 0);
}

__global__ void __launch_bounds__(TPB) k_random_actions(const void* states, int64_t n, int16_t* actions) {
    int64_t g = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (g >= n) return;
    State s;
    load_state(s, states, g);
    actions[g] = (int16_t)random_action(s, legal_of(s));
}

// choose_move_greedy (evaluation.py:137-196): one warp per game, one lane per legal move; a lane
// places its tile on a copy of the mover's board, scores it (K2+K3 fused) and the warp keeps the
// first strict maximum in ascending action order.  Taking a pile never changes the mover's
// score, so in the choose phase the first pile wins, as in the reference's loop.
constexpr int GWPB = 4;
__global__ void __launch_bounds__(GWPB * 32) k_greedy(const void* states, int64_t n, int16_t* actions) {
    __shared__ NbrLut lut;
    __shared__ uint32_t sw[GWPB][32];
    build_nbr_lut(&lut);
    __syncthreads();
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t g = (int64_t)blockIdx.x * GWPB + warp;
    if (g >= n) return;
    sw[warp][lane] = reinterpret_cast<const uint32_t*>(states)[g * 32 + lane];
    __syncwarp();
    State s;
#pragma unroll
    for (int i = 0; i < SW; i++) s.w[i] = sw[warp][i];
    Legal L = legal_of(s);
    int nl = legal_count(L), best_k = -1, best_score = -1000000;
    if (L.n_piles > 0) {
        best_k = 0;
    } else {
        Board b0 = board_of(s, player_of(s));
        Tops t = tops_of(b0);
        for (int base = 0; base < nl; base += 32) {
            int k = base + lane;
            if (k < nl) {
                int a = kth_action(L, k);
                int tile = (a - 5) / 23, hex = (a - 5) - 23 * tile;
                uint32_t bit = 1u << hex, code = (uint32_t)tile + 1u;
                uint32_t at0 = bit & ~t.occ0, at1 = bit & t.occ0 & ~t.occ1, at2 = bit & t.occ1;
                Board b = b0;
#pragma unroll
                for (int q = 0; q < 3; q++) {
                    uint32_t on = (code >> q) & 1u ? 0xFFFFFFFFu : 0u;
                    b.p[q] |= at0 & on; b.p[3 + q] |= at1 & on; b.p[6 + q] |= at2 & on;
                }
                int tm[5];
                score_board(&lut, b, tm);
                int sc = tm[0] + tm[1] + tm[2] + tm[3] + tm[4];
                if (sc > best_score) { best_score = sc; best_k = k; }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            int os = __shfl_xor_sync(0xFFFFFFFFu, best_score, o), ok = __shfl_xor_sync(0xFFFFFFFFu, best_k, o);
            bool take = ok >= 0 && (best_k < 0 || os > best_score || (os == best_score && ok < best_k));
            if (take) { best_score = os; best_k = ok; }
        }
    }
    if (lane == 0) actions[g] = (int16_t)(best_k < 0 ? -1 : kth_action(L, best_k));
}

// Fused playout (K9): the whole game stays in registers; HBM sees one load and one store of
// the state per game.  Threads of a warp run different games and diverge only on the phase
// (choose / place / end of turn); scoring runs once per game.
constexpr int PTPB = 64;   // 65,536 games -> 1024 blocks: 6.9 per SM, <2 % tail imbalance over 148 SMs
// FROM_KEYS: the game is created in registers from its 64-bit key (k_init fused in) and only
// (meta word, score word, actions played) leave the chip: 8 B in, 12 B out per game.
// 7 blocks per SM hold a 65,536-game wave: the register cap of 7 x 64 threads (<= 144 per thread) leaves the round path
// room without spills, where the compiler's own choice for __launch_bounds__(PTPB) alone was 80 registers and a spill.
#ifdef HZ_PLAYOUT_TIMELINE
// Device-side phase timeline of k_playout, profiling builds only (profiles/playout_timeline.py).  Per warp TL_WORDS
// uint64: [0] %smid, then per event e the pair [1 + 2e] %globaltimer (ns), [2 + 2e] clock64 (SM cycles), written by the
// warp's lowest active lane.  Events: kernel entry, tables ready (after the block barrier), records in registers, end of
// play_random, after partial_scores, after resolve_water, after the store, and TL_ROUND + i at the end of play_random's
// loop iteration i (a whole round on the round path; iterations >= TL_ROUNDS - 1 share the last slot).
enum { TL_ENTRY, TL_TABLES, TL_RECORDS, TL_PLAYED, TL_PARTIAL, TL_RESOLVED, TL_STORED, TL_ROUND };
constexpr int TL_ROUNDS = 24, TL_WORDS = 64, TL_SINK = 63;
static_assert(1 + 2 * (TL_ROUND + TL_ROUNDS) <= TL_SINK, "timeline slots overlap the sink word");
__device__ unsigned long long* g_tl = nullptr;
__device__ long long g_tl_warps = 0;
// dep: a value the stamp must wait for (the volatile store to the sink word orders the clock reads after its arrival)
__device__ __forceinline__ void tl_mark(unsigned long long* w, int e, uint32_t dep = 0) {
    if (w && (int)(threadIdx.x & 31) == __ffs(__activemask()) - 1) {
        *reinterpret_cast<volatile unsigned long long*>(w + TL_SINK) = dep;
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory");
        w[1 + 2 * e] = t;
        w[2 + 2 * e] = clock64();
    }
}
struct TlRoundMark {
    unsigned long long* w;
    __device__ __forceinline__ void operator()(int i) const { tl_mark(w, TL_ROUND + min(i, TL_ROUNDS - 1)); }
};
#define HZ_TL(e, ...) tl_mark(tl, e, ##__VA_ARGS__)
#else
#define HZ_TL(e, ...) do { } while (0)
#endif

// The block's two tables (3 KB neighbour LUT, 4 KB rand table) in one round trip: each thread issues all of its 16 loads
// before its first shared-memory store.  build_nbr_lut / build_rand_table loop over blockDim.x and wait for one batch of
// loads per iteration: four round trips in a row, 2.3-2.4 us of a 65,536-game wave on a B200 at 1,000 W (playout_timeline.py)
// during which no warp of the SM has anything else to do.  -DHZ_PLAYOUT_LOOPED_TABLES keeps the looped copy (A/B).
struct PlayoutTables {
    uint32_t lut[768 / PTPB];
    uint4 rt[RTAB_N / 2 / PTPB];
};
static_assert(768 % PTPB == 0 && (RTAB_N / 2) % PTPB == 0, "k_playout's table copy: whole rows per thread");
__device__ __forceinline__ void fetch_tables(PlayoutTables& t) {
#pragma unroll
    for (int i = 0; i < 768 / PTPB; i++) t.lut[i] = __ldg(NBR_LUT_G + threadIdx.x + i * PTPB);
#pragma unroll
    for (int i = 0; i < RTAB_N / 2 / PTPB; i++) t.rt[i] = __ldg(reinterpret_cast<const uint4*>(RAND_TAB_G) + threadIdx.x + i * PTPB);
}
__device__ __forceinline__ void store_tables(const PlayoutTables& t, NbrLut* lut, uint64_t* rtab) {
#pragma unroll
    for (int i = 0; i < 768 / PTPB; i++) (&lut->t[0][0])[threadIdx.x + i * PTPB] = t.lut[i];
#pragma unroll
    for (int i = 0; i < RTAB_N / 2 / PTPB; i++) reinterpret_cast<uint4*>(rtab)[threadIdx.x + i * PTPB] = t.rt[i];
}

template <bool FROM_KEYS>
__global__ void __launch_bounds__(PTPB, 7) k_playout(void* states, int64_t n, int max_steps, uint32_t* steps,
                                                  unsigned long long* total_steps, const uint64_t* keys,
                                                  uint64_t seed, uint64_t first_id, uint32_t* results) {
    __shared__ NbrLut lut;
    __shared__ __align__(16) uint64_t rtab_s[RTAB_N];
    __shared__ WaterQueue<2 * PTPB, 2 * PTPB> wq;
#ifdef HZ_PLAYOUT_TIMELINE
    unsigned long long* tl = nullptr;
    {
        const long long warp = ((long long)blockIdx.x * PTPB + threadIdx.x) >> 5;
        if (g_tl && warp < g_tl_warps) tl = g_tl + warp * TL_WORDS;
        uint32_t smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        if (tl && (threadIdx.x & 31) == 0) tl[0] = smid;
        HZ_TL(TL_ENTRY);
    }
#endif
#ifdef HZ_PLAYOUT_LOOPED_TABLES
    build_nbr_lut(&lut);
    build_rand_table(rtab_s);
#else
    {
        PlayoutTables tabs;
        fetch_tables(tabs);
        store_tables(tabs, &lut, rtab_s);
    }
#endif
    const RandTab rtab = rand_table_handle(rtab_s);
    water_queue_init(&wq);
    __syncthreads();
    HZ_TL(TL_TABLES);
    int64_t g = (int64_t)blockIdx.x * PTPB + threadIdx.x;
    uint32_t k = 0;
    State s;
    bool fin = false;
    int s0 = 0, s1 = 0;
    if (g < n) {
        if (FROM_KEYS) init_state(s, keys ? keys[g] : rand64(seed, first_id + (uint64_t)g), rtab);
        else load_state(s, states, g);
#ifdef HZ_PLAYOUT_TIMELINE
        uint32_t dep = 0;
#pragma unroll
        for (int i = 0; i < SW; i++) dep ^= s.w[i];
        HZ_TL(TL_RECORDS, dep);
        k = play_random(s, max_steps, &lut, rtab, TlRoundMark{tl});
        HZ_TL(TL_PLAYED);
#else
        k = play_random(s, max_steps, &lut, rtab);
#endif
        // final scoring deferred to here: the lanes of the warp are converged again; rivers of >= 5
        // hexes go to the block's queue and get a whole warp each (resolve_water)
        fin = phase_of(s) == HZ_PHASE_OVER && winner_code(s) == 0;
        if (fin) partial_scores(s, &lut, &wq, s0, s1);
        HZ_TL(TL_PARTIAL);
    }
    __syncthreads();
    resolve_water(&lut, &wq);
    __syncthreads();
    HZ_TL(TL_RESOLVED);
    if (g < n) {
        if (fin) store_final_scores(s, s0 + wq.extra[threadIdx.x * 2], s1 + wq.extra[threadIdx.x * 2 + 1]);
        if (FROM_KEYS) {
            results[g * 3] = s.w[HZ_W_BAG1META];
            results[g * 3 + 1] = s.w[HZ_W_SCORES];
            results[g * 3 + 2] = s.w[HZ_W_MOVES];
        } else {
            store_state(s, states, g);
            if (steps) steps[g] = k;
        }
    }
    HZ_TL(TL_STORED);
    if (total_steps) {
        uint32_t sum = k;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
        if ((threadIdx.x & 31) == 0 && sum) atomicAdd(total_steps, (unsigned long long)sum);
    }
}

// ---- encode (process_game_state.py:15-137) ------------------------------------------------------
// One WARP renders a group of G records (G*1330 elements = 665 16-byte vectors: G = 2 for fp32,
// 4 for bf16) with no block-level barrier at all — each warp has its own staging area and only
// __syncwarp()s, so the SM always has other warps to issue from.  The tensor is ~94 % zeros and
// every non-zero is 1.0 except the phase plane, so the group is first rendered as a BIT stream in
// output order (1 bit per element) and a store is then one table lookup: VEC bits -> 16 bytes of
// 0.0/1.0 (then the phase patch).  The records outside whole groups at a 16-byte-aligned board
// (the n mod G last ones, or all of them when the board is not aligned) are work items of the same
// loop, one warp per record with scalar stores (warp_encode).
constexpr int ENC_WARPS = 8;
template <typename T, bool NHWC>
__global__ void __launch_bounds__(ENC_WARPS * 32) k_encode(const void* states, int64_t n, T* board, T* glob) {
    constexpr int VEC = 16 / (int)sizeof(T);
    constexpr int G = VEC / 2;                       // 2 (fp32) or 4 (bf16) records per group
    constexpr int NV = G * 1330 / VEC;               // 665 vectors per group
    constexpr int SWORDS = (G * 1330 + 31) / 32 + 3;
    constexpr int ROWS = NHWC ? 35 : 38, ROW_BITS = NHWC ? 38 : 35;
    __shared__ __align__(16) uint32_t sw[ENC_WARPS][G][32];
    __shared__ uint32_t smask[ENC_WARPS][G][40];
    __shared__ uint32_t stream[ENC_WARPS][SWORDS], pstream[ENC_WARPS][SWORDS];
    __shared__ uint32_t sphase_bits[ENC_WARPS][G];
    __shared__ uint64_t perm[3][256];   // hex-order byte -> cell-order bits (NCHW rows)
    __shared__ uint4 vlut[1 << VEC];
    __shared__ uint8_t scell[36];       // shared copy: per-lane indices into __constant__ would serialise
    if (threadIdx.x < 35) scell[threadIdx.x] = CELL_HEX[threadIdx.x];
    build_onehot_lut<T>(vlut);
    if (!NHWC) {
        for (int e = threadIdx.x; e < 768; e += ENC_WARPS * 32) {
            int c = e >> 8, v = e & 255;
            uint64_t m = 0;
            for (int b = 0; b < 8; b++) {
                int i = c * 8 + b;
                if (((v >> b) & 1) && i < 23) m |= 1ull << HEX_CELL[i];
            }
            perm[c][v] = m;
        }
    }
    __syncthreads();                                  // the only block barrier: tables are ready
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* my_stream = stream[warp];
    uint32_t* my_pstream = pstream[warp];
    const int64_t n_warps = (int64_t)gridDim.x * ENC_WARPS;
    const int64_t n_groups = ((uintptr_t)board & 15) == 0 ? n / G : 0;   // the vector stores need an aligned base
    const int64_t n_items = n - n_groups * (G - 1);   // the groups, then one item per remaining record
    for (int64_t item = (int64_t)blockIdx.x * ENC_WARPS + warp; item < n_items; item += n_warps) {
        if (item >= n_groups) {
            const int64_t r = item + n_groups * (G - 1);
            sw[warp][0][lane] = reinterpret_cast<const uint32_t*>(states)[r * 32 + lane];
            __syncwarp();
            warp_encode<T, NHWC ? HZ_LAYOUT_NHWC : HZ_LAYOUT_NCHW>(sw[warp][0], smask[warp][0], board + r * 1330, glob + r * 42, lane);
            continue;
        }
        const int64_t base = item * G;
        for (int i = lane; i < G * 8; i += 32)
            reinterpret_cast<uint4*>(&sw[warp][0][0])[i] = reinterpret_cast<const uint4*>(states)[base * 8 + i];
        for (int i = lane; i < SWORDS; i += 32) { my_stream[i] = 0; my_pstream[i] = 0; }
        __syncwarp();
        // channel masks (hex order, NCHW rows) and the 42 global features of each record
        for (int it = lane; it < G * 80; it += 32) {
            int s = it / 80, c = it - 80 * s;
            const uint32_t* w = sw[warp][s];
            if (c >= 38) glob[(base + s) * 42 + (c - 38)] = cvt<T>(global_feature(w, c - 38));
            else if (!NHWC) smask[warp][s][c] = channel_mask(w, c);
        }
        if (lane < G) {
            float pv = phase_value(sw[warp][lane]);
            sphase_bits[warp][lane] = VEC == 4 ? __float_as_uint(pv) : (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(pv));
        }
        __syncwarp();
        // bit streams in output order: one task per (record, cell) [NHWC] or (record, channel) [NCHW]
        for (int it = lane; it < G * ROWS; it += 32) {
            int s = it / ROWS, row = it - ROWS * s;
            uint64_t bits;
            if (NHWC) {
                bits = cell_bits(sw[warp][s], scell[row]);
            } else {
                uint32_t m = smask[warp][s][row];                      // hex order -> cell order: 3 table lookups
                bits = perm[0][m & 255] | perm[1][(m >> 8) & 255] | perm[2][(m >> 16) & 127];
            }
            if (bits) {
                int off = s * 1330 + row * ROW_BITS, wd = off >> 5, sh = off & 31;
                uint64_t lo = bits << sh;
                uint32_t hi = sh ? (uint32_t)(bits >> (64 - sh)) : 0u;
                if ((uint32_t)lo) atomicOr(&my_stream[wd], (uint32_t)lo);
                if ((uint32_t)(lo >> 32)) atomicOr(&my_stream[wd + 1], (uint32_t)(lo >> 32));
                if (hi) atomicOr(&my_stream[wd + 2], hi);
                // second stream: the set elements of the phase plane (channel 37, value k/3)
                uint64_t pbits = NHWC ? (bits & (1ull << 37)) : (row == 37 ? bits : 0ull);
                if (pbits) {
                    uint64_t plo = pbits << sh;
                    uint32_t phi = sh ? (uint32_t)(pbits >> (64 - sh)) : 0u;
                    if ((uint32_t)plo) atomicOr(&my_pstream[wd], (uint32_t)plo);
                    if ((uint32_t)(plo >> 32)) atomicOr(&my_pstream[wd + 1], (uint32_t)(plo >> 32));
                    if (phi) atomicOr(&my_pstream[wd + 2], phi);
                }
            }
        }
        __syncwarp();
        uint4* out = reinterpret_cast<uint4*>(board + base * 1330);   // G*1330*sizeof(T) is a multiple of 16
        for (int v = lane; v < NV; v += 32) {
            int e0 = v * VEC;
            uint32_t nib = (my_stream[e0 >> 5] >> (e0 & 31)) & ((1u << VEC) - 1u);   // VEC divides 32: never straddles
            uint32_t pm = (my_pstream[e0 >> 5] >> (e0 & 31)) & ((1u << VEC) - 1u);
            uint4 o = vlut[nib];
            while (pm) {                                             // phase-plane elements hold k/3, not 1.0
                int j = __ffs(pm) - 1;
                pm &= pm - 1;
                uint32_t pb = sphase_bits[warp][(e0 + j) / 1330];
                int wi = VEC == 4 ? j : (j >> 1);
                uint32_t cur = wi == 0 ? o.x : wi == 1 ? o.y : wi == 2 ? o.z : o.w;
                uint32_t nw = VEC == 4 ? pb : ((j & 1) ? ((cur & 0x0000FFFFu) | (pb << 16)) : ((cur & 0xFFFF0000u) | pb));
                o.x = wi == 0 ? nw : o.x; o.y = wi == 1 ? nw : o.y; o.z = wi == 2 ? nw : o.z; o.w = wi == 3 ? nw : o.w;
            }
            out[v] = o;
        }
        __syncwarp();
    }
}

}  // namespace hz

using namespace hz;

static inline int blocks_for(int64_t n, int tpb) { return (int)((n + tpb - 1) / tpb); }

extern "C" {

int hz_init_states(void* states, int64_t n, const uint64_t* keys, uint64_t seed, uint64_t first_id, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || n < 0) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_init<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, keys, seed, first_id);
    return hz_launched(1);
}

int hz_legal_mask(const void* states, int64_t n, uint32_t* mask, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || !mask || n < 0) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_legal<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, mask);
    return hz_launched(1);
}

int hz_apply(void* states, int64_t n, const int16_t* actions, const uint16_t* draws, uint8_t* status, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || !actions || n < 0) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_apply<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, actions, draws, status);
    return hz_launched(1);
}

int hz_end_turn(void* states, int64_t n, const uint16_t* draws, uint8_t* status, void* stream) {
    if (n == 0) return HZ_OK;
    if (!states || n < 0) return HZ_ERR_ARG;
    k_end_turn<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, draws, status);
    return hz_launched(1);
}

int hz_replenish_piles(void* states, int64_t n, void* stream) {
    if (n == 0) return HZ_OK;
    if (!states || n < 0) return HZ_ERR_ARG;
    k_replenish<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n);
    return hz_launched(1);
}

int hz_draw_tiles(void* states, int64_t n, int count, uint8_t* tiles, void* stream) {
    if (n == 0) return HZ_OK;
    if (!states || !tiles || n < 0 || count < 0 || count > 15) return HZ_ERR_ARG;
    k_draw_tiles<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, count, tiles);
    return hz_launched(1);
}

int hz_score(const void* states, int64_t n, int16_t* scores, int16_t* terms, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || (!scores && !terms) || n < 0) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_score<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, scores, terms);
    return hz_launched(1);
}

int hz_encode(const void* states, int64_t n, void* board, void* glob, int dtype, int layout, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || !board || !glob || n < 0) return HZ_ERR_ARG;
    if (dtype != HZ_DTYPE_F32 && dtype != HZ_DTYPE_BF16) return HZ_ERR_ARG;
    if (layout != HZ_LAYOUT_NCHW && layout != HZ_LAYOUT_NHWC) return HZ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    // work items of one warp each: whole groups of G records at an aligned board, then the remaining records
    int64_t G = dtype == HZ_DTYPE_F32 ? 2 : 4, n_groups = ((uintptr_t)board & 15) == 0 ? n / G : 0;
    int64_t blocks = (n - n_groups * (G - 1) + ENC_WARPS - 1) / ENC_WARPS;
    int grid = (int)(blocks < 148 * 6 ? blocks : 148 * 6);
    if (dtype == HZ_DTYPE_F32) {
        if (layout == HZ_LAYOUT_NCHW) k_encode<float, false><<<grid, ENC_WARPS * 32, 0, st>>>(states, n, (float*)board, (float*)glob);
        else k_encode<float, true><<<grid, ENC_WARPS * 32, 0, st>>>(states, n, (float*)board, (float*)glob);
    } else {
        if (layout == HZ_LAYOUT_NCHW) k_encode<__nv_bfloat16, false><<<grid, ENC_WARPS * 32, 0, st>>>(states, n, (__nv_bfloat16*)board, (__nv_bfloat16*)glob);
        else k_encode<__nv_bfloat16, true><<<grid, ENC_WARPS * 32, 0, st>>>(states, n, (__nv_bfloat16*)board, (__nv_bfloat16*)glob);
    }
    return hz_launched(1);
}

int hz_canon_hash(const void* states, int64_t n, int key_mode, uint64_t* hashes, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || !hashes || n < 0 || (key_mode != HZ_KEY_EXACT && key_mode != HZ_KEY_REFERENCE)) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_hash<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, key_mode, hashes);
    return hz_launched(1);
}

int hz_outcome(const void* states, int64_t n, uint8_t* over, int8_t* outcome, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || (!over && !outcome) || n < 0) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_outcome<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, over, outcome);
    return hz_launched(1);
}

int hz_random_actions(const void* states, int64_t n, int16_t* actions, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || !actions || n < 0) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_random_actions<<<blocks_for(n, TPB), TPB, 0, (cudaStream_t)stream>>>(states, n, actions);
    return hz_launched(1);
}

int hz_greedy_actions(const void* states, int64_t n, int16_t* actions, void* stream) {
    if (n == 0) return HZ_OK;
    if (!states || !actions || n < 0) return HZ_ERR_ARG;
    k_greedy<<<blocks_for(n, GWPB), GWPB * 32, 0, (cudaStream_t)stream>>>(states, n, actions);
    return hz_launched(1);
}

int hz_playout(void* states, int64_t n, int max_steps, uint32_t* steps, unsigned long long* total_steps, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!states || n < 0 || max_steps < 0) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    k_playout<false><<<blocks_for(n, PTPB), PTPB, 0, (cudaStream_t)stream>>>(states, n, max_steps, steps, total_steps,
                                                                             nullptr, 0, 0, nullptr);
    return hz_launched(1);
}

int hz_playout_keys(const uint64_t* keys, int64_t n, uint64_t seed, uint64_t first_id, int max_steps,
                    uint32_t* results, unsigned long long* total_steps, void* stream) {
    if (n == 0) return HZ_OK;   // empty batch: nothing to do, pointers may be null
    if (!results || n < 0 || max_steps < 0) return HZ_ERR_ARG;
    k_playout<true><<<blocks_for(n, PTPB), PTPB, 0, (cudaStream_t)stream>>>(nullptr, n, max_steps, nullptr, total_steps,
                                                                            keys, seed, first_id, results);
    return hz_launched(1);
}

#ifdef HZ_PLAYOUT_TIMELINE
// Profiling builds only, not part of the ABI: the following k_playout launches write their phase timeline to buf
// (TL_WORDS uint64 per warp, in warp order; warps past n_warps record nothing).  buf = NULL turns it off.
int hz_playout_set_timeline(unsigned long long* buf, long long n_warps) {
    cudaError_t e = cudaMemcpyToSymbol(g_tl, &buf, sizeof buf);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_tl_warps, &n_warps, sizeof n_warps);
    return hz_record_launch(0, e);
}
#endif

}  // extern "C"
