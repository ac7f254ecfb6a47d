/*
 * harmonies_b200.h — C ABI of the B200-native batched Harmonies engine + MCTS core.
 *
 * This is the drop-in boundary for the hot path of IllyaArtemchuk/Harmonies-Alphazero
 * (reference files cited as file:line, relative to the reference root).  The reference
 * has no FFI: its boundary is the Python object API of `harmonies_engine.py`,
 * `process_game_state.py` and `MCTS.py`.  Each entry point below names the reference
 * function it replaces; `INTEGRATION.md` shows the ctypes stub a maintainer adds.
 *
 * Conventions
 *  - every function is `extern "C"`, returns an `int` status (HZ_OK == 0, negative = error),
 *    never throws, never synchronises the device unless stated;
 *  - all data pointers are DEVICE pointers owned by the caller unless the name ends in
 *    `_host`; `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream);
 *  - work is stream-ordered; one host thread per handle.
 *
 * ---------------------------------------------------------------------------------------
 * Packed game state: 128 bytes = 32 little-endian uint32 words, array-of-records.
 * (reference state fields: harmonies_engine.py:70-78)
 *
 *  hex index i (0..22)  = position of (q,r) in sorted(VALID_HEXES)   (constants.py:47-49)
 *  tile type t (0..5)   = index in TILE_TYPES: water,plant,wood,stone,building,field
 *                                                                     (constants.py:1)
 *  tile code            = t+1 (1..6), 0 = no tile at that level
 *
 *  w[ 0.. 8]  board of player 0 as 9 bit-planes: w[level*3 + b] has bit i set iff bit b of
 *             the tile code at stack level `level` (0 = bottom) of hex i is set
 *  w[ 9..17]  board of player 1, same layout
 *  w[18]      pile 0 (bits 0-15) | pile 1 (bits 16-31)
 *  w[19]      pile 2 | pile 3
 *  w[20]      pile 4 | hand (bits 16-31)
 *             a pile / the hand is a multiset of <=3 tiles: 6 x 2-bit counts, type t at
 *             bits 2t..2t+1 (the reference compares piles and hands as sorted tuples,
 *             harmonies_engine.py:98-100, so the multiset is the canonical form)
 *  w[21]      bag counts: water | plant<<8 | wood<<16 | stone<<24
 *  w[22]      bag building | bag field<<8 | n_piles<<16 | meta<<24
 *             meta: bit0 current_player; bits1-3 phase (0 choose_pile, 1..3 place_tile_k,
 *             4 game_over); bit4 the `game_over` attribute ("ending" flag,
 *             harmonies_engine.py:312-315); bits5-6 winner (0 None, 1 player 0,
 *             2 player 1, 3 tie == reference winner -1)
 *  w[23]      final_scores[0] (int16, bits 0-15) | final_scores[1] (bits 16-31)
 *  w[24..25]  rng key (uint64, lo/hi) of this game's draw stream
 *  w[26]      draw-event counter of the stream (one event per call that replenishes piles)
 *  w[27]      number of actions applied so far (game_move_count, trainer.py:466,509)
 *  w[28..31]  reserved, zero
 *
 *  What the kernels assume of a record (packed.pack_fields produces nothing else):
 *   - stacks without gaps: level l+1 of a hex holds a tile only where level l does.  Every
 *     kernel that reads a board assumes it (the stacking masks, place_random's counts); a
 *     gapped record is outside the format, not a supported input.  pack_fields builds the
 *     planes from stack lists, so it cannot produce one.
 *   - piles and hand: 2-bit counts (at most 3 tiles of a type).  The engine kernels take any
 *     such code; pack_fields also caps a pile and the hand at 3 tiles in all.
 *   - bag: any count 0..255 per type (pack_fields accepts exactly that range).  Every draw
 *     (hz_apply, hz_end_turn, hz_replenish_piles, hz_draw_tiles, in-tree expansion, the fused
 *     playouts) follows the rule below for any such bag; a game's bag never holds more than
 *     120 tiles, and the fused playout's whole-round path takes bags of 6..127 tiles only.
 *   - counters: w[26] and w[27] may take any uint32 value and wrap modulo 2^32.
 *
 *  Canonical identity (get_canonical_tuple, harmonies_engine.py:81-110) = words 0..22 with
 *  the ending flag and winner bits masked out (meta & 0x0F).
 *
 * Actions are the reference's flat action indices (process_game_state.py:156-177):
 *  a < 5: take pile a;  a >= 5: t=(a-5)/23, hex=(a-5)%23.   143 actions.
 *
 * Deterministic draw source (replaces the global `random` of harmonies_engine.py:126):
 *  mix(z): z=(z^(z>>30))*0xBF58476D1CE4E5B9; z=(z^(z>>27))*0x94D049BB133111EB; z^=z>>31
 *  rand(key,ctr) = mix(key ^ mix(ctr + 0x9E3779B97F4A7C15))
 *  pile k (k-th pile drawn inside one replenish) of draw event e of stream `key` uses
 *  z = rand(key, e*8 + k); tile j (j<min(3,total)) : x=(z>>(21*j))&0x1FFFFF;
 *  r=(x*total)>>21; the tile is the type whose cumulative bag count (TILE_TYPES order)
 *  first exceeds r; counts are decremented between tiles (sampling without replacement
 *  from the multiset, as random.sample over the flattened bag does).
 */
#ifndef HARMONIES_B200_H
#define HARMONIES_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HZ_ABI_VERSION      6
#define HZ_STATE_WORDS      32
#define HZ_STATE_BYTES      128
#define HZ_NUM_HEXES        23
#define HZ_NUM_TYPES        6
#define HZ_NUM_PILES        5
#define HZ_ACTION_SIZE      143
#define HZ_MASK_WORDS       5
#define HZ_BOARD_CHANNELS   38
#define HZ_BOARD_H          5
#define HZ_BOARD_W          7
#define HZ_GLOBAL_FEATURES  42
#define HZ_CANON_WORDS      23

/* word indices of the packed state */
#define HZ_W_BOARD0   0
#define HZ_W_BOARD1   9
#define HZ_W_PILES01  18
#define HZ_W_PILES23  19
#define HZ_W_PILE4H   20
#define HZ_W_BAG0     21
#define HZ_W_BAG1META 22
#define HZ_W_SCORES   23
#define HZ_W_KEYLO    24
#define HZ_W_KEYHI    25
#define HZ_W_EVENT    26
#define HZ_W_MOVES    27

/* phases */
#define HZ_PHASE_CHOOSE 0
#define HZ_PHASE_PLACE1 1
#define HZ_PHASE_PLACE2 2
#define HZ_PHASE_PLACE3 3
#define HZ_PHASE_OVER   4

/* call status */
#define HZ_OK               0
#define HZ_ERR_ARG         -1   /* null pointer / bad size */
#define HZ_ERR_CUDA        -2   /* a CUDA runtime call failed; see hz_last_cuda_error() */
#define HZ_ERR_NO_DEVICE   -3
#define HZ_ERR_WORKSPACE   -4   /* workspace too small / misaligned */

/* per-game status bytes written by hz_apply; each mirrors one ValueError site of
 * HarmoniesGameState.apply_move.  A game with status != 0 is left untouched. */
#define HZ_MOVE_OK            0
#define HZ_MOVE_BAD_PILE      1  /* harmonies_engine.py:220 */
#define HZ_MOVE_BAD_FORMAT    2  /* :234  (pile index given in a placement phase) */
#define HZ_MOVE_BAD_COORD     3  /* :242  (action index outside 0..142) */
#define HZ_MOVE_NOT_IN_HAND   4  /* :246 */
#define HZ_MOVE_ILLEGAL_STACK 5  /* :281 */
#define HZ_MOVE_BAD_PHASE     6  /* :296 */
#define HZ_MOVE_BAD_DRAW      7  /* explicit replay draw not available in the bag */

/* encode dtypes / layouts (HZ_DTYPE_I16 / HZ_DTYPE_I32: hz_sym_actions only) */
#define HZ_DTYPE_F32  0
#define HZ_DTYPE_BF16 1
#define HZ_DTYPE_I16  2
#define HZ_DTYPE_I32  3
#define HZ_LAYOUT_NCHW 0
#define HZ_LAYOUT_NHWC 1
#define HZ_LAYOUT_NHWC40 2  /* hz_tree_select only: [n,5,7,40], channels 38,39 = 0 (8-aligned C for the stem conv) */
#define HZ_LAYOUT_T16K   3  /* hz_tree_select only, bf16: the stem's tensor-core operand image of hz_tower_* ("T16K",
                             * 71,680 bytes per 16 leaves); bytes of channels 40..63 are not written: zero the buffer once */

/* node-key modes (hz_canon_hash, hz_tree_create):
 *  HZ_KEY_EXACT     identity = equality of get_canonical_tuple (harmonies_engine.py:81-118)
 *  HZ_KEY_REFERENCE identity = equality of Python's hash() of that tuple, which is what
 *                   MCTS.py keys nodes by (MCTS.py:14,177,185).  CPython has
 *                   hash(-1) == hash(-2), so board items at aliased coordinates
 *                   (q or r equal to -1 vs -2) are indistinguishable to the reference's tree;
 *                   this mode reproduces that relation exactly (needed for identical visit
 *                   counts).  Alias pairs of hex indices: {1,6},{2,7},{3,8},{4,5},{9,10},
 *                   {14,15},{19,20}; the key is the state with every board replaced by the
 *                   leftmost embedding of its sorted (alias class, stack) sequence. */
#define HZ_KEY_EXACT     0
#define HZ_KEY_REFERENCE 1

/* "no draw given" marker for hz_apply draws */
#define HZ_NO_DRAW 0xFFFFu

int         hz_abi_version(void);
const char *hz_status_string(int status);
const char *hz_last_cuda_error(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
uint64_t    hz_launch_count(void);

/* ---- engine (harmonies_engine.py) ------------------------------------------------ */

/* New games: HarmoniesGameState.__init__ (harmonies_engine.py:66-79) incl. the initial
 * _replenish_piles (:132-137) as draw event 0.  keys==NULL -> key_i = rand(seed, first_id+i). */
int hz_init_states(void *states, int64_t n, const uint64_t *keys, uint64_t seed,
                   uint64_t first_id, void *stream);

/* get_legal_moves (harmonies_engine.py:145-208) as a 143-bit mask per game, bit a of
 * mask[g*5 + a/32] set iff action a is legal.  Ascending bit order is the canonical
 * move order of this library. */
int hz_legal_mask(const void *states, int64_t n, uint32_t *mask, void *stream);

/* apply_move + _end_turn_actions + _replenish_piles + _draw_tiles + final scoring
 * (harmonies_engine.py:210-329,120-137,344-354), in place.  draws may be NULL; else
 * draws[g] != HZ_NO_DRAW is the pile (packed counts) to use for the first pile drawn by
 * this call instead of the state's rng stream (trace replay).  status may be NULL. */
int hz_apply(void *states, int64_t n, const int16_t *actions, const uint16_t *draws,
             uint8_t *status, void *stream);

/* calculate_score_for_player for both players (harmonies_engine.py:357-523):
 * scores[g*2+p].  terms (nullable): [g][p][5] = grass, mountains, fields, buildings, water. */
int hz_score(const void *states, int64_t n, int16_t *scores, int16_t *terms, void *stream);

/* create_state_tensors (process_game_state.py:15-137): board [n,38,5,7] (NCHW) or
 * [n,5,7,38] (NHWC) and glob [n,42], fp32 (bit-exact) or bf16 (RNE of the fp32 value). */
int hz_encode(const void *states, int64_t n, void *board, void *glob, int dtype, int layout,
              void *stream);

/* The reference's private turn helpers, for callers that drive them directly (its GUI calls
 * _end_turn_actions itself, GUI/main.py:364-365; harnesses patch _draw_tiles):
 * hz_end_turn       = _end_turn_actions (harmonies_engine.py:301-329) for the player to move:
 *                     replenish, end-of-game triggers, turn switch or final scoring; draws/status
 *                     as for hz_apply (HZ_MOVE_OK or HZ_MOVE_BAD_DRAW).
 * hz_replenish_piles = _replenish_piles (:132-137): top the piles up to five from the bag.
 * hz_draw_tiles     = _draw_tiles(count) (:120-130), count <= 15: tiles [n,16] uint8 = tile types
 *                     in draw order, byte 15 = number drawn; the bag is decremented.
 * Each call consumes one draw event of the state's stream. */
int hz_end_turn(void *states, int64_t n, const uint16_t *draws, uint8_t *status, void *stream);
int hz_replenish_piles(void *states, int64_t n, void *stream);
int hz_draw_tiles(void *states, int64_t n, int count, uint8_t *tiles, void *stream);

/* 64-bit key of get_canonical_tuple / __hash__ (harmonies_engine.py:81-113). */
int hz_canon_hash(const void *states, int64_t n, int key_mode, uint64_t *hashes, void *stream);

/* is_game_over / get_game_outcome (harmonies_engine.py:332-342): over[g] in {0,1},
 * outcome[g] in {+1,-1,0} from player 0's view (0 also when not over). Either may be NULL. */
int hz_outcome(const void *states, int64_t n, uint8_t *over, int8_t *outcome, void *stream);

/* The uniform-random playout policy of BASELINE.json configs[0..1]
 * (`random.choice(get_legal_moves())`): action = k-th legal action in ascending order,
 * k = ((rand(key ^ HZ_PLAYOUT_SALT, moves) >> 32) * n_legal) >> 32.  -1 if none. */
int hz_random_actions(const void *states, int64_t n, int16_t *actions, void *stream);

/* The 1-ply greedy agent of evaluation.py:137-196 (choose_move_greedy): the legal action whose
 * successor has the highest score for the mover, first strict maximum in ascending action
 * order; -1 if there is no legal action. */
int hz_greedy_actions(const void *states, int64_t n, int16_t *actions, void *stream);

/* Fused playout: repeat {legal -> random action -> apply} on-chip until the game is over
 * or max_steps actions were applied.  steps (nullable): actions applied per game.
 * total_steps (nullable): device uint64 to which the launch adds its step total. */
int hz_playout(void *states, int64_t n, int max_steps, uint32_t *steps,
               unsigned long long *total_steps, void *stream);

/* hz_init_states + hz_playout + result extraction in one launch, for callers that only want
 * the outcome of fresh games (the reference's `HarmoniesGameState()` followed by a random
 * playout loop, evaluation.py / tests): games are created on-chip from keys[i] (or from
 * rand(seed, first_id + i) when keys is NULL), played to the end, and only
 * results[i*3 + {0,1,2}] = {word HZ_W_BAG1META (phase, winner code), word HZ_W_SCORES,
 * word HZ_W_MOVES (actions played)} is written: 8 bytes in, 12 bytes out per game. */
int hz_playout_keys(const uint64_t *keys, int64_t n, uint64_t seed, uint64_t first_id,
                    int max_steps, uint32_t *results, unsigned long long *total_steps,
                    void *stream);

/* ---- game symmetries --------------------------------------------------------------------
 * The 23-hex board has exactly four automorphisms of its neighbour graph, all maps of the hex
 * lattice (axial coordinates): b = 0 identity, b = 1 (q,r) -> (q+r,-r), b = 2 (q,r) -> (-q-r,r),
 * b = 3 (q,r) -> (-q,-r) (hex i -> 22-i).  They form a Klein four-group (b1 o b2 = b1 ^ b2).  The
 * order of the piles carries no information either (pop(i) shifts the later piles, new ones are
 * appended).  Every rule (legality, the five scoring terms, the end-of-game trigger) reads only
 * stacks and adjacency, so a position and its image have the same value and the same legal moves
 * up to the action permutation below.
 *  element g (0..479, uint16): board part b = g & 3, pile part c = g >> 2 (0..119).
 *  T_g(state): the content of hex i moves to hex tau_b(i) in all 18 plane words; with m = n_piles,
 *           pi = itertools.permutations(range(m))[c mod m!], the pile at position i < m moves to
 *           position pi[i] (positions >= m stay put).  Hand, bag, meta, scores, rng key and the
 *           counters are unchanged.  m! divides 120, so a uniform g gives a uniform permutation.
 *  sigma_g(a): pi[a] for a < m; a for m <= a < 5; 5 + 23t + tau_b(h) for a = 5 + 23t + h.
 *           A policy, visit or mask row x transforms as x'[sigma_g(a)] = x[a].
 * The tables (tau_b, its inverse, the permutations) are generated from constants.py's geometry by
 * gen_tables.py into csrc/hz_tables.inc; harmonies_alphazero_b200/symmetry.py mirrors them. */
#define HZ_SYM_OFF   0   /* no symmetry (the default of a tree: reference-exact) */
#define HZ_SYM_BOARD 1   /* the 4 board symmetries (pile part 0) */
#define HZ_SYM_FULL  2   /* board x pile order: 480 elements */
#define HZ_SYMMETRY_SALT 0x53594D4D45545259ull   /* leaf frames of the search, see hz_tree_set_symmetry */

/* out[i] = T_{sym[i]}(states[i]).  out == states works (in place); other overlap does not.
 * Words 28..31 are copied unchanged. */
int hz_sym_states(const void *states, int64_t n, const uint16_t *sym, void *out, void *stream);

/* Rows x [n,143] of dtype HZ_DTYPE_F32, HZ_DTYPE_I16 or HZ_DTYPE_I32: out[i][sigma(a)] = x[i][a] with
 * sigma = sigma_{sym[i]} (inverse == 0) or sigma_{sym[i]}^-1 (inverse != 0).  n_piles is read from
 * states[i] (it is the same in either frame).  out must not overlap x. */
int hz_sym_actions(const void *x, int64_t n, int dtype, const uint16_t *sym, const void *states,
                   int inverse, void *out, void *stream);

/* ---- search tree (MCTS.py) ---------------------------------------------------------- */

typedef struct hz_tree hz_tree;   /* opaque: n_trees independent DAGs in flat arrays */

/* Bytes of device workspace for n_trees searches of at most max_sims simulations.
 * max_nodes == 0 selects the worst case (1 + 69*max_sims nodes per tree).
 * leaves = simulations in flight per tree and step: 1 is the reference's strictly sequential
 * search (MCTS.py:291-352, the parity mode); K > 1 is the virtual-loss throughput mode: every
 * hz_tree_select call descends K times per tree (edges on already chosen paths count one
 * provisional visit and one provisional loss: N' = N + V, W' = W - V), the evaluator sees
 * n_trees*K leaves (row t*K + j) and hz_tree_expand_backup lands them in order j = 0..K-1. */
size_t hz_tree_workspace_bytes(int n_trees, int max_sims, int max_nodes, int leaves);

/* Node/MCTS construction (MCTS.py:8-61) over caller-owned, 256-byte-aligned workspace. */
int hz_tree_create(hz_tree **out, void *workspace, size_t workspace_bytes, int n_trees,
                   int max_sims, int max_nodes, int key_mode, int leaves);
int hz_tree_destroy(hz_tree *t);

/* Start a new search per tree (get_best_action_and_pi, MCTS.py:288-289: no tree reuse).
 * root_states: [n_trees] packed states; search_keys: [n_trees] uint64, the key of the
 * in-tree draw stream: child of action a expanded in simulation s (0-based) draws event
 * (s<<8)|a.  search_keys == NULL -> key = rand(state key ^ HZ_SEARCH_SALT, state moves), a
 * stream per (game, move) that is independent of the game's own draws (the reference
 * re-draws the real move independently of the tree's sample, trainer.py:502). */
int hz_tree_reset(hz_tree *t, const void *root_states, const uint64_t *search_keys,
                  void *stream);

/* Active prefix (whole-game drivers whose games end at different times): n_active is a DEVICE
 * int32 (or NULL = all trees) read by every following hz_tree_reset / hz_tree_select /
 * hz_tree_fake_eval / hz_tree_expand_backup launch: only trees 0..*n_active-1 take part, the
 * others are skipped (their node and edge arrays keep the last search; hz_tree_reset still clears
 * every tree's hash index).  The word may change between launches (also between
 * replays of a captured CUDA graph); with the *_active network entry points below the evaluation
 * of a step then costs only the live rows.  The reference has no counterpart (one process per
 * game, trainer.py:104-107). */
int hz_tree_set_active(hz_tree *t, const int32_t *n_active);

/* Random-frame leaf evaluation (AlphaGo Zero's random rotation of the network's view): mode
 * HZ_SYM_OFF (the default, reference-exact), HZ_SYM_BOARD (G = 4) or HZ_SYM_FULL (G = 480).  With a
 * mode on, leaf row r of every following step gets one frame
 *   z = rand(sk ^ HZ_SYMMETRY_SALT, canon_hash(leaf, HZ_KEY_EXACT)),  g_r = ((z >> 32) * G) >> 32
 * (leaf = the node's stored words, sk = the tree's search key): it depends on the leaf and the search
 * key only, so two virtual-loss rows that reach one leaf share it.  The tree itself never changes frame:
 *  - hz_tree_select writes (board, glob) of T_{g_r}(leaf) in every layout; leaf_states stay untransformed;
 *  - hz_tree_expand_backup takes policy[r][sigma_{g_r}(a)] as the prior of action a (the fused softmax,
 *    its sums and the root Dirichlet mix run in the tree's order, as with the mode off);
 *  - hz_tree_fake_eval and hz_tree_rollout_eval write their result into the frame (entry sigma_{g_r}(a)
 *    gets what entry a gets with the mode off; values unchanged), so a search with them is the same
 *    with the mode on or off.
 * A leaf's frame is kept in the tree's node record for the rest of the search.  The mode acts on the
 * launches that follow the call; a captured CUDA graph keeps the mode it was captured with.  Set the
 * mode before hz_tree_reset: one search runs in one mode (switching it on after steps with the mode off
 * is fine; switching between HZ_SYM_BOARD and HZ_SYM_FULL inside a search is not). */
int hz_tree_set_symmetry(hz_tree *t, int mode);

/* frames[n_trees * leaves] (uint16): g_r of every leaf row of the last hz_tree_select (0 for all rows
 * when that select ran with the mode off).  Rows of trees beyond the active prefix keep the frames of
 * the last select that included them. */
int hz_tree_leaf_frames(hz_tree *t, uint16_t *frames, void *stream);

/* move_to_leaf (MCTS.py:63-149) for every tree, then create_state_tensors of the leaf
 * (MCTS.py:299) into board/glob (see hz_encode).  cpuct is applied as fp32(cpuct)*P in fp32
 * then promoted to fp64, the reference's numpy>=2 arithmetic (MCTS.py:107-112).
 * leaf_states (nullable): [n_trees] packed leaf states. */
int hz_tree_select(hz_tree *t, float cpuct, void *leaf_states, void *board, void *glob,
                   int dtype, int layout, void *stream);

/* expand_leaf + terminal value + back_fill (MCTS.py:151-264,297-352).  policy: [n,143]
 * softmax probabilities (or logits when is_logits != 0; softmax is then fused), value: [n].
 * noise (nullable): [n,143] unnormalised gamma samples indexed by action; at the root
 * expansion they are normalised over the legal moves and mixed with weight eps
 * (MCTS.py:308-326).  Advances each tree's simulation counter. */
int hz_tree_expand_backup(hz_tree *t, const float *policy, const float *value,
                          int is_logits, const float *noise, double eps, void *stream);

/* Synthetic evaluator for tests/benches: exact dyadic priors/values from the leaf's
 * canonical hash: P[a] = (mix(h ^ (a+1)) >> 40) * 2^-24, v = (mix(h ^ 0x5EED) >> 40) *
 * 2^-23 - 1.  Stands in for ModelManager.predict (model.py:81-110). */
int hz_tree_fake_eval(hz_tree *t, float *policy, float *value, void *stream);

/* Rollout evaluator: for every leaf row of the last hz_tree_select (rows of active trees only),
 * R = rollouts random playouts from the leaf, R in {1,2,4,8,16,32,64} (else HZ_ERR_ARG).  A
 * network-free evaluator with the same output contract as hz_tree_fake_eval.
 *  keys:     leaf = the node's stored 32 words, sk = the tree's search key (hz_tree_reset);
 *            base = rand(sk ^ HZ_ROLLOUT_SALT, canon_hash(leaf, HZ_KEY_EXACT)),
 *            key_r = rand(base, r) for r = 0..R-1.  Rollout r is a copy of leaf with words
 *            HZ_W_KEYLO/HI replaced by key_r (nothing else changes), played with hz_playout's
 *            semantics (random policy, draws, round path) for at most 1,000 actions.  The keys
 *            depend on the leaf and the search key only: a leaf that two virtual-loss rows reach
 *            in one step gets the same value.
 *  value:    value[row] = (float)(sigma * sum_r o_r) / (float)R, o_r in {+1,-1,0} = hz_outcome
 *            (player 0's view) of rollout r's final state (0 if it is not over: stuck or capped),
 *            sigma = +1 if the leaf's player to move is 0, else -1.  Exact (R is a power of two).
 *  policy:   policy[row][a] = 1.0f / (float)n_legal for legal a, 0 otherwise: probabilities
 *            (pass is_logits = 0 to hz_tree_expand_backup).
 *  A leaf that is over gets no rollouts, value 0 and a zero policy row (hz_tree_expand_backup
 *  uses its outcome).  A leaf with no legal move gets a zero policy row and value 0.
 *  total_steps (nullable): device uint64 to which the launch adds the rollout actions played.
 *  Rows of trees beyond the active prefix (hz_tree_set_active) are not written. */
int hz_tree_rollout_eval(hz_tree *t, int rollouts, float *policy, float *value,
                         unsigned long long *total_steps, void *stream);

/* Root visit counts and pi = N / sum N (MCTS.py:355-381): visits [n,143] int32,
 * pi [n,143] fp32 (either nullable). */
int hz_tree_root_policy(hz_tree *t, int32_t *visits, float *pi, void *stream);

/* Move choice (MCTS.py:394-441): u01 == NULL or exploratory[g]==0 -> first max-N edge in
 * ascending action order; else the edge where the running sum of N first exceeds
 * u01[g]*sum N.  action -1 = no edge (search failure, MCTS.py:439). */
int hz_tree_choose(hz_tree *t, const float *u01, const uint8_t *exploratory,
                   int16_t *actions, void *stream);

/* Per-tree counters: n_nodes, n_edges (int32 each, nullable) and status bytes (nullable):
 * bits 0-3 = the current search: 1 node arena overflow, 2 edge arena overflow, 4 path overflow;
 * bits 4-7 = the same flags raised by any EARLIER search of this handle (hz_tree_reset moves
 * them up instead of clearing them, so a truncated search can never go unnoticed). */
int hz_tree_stats(hz_tree *t, int32_t *n_nodes, int32_t *n_edges, uint8_t *status,
                  void *stream);

/* Root edge statistics for parity checks: N int32, W fp64, P fp32, child node id int32,
 * all [n,143] indexed by action (absent edges: N=0,W=0,P=0,child=-1). Any may be NULL. */
int hz_tree_root_edges(hz_tree *t, int32_t *N, double *W, float *P, int32_t *child,
                       void *stream);

/* ---- network tail (model.py) ----------------------------------------------------------- */

/* Fused policy/value heads of AlphaZeroModel.forward (model.py:340-355) on the residual
 * tower's output: x [n,35,C] bf16 NHWC, glob [n,42] bf16 -> logits [n,143] fp32, value [n] fp32.
 * Weights fp32 with BatchNorm folded: w_conv [3][C] (policy ch0, policy ch1, value ch0),
 * b_conv [3], w_pol_t [112][143] (policy_fc weight transposed), b_pol [143], w_v1_t [77][H]
 * (value_fc1 transposed), b_v1 [H], w_v2 [H], b_v2.  C multiple of 8, x 16-byte aligned. */
int hz_net_heads(const void *x, const void *glob, int64_t n, int C, int H, const float *w_conv,
                 const float *b_conv, const float *w_pol_t, const float *b_pol,
                 const float *w_v1_t, const float *b_v1, const float *w_v2, float b_v2,
                 float *logits, float *value, void *stream);

/* The FC layers of the same heads (model.py:344-355; the default network's shape only: H = 256)
 * when the 1x1 head convolutions + BatchNorm + ReLU are already evaluated by the head item of
 * hz_tower_forward_heads: head_conv in the layout it writes, [tile of 16 boards][filter * 35 +
 * cell][board in tile] fp32 (filters policy 0, policy 1, value).  Rows min(n, *n_active) are
 * evaluated (n_active: a DEVICE int32, NULL = n; see hz_tree_set_active). */
int hz_net_heads_fc_active(const float *head_conv, const void *glob, int64_t n,
                           const int32_t *n_active, int H, const float *w_pol_t, const float *b_pol,
                           const float *w_v1_t, const float *b_v1, const float *w_v2, float b_v2,
                           float *logits, float *value, void *stream);

/* ---- residual tower (model.py:325-339, ResidualBlock.forward model.py:380-392) -----------
 * Hand-written sm_100a 3x3 convolution (tcgen05.mma, accumulators in tensor memory, operands
 * brought in by the bulk copy engine), BatchNorm folded, bf16 in / fp32 accumulate / bf16 out.
 *
 * Activations are kept in 16-board tiles that are byte-for-byte the shared-memory image of the
 * tensor-core operand (a tile half = 71,680 bytes = one bulk copy).  Position p = cell*16 + board
 * (cell = y*7 + x of the 5x7 plane, board = index inside the tile).
 *   "T16"  (outputs, residual-block inputs; 128 channels = 143,360 bytes per tile): MN-major, no
 *          swizzle: element (p, c) at  (c/8)*8960 + (p/8)*128 + (c%8)*16 + (p%8)*2.
 *   "T16K" (the stem's input; <= 64 channels, one half per tile): K-major SWIZZLE_128B: element
 *          (p, c) at  p*128 + (((c/8) ^ (p%8)) * 16) + (c%8)*2.
 * Weights: [tap = ky*3+kx][channel half][out channel 0..127] rows of 128 bytes, K-major
 * SWIZZLE_128B (input-channel group g of the half at g ^ (out & 7)): 16 KB per (tap, half). */
size_t hz_tower_tile_bytes(int64_t n_boards, int channel_halves);
/* Upper bound on the persistent grid of hz_tower_conv3x3 (0 = one CTA per SM, the default).
 * Process-wide; meant for tests that push many tiles through few CTAs. */
int hz_tower_set_max_ctas(int max_ctas);
/* Profiling switches of hz_tower_conv3x3 (0 = normal operation; results are WRONG otherwise):
 * 1 skip the MMAs, 2 skip the epilogue's memory traffic, 4 skip the weight copies, 8 skip the
 * activation copies.
 * Used by profiles/tower_bench.py to attribute the kernel's time. */
int hz_tower_set_debug(int flags);
/* Profiling: a device buffer of 4096 uint64 (or NULL to switch off) into which CTA 0 of every
 * following hz_tower_conv3x3 launch writes SM-clock timestamps of its producer / MMA / epilogue
 * roles (slot map in csrc/hz_tower.cu).  The time stamps are compiled in only with
 * -DHZ_TOWER_TRACE=1 (they cost instruction-cache space); otherwise a non-NULL buffer is refused
 * with HZ_ERR_ARG. */
int hz_tower_set_trace(unsigned long long *device_buffer_4096);

/* NHWC bf16 [n,35,channels] -> tiles.  kmajor != 0: T16K (channels % 8 == 0, <= 64; missing
 * channels zero); kmajor == 0: T16 (channels must be 128).  Boards that pad n up to a multiple
 * of 16 are written as zero. */
int hz_tower_to_tiles(const void *src_nhwc, void *dst_tiles, int64_t n_boards, int channels,
                      int kmajor, void *stream);
/* T16 tiles -> NHWC bf16 [n,35,128] (the layout hz_net_heads reads) */
int hz_tower_from_tiles(const void *src_tiles, void *dst_nhwc, int64_t n_boards, void *stream);

/* y = [relu]( conv3x3(x, w) + bias [+ residual] ) for n_boards (multiple of 16) boards.
 * x: in_kmajor != 0: T16K tiles, in_channel_halves must be 1 (the stem: 38 input planes
 * zero-padded to 64); in_kmajor == 0: T16 tiles with in_channel_halves * 64 channels.
 * residual (nullable) and y: T16 tiles, 128 channels.  fault (nullable): a host-mapped word that
 * receives the id of a barrier wait that timed out before the kernel traps. */
int hz_tower_conv3x3(const void *x_tiles, int in_channel_halves, int in_kmajor, const void *w_tiles,
                     const float *bias, const void *residual_tiles, void *y, int64_t n_boards,
                     int relu, unsigned int *fault, void *stream);
/* The whole body in ONE persistent launch: stem (layer 0, input x0 = T16K tiles) followed by
 * n_blocks residual blocks (layers 1 + 2i: conv+bn+relu, 2 + 2i: conv+bn, + block input, relu).
 * w_tiles / biases: HOST arrays of 1 + 2*n_blocks DEVICE pointers (weight tiles as above, fp32
 * bias[128]).  buf_a/b/c: three T16 scratch buffers of hz_tower_tile_bytes(n_boards, 2) bytes;
 * *out_tiles receives the one that holds the result (buf_a or buf_c).  sched: device scratch of
 * hz_tower_sched_bytes() bytes (initialised by the call on `stream`).
 * Boards are independent, so work item (layer l, tile t) depends on (l-1, t) only: the CTAs take
 * the (1 + 2*n_blocks) * n_boards/16 items from a ready queue in `sched` that starts with the
 * stem items and to which the completion of (l, t) appends (l+1, t) — no grid-wide
 * synchronisation, no dependency stalls, and the load balances to within one item per CTA
 * whatever the tile count.
 * Only the tiles that hold boards 0..min(n_boards, *n_active)-1 are computed (n_active: a DEVICE
 * int32, NULL = all; see hz_tree_set_active).  The launch geometry and every address are those of
 * n_boards, so one captured CUDA graph serves every active count.
 * After the body, in the same launch, the 1x1 head convolutions + BatchNorm + ReLU
 * (model.py:340-343,349-351) run as one more work item per tile: a single-tap tcgen05.mma pass
 * over the tile the last block just wrote.  w_head_tiles: [2 channel halves][128 rows][128 B]
 * K-major SWIZZLE_128B bf16 with rows 0..2 = high parts of the three head filters (policy 0,
 * policy 1, value), rows 3..5 = low parts (filter = hi + lo: fp32-weight accuracy), other rows
 * zero; b_head [3] fp32; head_conv_tiled: [n_boards/16][3*35][16] fp32 (read it with
 * hz_net_heads_fc_active).  w_head_tiles == NULL: no head item. */
size_t hz_tower_sched_bytes(int64_t n_boards, int n_blocks);
int hz_tower_forward_heads(const void *x0_tiles, const void *const *w_tiles,
                           const float *const *biases, int n_blocks, void *buf_a, void *buf_b,
                           void *buf_c, void *sched, void **out_tiles, int64_t n_boards,
                           const int32_t *n_active, const void *w_head_tiles, const float *b_head,
                           float *head_conv_tiled, unsigned int *fault, void *stream);

#define HZ_PLAYOUT_SALT 0xA5A5F00DC0FFEE11ull
#define HZ_SEARCH_SALT  0x5EA2C47EE5A17B00ull
#define HZ_ROLLOUT_SALT 0x2011C0A75EED5A17ull

#ifdef __cplusplus
}
#endif
#endif /* HARMONIES_B200_H */
