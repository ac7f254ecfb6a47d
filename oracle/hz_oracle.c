/*
 * hz_oracle.c — TEST INFRASTRUCTURE.  CPU restatement of the reference's hot path
 * (IllyaArtemchuk/Harmonies-Alphazero: harmonies_engine.py, process_game_state.py, MCTS.py)
 * in plain C, written the straightforward way (per-hex stacks, lists, queue BFS) so that
 * it is an independent check on the bit-board CUDA kernels.
 *
 * PARITY PIN: this file is checked against tests/golden/*.npz, which were produced by
 * running the unmodified Python reference (oracle/gen_golden.py) — engine traces, legal
 * masks, per-term scores, state tensors, equivalence classes and full MCTS searches.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load this library.  The product path (harmonies_alphazero_b200/) never does.
 *
 * Each function names the reference lines it follows.  Data crosses the boundary in the
 * packed 128-byte format of include/harmonies_b200.h.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../include/harmonies_b200.h"

enum { WATER = 0, PLANT, WOOD, STONE, BUILDING, FIELD };
#define NO_WINNER (-2)

typedef struct {
    uint8_t height[2][23];
    uint8_t stack[2][23][3];
    int bag[6];
    int n_piles;
    int pile_len[5];
    uint8_t pile[5][3];
    int hand_len;
    uint8_t hand[3];
    int player, phase, ending, winner;
    int scores[2];
    uint64_t key;
    uint32_t event, moves;
} ostate;

/* ---- geometry: constants.py:4-49 ---------------------------------------------------- */
static int g_q[23], g_r[23], g_nn[23], g_nb[23][6], g_ready = 0;
static const int INIT_BAG[6] = {23, 19, 21, 23, 15, 19}; /* TILE_TYPES order, constants.py:41 */

static void geometry(void) {
    if (g_ready) return;
    static const int row_len[5] = {5, 4, 5, 4, 5}, row_q0[5] = {-1, -1, -2, -2, -3};
    int n = 0, qs[23], rs[23];
    for (int row = 0; row < 5; row++)
        for (int i = 0; i < row_len[row]; i++) { qs[n] = row_q0[row] + i; rs[n] = row - 2; n++; }
    /* sorted(list(VALID_HEXES)): lexicographic on (q, r)  (constants.py:47) */
    for (int i = 0; i < 23; i++) {
        int rank = 0;
        for (int j = 0; j < 23; j++)
            if (qs[j] < qs[i] || (qs[j] == qs[i] && rs[j] < rs[i])) rank++;
        g_q[rank] = qs[i]; g_r[rank] = rs[i];
    }
    static const int dq[6] = {1, -1, 0, 0, 1, -1}, dr[6] = {0, 0, 1, -1, -1, 1}; /* constants.py:35 */
    for (int i = 0; i < 23; i++) {
        g_nn[i] = 0;
        for (int d = 0; d < 6; d++)
            for (int j = 0; j < 23; j++)
                if (g_q[j] == g_q[i] + dq[d] && g_r[j] == g_r[i] + dr[d]) g_nb[i][g_nn[i]++] = j;
    }
    g_ready = 1;
}

/* ---- draw source (include/harmonies_b200.h) ----------------------------------------- */
static uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
static uint64_t rand64(uint64_t key, uint64_t ctr) { return mix64(key ^ mix64(ctr + 0x9E3779B97F4A7C15ull)); }

/* ---- packed <-> plain ---------------------------------------------------------------- */
static int unpack_multiset(uint32_t code, uint8_t *out) {
    int n = 0;
    for (int t = 0; t < 6; t++)
        for (uint32_t c = (code >> (2 * t)) & 3; c > 0 && n < 3; c--) out[n++] = (uint8_t)t;
    return n;
}
static uint32_t pack_multiset(const uint8_t *tiles, int n) {
    uint32_t code = 0;
    for (int i = 0; i < n; i++) code += 1u << (2 * tiles[i]);
    return code;
}

static void unpack(const uint32_t *w, ostate *s) {
    memset(s, 0, sizeof *s);
    for (int p = 0; p < 2; p++)
        for (int i = 0; i < 23; i++) {
            int h = 0;
            for (int l = 0; l < 3; l++) {
                int code = 0;
                for (int b = 0; b < 3; b++) code |= ((w[p * 9 + l * 3 + b] >> i) & 1) << b;
                if (!code) break;
                s->stack[p][i][h++] = (uint8_t)(code - 1);
            }
            s->height[p][i] = (uint8_t)h;
        }
    uint32_t codes[5] = {w[18] & 0xFFFF, w[18] >> 16, w[19] & 0xFFFF, w[19] >> 16, w[20] & 0xFFFF};
    s->n_piles = (w[22] >> 16) & 0xFF;
    for (int i = 0; i < s->n_piles && i < 5; i++) s->pile_len[i] = unpack_multiset(codes[i], s->pile[i]);
    s->hand_len = unpack_multiset(w[20] >> 16, s->hand);
    s->bag[0] = w[21] & 0xFF; s->bag[1] = (w[21] >> 8) & 0xFF; s->bag[2] = (w[21] >> 16) & 0xFF;
    s->bag[3] = w[21] >> 24;  s->bag[4] = w[22] & 0xFF;        s->bag[5] = (w[22] >> 8) & 0xFF;
    uint32_t meta = w[22] >> 24;
    s->player = meta & 1; s->phase = (meta >> 1) & 7; s->ending = (meta >> 4) & 1;
    int wc = (meta >> 5) & 3;
    s->winner = wc == 0 ? NO_WINNER : wc == 1 ? 0 : wc == 2 ? 1 : -1;
    s->scores[0] = (int16_t)(w[23] & 0xFFFF); s->scores[1] = (int16_t)(w[23] >> 16);
    s->key = (uint64_t)w[24] | ((uint64_t)w[25] << 32);
    s->event = w[26]; s->moves = w[27];
}

static void pack(const ostate *s, uint32_t *w) {
    memset(w, 0, 32 * sizeof(uint32_t));
    for (int p = 0; p < 2; p++)
        for (int i = 0; i < 23; i++)
            for (int l = 0; l < s->height[p][i]; l++) {
                int code = s->stack[p][i][l] + 1;
                for (int b = 0; b < 3; b++)
                    if ((code >> b) & 1) w[p * 9 + l * 3 + b] |= 1u << i;
            }
    uint32_t codes[5] = {0, 0, 0, 0, 0};
    for (int i = 0; i < s->n_piles; i++) codes[i] = pack_multiset(s->pile[i], s->pile_len[i]);
    w[18] = codes[0] | (codes[1] << 16);
    w[19] = codes[2] | (codes[3] << 16);
    w[20] = codes[4] | (pack_multiset(s->hand, s->hand_len) << 16);
    w[21] = (uint32_t)s->bag[0] | ((uint32_t)s->bag[1] << 8) | ((uint32_t)s->bag[2] << 16) | ((uint32_t)s->bag[3] << 24);
    int wc = s->winner == NO_WINNER ? 0 : s->winner == 0 ? 1 : s->winner == 1 ? 2 : 3;
    uint32_t meta = (uint32_t)s->player | ((uint32_t)s->phase << 1) | ((uint32_t)s->ending << 4) | ((uint32_t)wc << 5);
    w[22] = (uint32_t)s->bag[4] | ((uint32_t)s->bag[5] << 8) | ((uint32_t)s->n_piles << 16) | (meta << 24);
    w[23] = ((uint32_t)s->scores[0] & 0xFFFF) | (((uint32_t)s->scores[1] & 0xFFFF) << 16);
    w[24] = (uint32_t)s->key; w[25] = (uint32_t)(s->key >> 32);
    w[26] = s->event; w[27] = s->moves;
}

/* ---- _draw_tiles / _replenish_piles: harmonies_engine.py:120-137 --------------------- */
static int draw_tiles(ostate *s, uint64_t z, int num, uint8_t *out) {
    int n = 0;
    for (int j = 0; j < num; j++) {
        int total = 0;
        for (int t = 0; t < 6; t++) total += s->bag[t];
        if (total == 0) break;                                   /* :123-125 */
        uint64_t x = (z >> (21 * j)) & 0x1FFFFF;
        int r = (int)((x * (uint64_t)total) >> 21), t = 0;
        while (r >= s->bag[t]) { r -= s->bag[t]; t++; }
        s->bag[t]--;                                             /* :128-129 */
        out[n++] = (uint8_t)t;
    }
    return n;
}

/* explicit != HZ_NO_DRAW: first pile of this replenish is the given multiset (trace replay) */
static int replenish(ostate *s, uint32_t explicit_code) {
    int k = 0;
    while (s->n_piles < 5) {                                     /* :133 */
        uint8_t tiles[3];
        int n;
        if (k == 0 && explicit_code != HZ_NO_DRAW) {
            n = unpack_multiset(explicit_code, tiles);
            for (int i = 0; i < n; i++) {
                if (s->bag[tiles[i]] == 0) return -1;
                s->bag[tiles[i]]--;
            }
        } else {
            n = draw_tiles(s, rand64(s->key, (uint64_t)s->event * 8 + (uint64_t)k), 3, tiles);
        }
        if (n == 0) break;                                       /* :135-136 */
        memcpy(s->pile[s->n_piles], tiles, 3);
        s->pile_len[s->n_piles] = n;
        s->n_piles++;                                            /* :137 */
        k++;
    }
    s->event++;
    return 0;
}

/* ---- get_legal_moves: harmonies_engine.py:145-208 ------------------------------------ */
static int stack_ok(int tile, int top, int h) {                  /* :183-194 == :263-272 */
    if (tile == PLANT && top == WOOD && h <= 2) return 1;
    if (tile == STONE && top == STONE && h < 3) return 1;
    if (tile == BUILDING && (top == WOOD || top == STONE || top == BUILDING) && h < 2) return 1;
    return 0;
}

static int legal_actions(const ostate *s, int *out) {
    int n = 0;
    if (s->phase == HZ_PHASE_CHOOSE) {
        for (int i = 0; i < s->n_piles; i++) out[n++] = i;       /* :158 */
    } else if (s->phase >= HZ_PHASE_PLACE1 && s->phase <= HZ_PHASE_PLACE3) {
        int in_hand[6] = {0, 0, 0, 0, 0, 0};
        for (int i = 0; i < s->hand_len; i++) in_hand[s->hand[i]] = 1;   /* :167 */
        for (int t = 0; t < 6; t++) {
            if (!in_hand[t]) continue;
            for (int i = 0; i < 23; i++) {
                int h = s->height[s->player][i];
                if (h == 0 || stack_ok(t, s->stack[s->player][i][h - 1], h))
                    out[n++] = 5 + 23 * t + i;                   /* process_game_state.py:177 */
            }
        }
    }
    return n;                                                    /* else: :205-208 */
}

/* ---- scoring: harmonies_engine.py:357-523 -------------------------------------------- */
static int top_of(const ostate *s, int p, int i) { int h = s->height[p][i]; return h ? s->stack[p][i][h - 1] : -1; }

static int score_grass(const ostate *s, int p) {                 /* :369-385 */
    int sc = 0;
    for (int i = 0; i < 23; i++) {
        int h = s->height[p][i];
        if (!h || s->stack[p][i][h - 1] != PLANT) continue;
        if (h == 1) sc += 1;
        else if (h == 2 && s->stack[p][i][0] == WOOD) sc += 3;
        else if (h == 3 && s->stack[p][i][0] == WOOD && s->stack[p][i][1] == WOOD) sc += 7;
    }
    return sc;
}
static int score_mountains(const ostate *s, int p) {             /* :392-413 */
    int sc = 0;
    for (int i = 0; i < 23; i++) {
        if (top_of(s, p, i) != STONE) continue;
        int adj = 0;
        for (int k = 0; k < g_nn[i]; k++) adj |= top_of(s, p, g_nb[i][k]) == STONE;
        if (!adj) continue;
        int h = s->height[p][i];
        sc += h == 1 ? 1 : h == 2 ? 3 : 7;
    }
    return sc;
}
/* flood fill of the top-`type` component containing `start`; returns its size */
static int component(const ostate *s, int p, int type, int start, int *visited, int *comp) {
    int queue[23], qh = 0, qt = 0, n = 0;
    queue[qt++] = start; visited[start] = 1; comp[n++] = start;
    while (qh < qt) {
        int cur = queue[qh++];
        for (int k = 0; k < g_nn[cur]; k++) {
            int nb = g_nb[cur][k];
            if (!visited[nb] && top_of(s, p, nb) == type) { visited[nb] = 1; comp[n++] = nb; queue[qt++] = nb; }
        }
    }
    return n;
}
static int score_fields(const ostate *s, int p) {                /* :424-443 */
    int sc = 0, visited[23] = {0}, comp[23];
    for (int i = 0; i < 23; i++)
        if (top_of(s, p, i) == FIELD && !visited[i])
            if (component(s, p, FIELD, i, visited, comp) >= 2) sc += 5;
    return sc;
}
static int score_buildings(const ostate *s, int p) {             /* :454-469 */
    int sc = 0;
    for (int i = 0; i < 23; i++) {
        if (top_of(s, p, i) != BUILDING || s->height[p][i] != 2) continue;
        int seen[6] = {0}, kinds = 0;
        for (int k = 0; k < g_nn[i]; k++) {
            int t = top_of(s, p, g_nb[i][k]);
            if (t >= 0 && !seen[t]) { seen[t] = 1; kinds++; }
        }
        if (kinds >= 3) sc += 5;
    }
    return sc;
}
static int water_score(int len) {                                /* :18-27 */
    static const int tab[7] = {0, 0, 2, 5, 8, 11, 15};
    if (len <= 0) return 0;
    return len <= 6 ? tab[len] : 15 + (len - 6) * 4;
}
static int score_water(const ostate *s, int p) {                 /* :480-518 */
    int sc = 0, visited[23] = {0}, comp[23];
    for (int i = 0; i < 23; i++) {
        if (top_of(s, p, i) != WATER || visited[i]) continue;
        int n = component(s, p, WATER, i, visited, comp);
        if (n < 2) continue;
        int in_comp[23] = {0}, diameter = 0;
        for (int k = 0; k < n; k++) in_comp[comp[k]] = 1;
        for (int k = 0; k < n; k++) {                            /* BFS eccentricity, :505-517 */
            int dist[23], queue[23], qh = 0, qt = 0;
            for (int j = 0; j < 23; j++) dist[j] = -1;
            dist[comp[k]] = 0; queue[qt++] = comp[k];
            while (qh < qt) {
                int cur = queue[qh++];
                if (dist[cur] > diameter) diameter = dist[cur];
                for (int m = 0; m < g_nn[cur]; m++) {
                    int nb = g_nb[cur][m];
                    if (in_comp[nb] && dist[nb] < 0) { dist[nb] = dist[cur] + 1; queue[qt++] = nb; }
                }
            }
        }
        sc += water_score(diameter + 1);
    }
    return sc;
}
static void score_terms(const ostate *s, int p, int *t5) {
    t5[0] = score_grass(s, p); t5[1] = score_mountains(s, p); t5[2] = score_fields(s, p);
    t5[3] = score_buildings(s, p); t5[4] = score_water(s, p);
}
static int score_player(const ostate *s, int p) {                /* :357-367 */
    int t[5]; score_terms(s, p, t);
    return t[0] + t[1] + t[2] + t[3] + t[4];
}

/* ---- _end_turn_actions: harmonies_engine.py:301-329 ---------------------------------- */
static void finish_game(ostate *s) {
    s->phase = HZ_PHASE_OVER;
    s->scores[0] = score_player(s, 0); s->scores[1] = score_player(s, 1);       /* :344-346 */
    s->winner = s->scores[0] > s->scores[1] ? 0 : s->scores[1] > s->scores[0] ? 1 : -1; /* :348-354 */
}
static int end_turn(ostate *s, uint32_t explicit_code) {
    int finisher = s->player, occupied = 0, bag_total = 0;
    for (int i = 0; i < 23; i++) occupied += s->height[finisher][i] > 0;
    int player_trigger = (23 - occupied) <= 2;                   /* :304-305 */
    for (int t = 0; t < 6; t++) bag_total += s->bag[t];
    int bag_empty_before = bag_total == 0;                       /* :307 */
    if (replenish(s, explicit_code) < 0) return -1;
    int bag_trigger = bag_empty_before && s->n_piles == 0;       /* :309 */
    int triggered = player_trigger || bag_trigger, ending = s->ending;
    if (triggered && !ending) {
        s->ending = 1;
        if (finisher == 0) { s->player = 1; s->phase = HZ_PHASE_CHOOSE; }
        else finish_game(s);
    } else if (ending) {
        finish_game(s);
    } else {
        s->player = 1 - s->player; s->phase = HZ_PHASE_CHOOSE;
    }
    return 0;
}

/* ---- apply_move: harmonies_engine.py:210-298 ----------------------------------------- */
static int apply_action(ostate *s, int a, uint32_t explicit_code) {
    ostate n = *s;                                               /* clone(), :211 */
    if (n.phase == HZ_PHASE_CHOOSE) {
        if (a < 0 || a >= 5 || a >= n.n_piles) return HZ_MOVE_BAD_PILE;         /* :217-220 */
        n.hand_len = n.pile_len[a];
        memcpy(n.hand, n.pile[a], 3);
        for (int i = a; i + 1 < n.n_piles; i++) { memcpy(n.pile[i], n.pile[i + 1], 3); n.pile_len[i] = n.pile_len[i + 1]; }
        n.n_piles--;                                             /* pop, :221 */
        n.phase = HZ_PHASE_PLACE1;
    } else if (n.phase >= HZ_PHASE_PLACE1 && n.phase <= HZ_PHASE_PLACE3) {
        if (a < 5) return HZ_MOVE_BAD_FORMAT;                    /* :227-236 */
        if (a >= HZ_ACTION_SIZE) return HZ_MOVE_BAD_COORD;       /* :241-242 */
        int tile = (a - 5) / 23, hex = (a - 5) % 23, pos = -1, p = n.player;
        for (int i = 0; i < n.hand_len; i++) if (n.hand[i] == tile) { pos = i; break; }
        if (pos < 0) return HZ_MOVE_NOT_IN_HAND;                 /* :244-248 */
        for (int i = pos; i + 1 < n.hand_len; i++) n.hand[i] = n.hand[i + 1];   /* remove, :250 */
        n.hand_len--;
        int h = n.height[p][hex];
        if (h != 0 && !stack_ok(tile, n.stack[p][hex][h - 1], h)) return HZ_MOVE_ILLEGAL_STACK; /* :281 */
        n.stack[p][hex][h] = (uint8_t)tile; n.height[p][hex] = (uint8_t)(h + 1);
        if (n.phase == HZ_PHASE_PLACE3) { if (end_turn(&n, explicit_code) < 0) return HZ_MOVE_BAD_DRAW; }
        else n.phase++;                                          /* :287-292 */
    } else {
        return HZ_MOVE_BAD_PHASE;                                /* :296 */
    }
    n.moves++;
    *s = n;
    return HZ_MOVE_OK;
}

static int is_over(const ostate *s) { return s->ending && s->winner != NO_WINNER; }      /* :332-333 */
static int outcome(const ostate *s) { return !is_over(s) ? 0 : s->winner == 0 ? 1 : s->winner == 1 ? -1 : 0; }

/* ---- canonical key: get_canonical_tuple / __hash__, harmonies_engine.py:81-113 -------- */
static uint64_t hash_words23(const uint32_t *w) {
    uint64_t h = 0x9E3779B97F4A7C15ull;
    for (int i = 0; i < HZ_CANON_WORDS; i++) {
        uint32_t x = w[i];
        if (i == 22) x &= 0x0FFFFFFFu;           /* ending flag and winner are not in the tuple */
        h = (h ^ x) * 0x9FB21C651E98DF25ull;
        h ^= h >> 32;
    }
    return mix64(h);
}
/* HZ_KEY_EXACT: identity == equality of get_canonical_tuple (what __eq__ defines). */
static uint64_t canon_hash_words(const uint32_t *w) { return hash_words23(w); }

/* HZ_KEY_REFERENCE: identity == equality of Python's hash(get_canonical_tuple()), which is
 * what MCTS.py actually keys nodes by (Node.id = hash(state), MCTS.py:14; lookup by id only,
 * MCTS.py:177,185).  CPython hashes ints to themselves except hash(-1) == -2 == hash(-2), and
 * a tuple's hash is a function of its items' hashes, so two states share a key iff their
 * tuples agree after replacing every coordinate -1 by -2: the board items, listed in sorted
 * coordinate order (harmonies_engine.py:83-96), must have equal (alias(q), alias(r), stack)
 * sequences.  The normal form used here is the leftmost embedding of that sequence. */
static int py_int_hash(int x) { return x == -1 ? -2 : x; }
static void ref_key_words(const uint32_t *w, uint32_t *out) {
    ostate s, c; unpack(w, &s); c = s;
    for (int p = 0; p < 2; p++) {
        memset(c.height[p], 0, sizeof c.height[p]);
        int next = 0;                            /* first hex index still free for embedding */
        for (int i = 0; i < 23; i++) {
            if (!s.height[p][i]) continue;
            int j = next;
            while (py_int_hash(g_q[j]) != py_int_hash(g_q[i]) || py_int_hash(g_r[j]) != py_int_hash(g_r[i])) j++;
            c.height[p][j] = s.height[p][i];
            memcpy(c.stack[p][j], s.stack[p][i], 3);
            next = j + 1;
        }
    }
    uint32_t full[32]; pack(&c, full);
    memcpy(out, full, HZ_CANON_WORDS * sizeof(uint32_t));
    out[22] &= 0x0FFFFFFFu;
}
static uint64_t key_hash(const uint32_t *w, int mode) {
    if (mode == HZ_KEY_EXACT) return hash_words23(w);
    uint32_t k[HZ_CANON_WORDS]; ref_key_words(w, k);
    return hash_words23(k);
}
static int key_equal(const uint32_t *a, const uint32_t *b, int mode) {
    uint32_t ka[HZ_CANON_WORDS], kb[HZ_CANON_WORDS];
    if (mode == HZ_KEY_EXACT) { memcpy(ka, a, sizeof ka); memcpy(kb, b, sizeof kb); ka[22] &= 0x0FFFFFFFu; kb[22] &= 0x0FFFFFFFu; }
    else { ref_key_words(a, ka); ref_key_words(b, kb); }
    return memcmp(ka, kb, sizeof ka) == 0;
}

/* ---- create_state_tensors: process_game_state.py:15-137 ------------------------------ */
static void encode(const ostate *s, float *board, float *glob) {
    memset(board, 0, 38 * 35 * sizeof(float));
    for (int p = 0; p < 2; p++)
        for (int i = 0; i < 23; i++) {
            int y = g_r[i] + 2, x = g_q[i] + 3;                  /* :48-49 */
            for (int l = 0; l < s->height[p][i]; l++)
                board[(p * 18 + s->stack[p][i][l] * 3 + l) * 35 + y * 7 + x] = 1.0f;    /* :66-67 */
        }
    float phase_val = (s->phase >= 0 && s->phase <= 3) ? (float)(s->phase / 3.0) : 0.0f; /* :75-81 */
    for (int i = 0; i < 23; i++) {                               /* mask: only valid hexes, :34-39,85 */
        int cell = (g_r[i] + 2) * 7 + g_q[i] + 3;
        board[36 * 35 + cell] = (float)s->player;                /* :71 */
        board[37 * 35 + cell] = phase_val;
    }
    memset(glob, 0, 42 * sizeof(float));
    for (int i = 0; i < 5 && i < s->n_piles; i++)                /* :98-107 */
        for (int k = 0; k < s->pile_len[i]; k++) glob[i * 6 + s->pile[i][k]] += 1.0f;
    for (int k = 0; k < s->hand_len; k++) glob[30 + s->hand[k]] += 1.0f;            /* :112-118 */
    for (int i = 0; i < 36; i++) glob[i] = (float)((double)glob[i] / 3.0);
    for (int t = 0; t < 6; t++) glob[36 + t] = (float)((double)s->bag[t] / (double)INIT_BAG[t]);  /* :122-130 */
}

/* ====================================================================================== */
/* exported batch functions                                                                 */
/* ====================================================================================== */
void hzo_init_states(uint32_t *states, int64_t n, const uint64_t *keys, uint64_t seed, uint64_t first_id) {
    geometry();
    for (int64_t g = 0; g < n; g++) {                            /* __init__, :66-79 */
        ostate s; memset(&s, 0, sizeof s);
        for (int t = 0; t < 6; t++) s.bag[t] = INIT_BAG[t];
        s.winner = NO_WINNER;
        s.key = keys ? keys[g] : rand64(seed, first_id + (uint64_t)g);
        replenish(&s, HZ_NO_DRAW);
        pack(&s, states + g * 32);
    }
}

void hzo_legal_mask(const uint32_t *states, int64_t n, uint32_t *mask) {
    geometry();
    for (int64_t g = 0; g < n; g++) {
        ostate s; unpack(states + g * 32, &s);
        int acts[HZ_ACTION_SIZE], k = legal_actions(&s, acts);
        uint32_t *m = mask + g * 5; memset(m, 0, 5 * sizeof(uint32_t));
        for (int i = 0; i < k; i++) m[acts[i] >> 5] |= 1u << (acts[i] & 31);
    }
}

void hzo_apply(uint32_t *states, int64_t n, const int16_t *actions, const uint16_t *draws, uint8_t *status) {
    geometry();
    for (int64_t g = 0; g < n; g++) {
        ostate s; unpack(states + g * 32, &s);
        int st = apply_action(&s, actions[g], draws ? draws[g] : HZ_NO_DRAW);
        if (st == HZ_MOVE_OK) pack(&s, states + g * 32);
        if (status) status[g] = (uint8_t)st;
    }
}

void hzo_score(const uint32_t *states, int64_t n, int16_t *scores, int16_t *terms) {
    geometry();
    for (int64_t g = 0; g < n; g++) {
        ostate s; unpack(states + g * 32, &s);
        for (int p = 0; p < 2; p++) {
            int t[5]; score_terms(&s, p, t);
            if (terms) for (int k = 0; k < 5; k++) terms[(g * 2 + p) * 5 + k] = (int16_t)t[k];
            if (scores) scores[g * 2 + p] = (int16_t)(t[0] + t[1] + t[2] + t[3] + t[4]);
        }
    }
}

void hzo_encode(const uint32_t *states, int64_t n, float *board, float *glob) {
    geometry();
    for (int64_t g = 0; g < n; g++) {
        ostate s; unpack(states + g * 32, &s);
        encode(&s, board + g * 38 * 35, glob + g * 42);
    }
}

void hzo_canon_hash(const uint32_t *states, int64_t n, int mode, uint64_t *out) {
    geometry();
    for (int64_t g = 0; g < n; g++) out[g] = key_hash(states + g * 32, mode);
}

void hzo_outcome(const uint32_t *states, int64_t n, uint8_t *over, int8_t *out) {
    for (int64_t g = 0; g < n; g++) {
        ostate s; unpack(states + g * 32, &s);
        if (over) over[g] = (uint8_t)is_over(&s);
        if (out) out[g] = (int8_t)outcome(&s);
    }
}

static int random_action(const ostate *s) {
    int acts[HZ_ACTION_SIZE], k = legal_actions(s, acts);
    if (k == 0) return -1;
    uint64_t r = rand64(s->key ^ HZ_PLAYOUT_SALT, s->moves);
    return acts[((r >> 32) * (uint64_t)k) >> 32];
}

void hzo_random_actions(const uint32_t *states, int64_t n, int16_t *actions) {
    geometry();
    for (int64_t g = 0; g < n; g++) {
        ostate s; unpack(states + g * 32, &s);
        actions[g] = (int16_t)random_action(&s);
    }
}

/* choose_move_greedy (evaluation.py:137-196): the legal move whose successor state has the
 * highest score for the mover; first strict maximum in legal (ascending action) order. */
void hzo_greedy_actions(const uint32_t *states, int64_t n, int16_t *actions) {
    geometry();
    for (int64_t g = 0; g < n; g++) {
        ostate s; unpack(states + g * 32, &s);
        int acts[HZ_ACTION_SIZE], k = legal_actions(&s, acts), best = -1, best_score = -1000000;
        for (int i = 0; i < k; i++) {
            ostate c = s;
            if (apply_action(&c, acts[i], HZ_NO_DRAW) != HZ_MOVE_OK) continue;    /* evaluation.py:172-178 */
            int sc = score_player(&c, s.player);                                  /* :162 */
            if (sc > best_score) { best_score = sc; best = acts[i]; }             /* :167-169 */
        }
        actions[g] = (int16_t)best;
    }
}

typedef struct { uint32_t *states; int64_t lo, hi; int max_steps; uint32_t *steps; uint64_t total; } playout_job;

static void *playout_worker(void *arg) {
    playout_job *j = (playout_job *)arg;
    for (int64_t g = j->lo; g < j->hi; g++) {
        ostate s; unpack(j->states + g * 32, &s);
        uint32_t k = 0;
        while ((int)k < j->max_steps && !is_over(&s)) {
            int a = random_action(&s);
            if (a < 0 || apply_action(&s, a, HZ_NO_DRAW) != HZ_MOVE_OK) break;
            k++;
        }
        pack(&s, j->states + g * 32);
        if (j->steps) j->steps[g] = k;
        j->total += k;
    }
    return NULL;
}

/* random playouts to the end of the game (BASELINE.json configs[0..1]); returns total steps */
uint64_t hzo_playout(uint32_t *states, int64_t n, int max_steps, uint32_t *steps, int n_threads) {
    geometry();
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    pthread_t th[256]; playout_job jobs[256];
    for (int t = 0; t < n_threads; t++) {
        jobs[t] = (playout_job){states, n * t / n_threads, n * (t + 1) / n_threads, max_steps, steps, 0};
        pthread_create(&th[t], NULL, playout_worker, &jobs[t]);
    }
    uint64_t total = 0;
    for (int t = 0; t < n_threads; t++) { pthread_join(th[t], NULL); total += jobs[t].total; }
    return total;
}

/* ====================================================================================== */
/* MCTS: MCTS.py:8-441                                                                      */
/* ====================================================================================== */
typedef void (*hzo_eval_fn)(const uint32_t *leaf_state, float *policy143, double *value, void *user);

typedef struct { int child, N, action, mover, V; double W; float P; } oedge;   /* V: in-flight (virtual-loss) visits */
typedef struct { uint32_t w[32]; uint64_t hash; int first_edge, n_edges, player; } onode;   /* hash = tree key */
typedef struct {
    onode *nodes; int n_nodes, cap_nodes;
    oedge *edges; int n_edges, cap_edges;
    int *table; int table_mask, key_mode;
} otree;

static void fake_eval(const uint32_t *leaf, float *policy, double *value, void *user) {
    (void)user;
    uint64_t h = canon_hash_words(leaf);
    for (int a = 0; a < HZ_ACTION_SIZE; a++) policy[a] = (float)(mix64(h ^ (uint64_t)(a + 1)) >> 40) * 0x1p-24f;
    *value = (double)(mix64(h ^ 0x5EEDull) >> 40) * 0x1p-23 - 1.0;
}

/* MCTS.tree lookup (MCTS.py:184-186) keyed by the canonical hash, with full-key compare */
static int tree_find_or_add(otree *t, const uint32_t *w, uint64_t h, int *was_new) {
    int slot = (int)(h & (uint64_t)t->table_mask);
    while (t->table[slot] >= 0) {
        onode *nd = &t->nodes[t->table[slot]];
        if (nd->hash == h && key_equal(nd->w, w, t->key_mode)) { *was_new = 0; return t->table[slot]; }
        slot = (slot + 1) & t->table_mask;
    }
    if (t->n_nodes == t->cap_nodes) return -1;
    int id = t->n_nodes++;
    onode *nd = &t->nodes[id];
    memcpy(nd->w, w, sizeof nd->w);
    nd->hash = h; nd->first_edge = 0; nd->n_edges = 0;
    nd->player = (w[22] >> 24) & 1;                              /* Node.current_player, MCTS.py:11 */
    t->table[slot] = id;
    *was_new = 1;
    return id;
}

/* Whole-tree copy of a finished search (tests compare it node for node with the device arenas).
 * Caller-owned arrays of cap_nodes / cap_edges entries; nodes in creation order, edges in
 * append order, so ids are the tree's own.  Entries past the caps are not copied. */
typedef struct {
    int cap_nodes, cap_edges;
    uint32_t *words;                                   /* [cap_nodes * 32] */
    uint64_t *hash;                                    /* tree key */
    int32_t *first_edge, *n_edges, *player;
    int32_t *child, *N, *action, *mover, *V;
    double *W;
    float *P;
} hzo_tree_dump;

static void dump_tree(const otree *t, hzo_tree_dump *d) {
    if (!d) return;
    for (int i = 0; i < t->n_nodes && i < d->cap_nodes; i++) {
        const onode *nd = &t->nodes[i];
        memcpy(d->words + (size_t)i * 32, nd->w, sizeof nd->w);
        d->hash[i] = nd->hash; d->first_edge[i] = nd->first_edge; d->n_edges[i] = nd->n_edges; d->player[i] = nd->player;
    }
    for (int i = 0; i < t->n_edges && i < d->cap_edges; i++) {
        const oedge *e = &t->edges[i];
        d->child[i] = e->child; d->N[i] = e->N; d->W[i] = e->W; d->P[i] = e->P;
        d->action[i] = e->action; d->mover[i] = e->mover; d->V[i] = e->V;
    }
}

/* One full search = get_best_action_and_pi (MCTS.py:272-381) up to the root statistics.
 * Outputs (each [143], indexed by action, nullable): N, W, P, child; `dump` (nullable) receives
 * the whole tree.  Returns 0 or -1 on arena overflow. */
int hzo_search(const uint32_t *root, uint64_t search_key, int sims, double cpuct, int key_mode,
               const float *noise, double eps, hzo_eval_fn eval, void *user, int32_t *outN, double *outW, float *outP,
               int32_t *out_child, int32_t *out_nodes, int32_t *out_edges, hzo_tree_dump *dump) {
    geometry();
    if (!eval) eval = fake_eval;
    otree t;
    t.cap_nodes = 1 + 69 * sims; t.cap_edges = 69 * sims + 1;
    int tsize = 1; while (tsize < 2 * t.cap_nodes) tsize <<= 1;
    t.table_mask = tsize - 1;
    t.nodes = (onode *)malloc(sizeof(onode) * (size_t)t.cap_nodes);
    t.edges = (oedge *)malloc(sizeof(oedge) * (size_t)t.cap_edges);
    t.table = (int *)malloc(sizeof(int) * (size_t)tsize);
    int *path = (int *)malloc(sizeof(int) * (size_t)(sims + 2));
    for (int i = 0; i < tsize; i++) t.table[i] = -1;
    t.n_nodes = 0; t.n_edges = 0; t.key_mode = key_mode;
    int was_new, rc = 0;
    tree_find_or_add(&t, root, key_hash(root, key_mode), &was_new);          /* MCTS.py:288-289,54 */
    float cpuct_f = (float)cpuct;

    for (int sim = 0; sim < sims && rc == 0; sim++) {                       /* MCTS.py:291 */
        /* move_to_leaf, MCTS.py:63-149 */
        int cur = 0, depth = 0;
        while (t.nodes[cur].n_edges > 0) {
            onode *nd = &t.nodes[cur];
            long ns = 0;
            for (int k = 0; k < nd->n_edges; k++) ns += t.edges[nd->first_edge + k].N;     /* :95-97 */
            double sqrt_ns = sqrt(ns > 1 ? (double)ns : 1.0);                                /* :99 */
            double best = -INFINITY; int best_e = -1;
            for (int k = 0; k < nd->n_edges; k++) {
                oedge *e = &t.edges[nd->first_edge + k];
                float cp = cpuct_f * e->P;                       /* np.float32 product, :107-109 */
                double u = (double)cp * sqrt_ns / (double)(1 + e->N);                        /* :110-111 */
                double q = e->N ? e->W / (double)e->N : 0.0;                                 /* Q, :254 */
                if (q + u > best) { best = q + u; best_e = nd->first_edge + k; }             /* :118 */
            }
            if (best_e < 0) break;                               /* :125-133 (NaN priors only) */
            path[depth++] = best_e;
            cur = t.edges[best_e].child;                         /* :145-146 */
        }
        onode *leaf = &t.nodes[cur];
        ostate ls; unpack(leaf->w, &ls);
        double value;
        if (!is_over(&ls)) {                                     /* :297 */
            float policy[HZ_ACTION_SIZE];
            eval(leaf->w, policy, &value, user);                 /* :299-304 */
            int acts[HZ_ACTION_SIZE], k = legal_actions(&ls, acts);
            if (cur == 0 && noise && k > 0) {                    /* root Dirichlet mix, :308-326 */
                double sum = 0.0;
                for (int i = 0; i < k; i++) sum += (double)noise[acts[i]];
                float one_minus = (float)(1.0 - eps);
                for (int i = 0; i < k; i++) {
                    float keep = one_minus * policy[acts[i]];
                    policy[acts[i]] = (float)((double)keep + eps * ((double)noise[acts[i]] / sum));   /* :323 */
                }
            }
            /* expand_leaf, MCTS.py:151-218 */
            int first = t.n_edges, cnt = 0;
            for (int i = 0; i < k; i++) {
                ostate cs = ls;
                cs.key = search_key; cs.event = ((uint32_t)sim << 8) | (uint32_t)acts[i];
                if (apply_action(&cs, acts[i], HZ_NO_DRAW) != HZ_MOVE_OK) continue;
                cs.key = ls.key; cs.event = ls.event;            /* rng fields are not identity */
                uint32_t cw[32]; pack(&cs, cw);
                uint64_t h = key_hash(cw, key_mode);
                if (h == leaf->hash) continue;                   /* self-loop guard, :189-194 */
                int child = tree_find_or_add(&t, cw, h, &was_new);                   /* :185-204 */
                leaf = &t.nodes[cur];
                if (child < 0 || t.n_edges == t.cap_edges) { rc = -1; break; }
                oedge *e = &t.edges[t.n_edges++];
                e->child = child; e->N = 0; e->V = 0; e->W = 0.0; e->P = policy[acts[i]];
                e->action = acts[i]; e->mover = leaf->player;    /* Edge, MCTS.py:23-39 */
                cnt++;
            }
            leaf->first_edge = first; leaf->n_edges = cnt;
        } else {                                                 /* terminal leaf, :333-341 */
            int oc = outcome(&ls);
            value = oc == 0 ? 0.0 : (leaf->player == 0 ? (double)oc : -(double)oc);
        }
        for (int d = depth - 1; d >= 0; d--) {                   /* back_fill, :220-264 */
            oedge *e = &t.edges[path[d]];
            double dir = e->mover == t.nodes[cur].player ? 1.0 : -1.0;
            e->N += 1; e->W += value * dir;
        }
    }
    for (int a = 0; a < HZ_ACTION_SIZE; a++) {
        if (outN) outN[a] = 0;
        if (outW) outW[a] = 0.0;
        if (outP) outP[a] = 0.0f;
        if (out_child) out_child[a] = -1;
    }
    for (int k = 0; k < t.nodes[0].n_edges; k++) {               /* root statistics, :355-376 */
        oedge *e = &t.edges[t.nodes[0].first_edge + k];
        if (outN) outN[e->action] = e->N;
        if (outW) outW[e->action] = e->W;
        if (outP) outP[e->action] = e->P;
        if (out_child) out_child[e->action] = e->child;
    }
    if (out_nodes) *out_nodes = t.n_nodes;
    if (out_edges) *out_edges = t.n_edges;
    dump_tree(&t, dump);
    free(t.nodes); free(t.edges); free(t.table); free(path);
    return rc;
}


/* Virtual-loss search (throughput mode; north_star "select, expand and backup kernels using
 * virtual loss"): `steps` rounds of `leaves` simulations per tree.  Within a round the K
 * descents run one after the other; every edge on a chosen path carries one in-flight visit
 * (N' = N + V, W' = W - V: a provisional loss for the mover) so that later descents of the
 * round spread out.  Then the K leaves are evaluated together and, in order j = 0..K-1,
 * expanded (if still unexpanded) and backed up (N += 1, W += v*dir, V -= 1).  Simulation
 * index of leaf j of round r is r*K + j (draw events, node ids).  leaves == 1 is exactly
 * hzo_search (the reference's sequential search). */
int hzo_search_vl(const uint32_t *root, uint64_t search_key, int steps, int leaves, double cpuct, int key_mode,
                  const float *noise, double eps, hzo_eval_fn eval, void *user, int32_t *outN, double *outW,
                  float *outP, int32_t *out_child, int32_t *out_nodes, int32_t *out_edges, hzo_tree_dump *dump) {
    geometry();
    if (!eval) eval = fake_eval;
    int sims = steps * leaves;
    otree t;
    t.cap_nodes = 1 + 69 * sims; t.cap_edges = 69 * sims + 1;
    int tsize = 1; while (tsize < 2 * t.cap_nodes) tsize <<= 1;
    t.table_mask = tsize - 1;
    t.nodes = (onode *)malloc(sizeof(onode) * (size_t)t.cap_nodes);
    t.edges = (oedge *)malloc(sizeof(oedge) * (size_t)t.cap_edges);
    t.table = (int *)malloc(sizeof(int) * (size_t)tsize);
    int *path = (int *)malloc(sizeof(int) * (size_t)leaves * (size_t)(sims + 2));
    int *depth = (int *)malloc(sizeof(int) * (size_t)leaves), *leafs = (int *)malloc(sizeof(int) * (size_t)leaves);
    for (int i = 0; i < tsize; i++) t.table[i] = -1;
    t.n_nodes = 0; t.n_edges = 0; t.key_mode = key_mode;
    int was_new, rc = 0;
    tree_find_or_add(&t, root, key_hash(root, key_mode), &was_new);
    float cpuct_f = (float)cpuct;
    for (int step = 0; step < steps && rc == 0; step++) {
        for (int j = 0; j < leaves; j++) {                        /* K descents with virtual loss */
            int *pj = path + (size_t)j * (size_t)(sims + 2);
            int cur = 0, d = 0;
            while (t.nodes[cur].n_edges > 0) {
                onode *nd = &t.nodes[cur];
                long ns = 0;
                for (int k = 0; k < nd->n_edges; k++) ns += t.edges[nd->first_edge + k].N + t.edges[nd->first_edge + k].V;
                double sqrt_ns = sqrt(ns > 1 ? (double)ns : 1.0);
                double best = -INFINITY; int best_e = -1;
                for (int k = 0; k < nd->n_edges; k++) {
                    oedge *e = &t.edges[nd->first_edge + k];
                    int n_eff = e->N + e->V;
                    double w_eff = e->W - (double)e->V;
                    float cp = cpuct_f * e->P;
                    double u = (double)cp * sqrt_ns / (double)(1 + n_eff);
                    double q = n_eff ? w_eff / (double)n_eff : 0.0;
                    if (q + u > best) { best = q + u; best_e = nd->first_edge + k; }
                }
                if (best_e < 0) break;
                pj[d++] = best_e;
                cur = t.edges[best_e].child;
            }
            for (int i = 0; i < d; i++) t.edges[pj[i]].V += 1;
            depth[j] = d; leafs[j] = cur;
        }
        for (int j = 0; j < leaves && rc == 0; j++) {             /* evaluate, expand, back up in order */
            int sim = step * leaves + j, cur = leafs[j];
            int *pj = path + (size_t)j * (size_t)(sims + 2);
            onode *leaf = &t.nodes[cur];
            ostate ls; unpack(leaf->w, &ls);
            double value;
            if (!is_over(&ls)) {
                float policy[HZ_ACTION_SIZE];
                eval(leaf->w, policy, &value, user);
                if (leaf->n_edges == 0) {                         /* not expanded earlier in this round */
                    int acts[HZ_ACTION_SIZE], k = legal_actions(&ls, acts);
                    if (cur == 0 && noise && k > 0) {
                        double sum = 0.0;
                        for (int i = 0; i < k; i++) sum += (double)noise[acts[i]];
                        float one_minus = (float)(1.0 - eps);
                        for (int i = 0; i < k; i++) {
                            float keep = one_minus * policy[acts[i]];
                            policy[acts[i]] = (float)((double)keep + eps * ((double)noise[acts[i]] / sum));
                        }
                    }
                    int first = t.n_edges, cnt = 0;
                    for (int i = 0; i < k; i++) {
                        ostate cs = ls;
                        cs.key = search_key; cs.event = ((uint32_t)sim << 8) | (uint32_t)acts[i];
                        if (apply_action(&cs, acts[i], HZ_NO_DRAW) != HZ_MOVE_OK) continue;
                        cs.key = ls.key; cs.event = ls.event;
                        uint32_t cw[32]; pack(&cs, cw);
                        uint64_t h = key_hash(cw, key_mode);
                        if (h == leaf->hash) continue;
                        int child = tree_find_or_add(&t, cw, h, &was_new);
                        leaf = &t.nodes[cur];
                        if (child < 0 || t.n_edges == t.cap_edges) { rc = -1; break; }
                        oedge *e = &t.edges[t.n_edges++];
                        e->child = child; e->N = 0; e->V = 0; e->W = 0.0; e->P = policy[acts[i]];
                        e->action = acts[i]; e->mover = leaf->player;
                        cnt++;
                    }
                    leaf->first_edge = first; leaf->n_edges = cnt;
                }
            } else {
                int oc = outcome(&ls);
                value = oc == 0 ? 0.0 : (leaf->player == 0 ? (double)oc : -(double)oc);
            }
            for (int d = depth[j] - 1; d >= 0; d--) {
                oedge *e = &t.edges[pj[d]];
                double dir = e->mover == t.nodes[cur].player ? 1.0 : -1.0;
                e->N += 1; e->W += value * dir; e->V -= 1;
            }
        }
    }
    for (int a = 0; a < HZ_ACTION_SIZE; a++) {
        if (outN) outN[a] = 0;
        if (outW) outW[a] = 0.0;
        if (outP) outP[a] = 0.0f;
        if (out_child) out_child[a] = -1;
    }
    for (int k = 0; k < t.nodes[0].n_edges; k++) {
        oedge *e = &t.edges[t.nodes[0].first_edge + k];
        if (outN) outN[e->action] = e->N;
        if (outW) outW[e->action] = e->W;
        if (outP) outP[e->action] = e->P;
        if (out_child) out_child[e->action] = e->child;
    }
    if (out_nodes) *out_nodes = t.n_nodes;
    if (out_edges) *out_edges = t.n_edges;
    dump_tree(&t, dump);
    free(t.nodes); free(t.edges); free(t.table); free(path); free(depth); free(leafs);
    return rc;
}

/* Move choice, MCTS.py:394-423: greedy = first max N in ascending action order; exploratory
 * = first action whose running visit sum exceeds u*total.  Returns -1 without visits. */
int hzo_choose(const int32_t *N, float u, int exploratory) {
    long total = 0;
    for (int a = 0; a < HZ_ACTION_SIZE; a++) total += N[a];
    if (total <= 0) return -1;
    if (exploratory) {
        long acc = 0; int last = -1;
        for (int a = 0; a < HZ_ACTION_SIZE; a++) {
            if (N[a] <= 0) continue;
            acc += N[a]; last = a;
            if ((double)acc > (double)u * (double)total) return a;
        }
        return last;
    }
    int best = -1, bestN = 0;
    for (int a = 0; a < HZ_ACTION_SIZE; a++) if (N[a] > bestN) { bestN = N[a]; best = a; }   /* :420-423 */
    return best;
}

typedef struct { const uint32_t *roots; const uint64_t *keys; int64_t lo, hi; int sims; double cpuct; int32_t *N; } search_job;
static void *search_worker(void *arg) {
    search_job *j = (search_job *)arg;
    for (int64_t g = j->lo; g < j->hi; g++)
        hzo_search(j->roots + g * 32, j->keys[g], j->sims, j->cpuct, HZ_KEY_REFERENCE, NULL, 0.0, NULL, NULL,
                   j->N ? j->N + g * HZ_ACTION_SIZE : NULL, NULL, NULL, NULL, NULL, NULL, NULL);
    return NULL;
}
/* many independent searches with the synthetic evaluator, for CPU-baseline timing */
void hzo_search_batch(const uint32_t *roots, const uint64_t *keys, int64_t n, int sims, double cpuct,
                      int32_t *N, int n_threads) {
    geometry();
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    pthread_t th[256]; search_job jobs[256];
    for (int t = 0; t < n_threads; t++) {
        jobs[t] = (search_job){roots, keys, n * t / n_threads, n * (t + 1) / n_threads, sims, cpuct, N};
        pthread_create(&th[t], NULL, search_worker, &jobs[t]);
    }
    for (int t = 0; t < n_threads; t++) pthread_join(th[t], NULL);
}
