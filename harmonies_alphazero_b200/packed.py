"""Host-side view of the 128-byte packed game state (layout: include/harmonies_b200.h).

Pure-Python/numpy conversions between the reference's attribute-level state
(``harmonies_engine.py:70-78``: dict boards, string tile names) and the packed record the
CUDA kernels work on, plus the integer draw-source primitives (mix / rand / draw_pile)
that define the deterministic replacement of ``random.sample`` in ``_draw_tiles``
(``harmonies_engine.py:120-130``).  No game logic lives here.
"""

import numpy as np

from .constants import (
    TILE_TYPES,
    TYPE_INDEX,
    PHASES,
    PHASE_INDEX,
    sorted_coords,
    coordinate_to_index_map,
    INITIAL_BAG_BY_TYPE,
    NUM_HEXES,
)

STATE_WORDS = 32
STATE_BYTES = 128
CANON_WORDS = 23
MASK_WORDS = 5
NO_DRAW = 0xFFFF
M64 = (1 << 64) - 1
PLAYOUT_SALT = 0xA5A5F00DC0FFEE11
SEARCH_SALT = 0x5EA2C47EE5A17B00   # default in-tree draw stream key: rand(state key ^ SEARCH_SALT, moves)
ROLLOUT_SALT = 0x2011C0A75EED5A17  # rollout keys of hz_tree_rollout_eval: rand(search key ^ ROLLOUT_SALT, exact canonical hash)

W_BOARD0, W_BOARD1 = 0, 9
W_PILES01, W_PILES23, W_PILE4H = 18, 19, 20
W_BAG0, W_BAG1META, W_SCORES = 21, 22, 23
W_KEYLO, W_KEYHI, W_EVENT, W_MOVES = 24, 25, 26, 27


# ---- draw source -------------------------------------------------------------------
def mix(z):
    z &= M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def rand(key, ctr):
    return mix((key & M64) ^ mix((ctr + 0x9E3779B97F4A7C15) & M64))


def draw_pile(bag_counts, z, n=3):
    """Draw min(n, total) tiles from ``bag_counts`` (list of 6, TILE_TYPES order, mutated).

    Returns the list of drawn type indices in draw order."""
    out = []
    for j in range(n):
        total = sum(bag_counts)
        if total == 0:
            break
        x = (z >> (21 * j)) & 0x1FFFFF
        r = (x * total) >> 21
        for t in range(6):
            if r < bag_counts[t]:
                break
            r -= bag_counts[t]
        bag_counts[t] -= 1
        out.append(t)
    return out


def multiset_code(tiles):
    """<=3 tile names/type indices -> 6 x 2-bit counts."""
    code = 0
    for t in tiles:
        ti = TYPE_INDEX[t] if isinstance(t, str) else int(t)
        code += 1 << (2 * ti)
    return code


def multiset_tiles(code):
    """6 x 2-bit counts -> list of tile names in TILE_TYPES order."""
    out = []
    for t in range(6):
        out.extend([TILE_TYPES[t]] * ((code >> (2 * t)) & 3))
    return out


# ---- pack / unpack -----------------------------------------------------------------
def _winner_code(game_over, winner):
    if winner is None:
        return 0
    return {0: 1, 1: 2, -1: 3}[winner]


def pack_fields(
    player_boards,
    tile_bag,
    available_piles,
    current_player,
    tiles_in_hand,
    turn_phase,
    game_over=False,
    winner=None,
    final_scores=(0, 0),
    rng_key=0,
    rng_event=0,
    moves=0,
):
    """Reference-style fields -> np.uint32[32].  Raises ValueError on anything the packed
    format cannot hold (unknown tile / coordinate / phase, stack higher than 3, ...)."""
    w = [0] * STATE_WORDS
    for p in (0, 1):
        base = W_BOARD0 if p == 0 else W_BOARD1
        for coord, stack in player_boards[p].items():
            if coord not in coordinate_to_index_map:
                raise ValueError(f"Invalid coordinate: {coord}")
            if len(stack) > 3:
                raise ValueError(f"Stack higher than 3 at {coord}: {stack}")
            i = coordinate_to_index_map[coord]
            for level, tile in enumerate(stack):
                if tile not in TYPE_INDEX:
                    raise ValueError(f"Unknown tile type: {tile!r}")
                code = TYPE_INDEX[tile] + 1
                for b in range(3):
                    if (code >> b) & 1:
                        w[base + level * 3 + b] |= 1 << i
    if len(available_piles) > 5:
        raise ValueError("more than 5 piles")
    codes = []
    for pile in available_piles:
        if len(pile) > 3:
            raise ValueError(f"pile larger than 3: {pile}")
        for t in pile:
            if t not in TYPE_INDEX:
                raise ValueError(f"Unknown tile type: {t!r}")
        codes.append(multiset_code(pile))
    codes += [0] * (5 - len(codes))
    if len(tiles_in_hand) > 3:
        raise ValueError(f"hand larger than 3: {tiles_in_hand}")
    for t in tiles_in_hand:
        if t not in TYPE_INDEX:
            raise ValueError(f"Unknown tile type: {t!r}")
    hand = multiset_code(tiles_in_hand)
    w[W_PILES01] = codes[0] | (codes[1] << 16)
    w[W_PILES23] = codes[2] | (codes[3] << 16)
    w[W_PILE4H] = codes[4] | (hand << 16)
    bag = [int(tile_bag.get(t, 0)) for t in TILE_TYPES]
    if any(not (0 <= c <= 255) for c in bag):
        raise ValueError(f"bag count out of range: {tile_bag}")
    if turn_phase not in PHASE_INDEX:
        raise ValueError(f"Invalid turn phase: {turn_phase}")
    meta = (
        (int(current_player) & 1)
        | (PHASE_INDEX[turn_phase] << 1)
        | ((1 if game_over else 0) << 4)
        | (_winner_code(game_over, winner) << 5)
    )
    w[W_BAG0] = bag[0] | (bag[1] << 8) | (bag[2] << 16) | (bag[3] << 24)
    w[W_BAG1META] = bag[4] | (bag[5] << 8) | (len(available_piles) << 16) | (meta << 24)
    s0, s1 = int(final_scores[0]), int(final_scores[1])
    w[W_SCORES] = (s0 & 0xFFFF) | ((s1 & 0xFFFF) << 16)
    w[W_KEYLO] = rng_key & 0xFFFFFFFF
    w[W_KEYHI] = (rng_key >> 32) & 0xFFFFFFFF
    w[W_EVENT] = rng_event & 0xFFFFFFFF
    w[W_MOVES] = moves & 0xFFFFFFFF
    return np.array(w, dtype=np.uint32)


def pack_state(state, rng_key=0, rng_event=0, moves=0):
    """Any object with the reference's attributes (harmonies_engine.py:70-78) -> words."""
    return pack_fields(
        state.player_boards,
        state.tile_bag,
        state.available_piles,
        state.current_player,
        state.tiles_in_hand,
        state.turn_phase,
        state.game_over,
        state.winner,
        state.final_scores,
        rng_key=rng_key,
        rng_event=rng_event,
        moves=moves,
    )


def _i16(x):
    x &= 0xFFFF
    return x - 0x10000 if x & 0x8000 else x


def unpack_fields(words):
    """np.uint32[32] -> dict of reference-style fields (plus rng_key/rng_event/moves)."""
    w = [int(x) for x in np.asarray(words, dtype=np.uint32).reshape(-1)[:STATE_WORDS]]
    boards = [{}, {}]
    for p in (0, 1):
        base = W_BOARD0 if p == 0 else W_BOARD1
        for i in range(NUM_HEXES):
            stack = []
            for level in range(3):
                code = sum(((w[base + level * 3 + b] >> i) & 1) << b for b in range(3))
                if code == 0:
                    break
                stack.append(TILE_TYPES[code - 1])
            if stack:
                boards[p][sorted_coords[i]] = stack
    codes = [
        w[W_PILES01] & 0xFFFF,
        w[W_PILES01] >> 16,
        w[W_PILES23] & 0xFFFF,
        w[W_PILES23] >> 16,
        w[W_PILE4H] & 0xFFFF,
    ]
    hand = w[W_PILE4H] >> 16
    n_piles = (w[W_BAG1META] >> 16) & 0xFF
    meta = w[W_BAG1META] >> 24
    bag = [
        w[W_BAG0] & 0xFF,
        (w[W_BAG0] >> 8) & 0xFF,
        (w[W_BAG0] >> 16) & 0xFF,
        (w[W_BAG0] >> 24) & 0xFF,
        w[W_BAG1META] & 0xFF,
        (w[W_BAG1META] >> 8) & 0xFF,
    ]
    winner = {0: None, 1: 0, 2: 1, 3: -1}[(meta >> 5) & 3]
    return {
        "player_boards": boards,
        # same key order as the reference's INITIAL_BAG (constants.py:41)
        "tile_bag": {
            "water": bag[0],
            "plant": bag[1],
            "wood": bag[2],
            "stone": bag[3],
            "field": bag[5],
            "building": bag[4],
        },
        "available_piles": [multiset_tiles(c) for c in codes[:n_piles]],
        "current_player": meta & 1,
        "tiles_in_hand": multiset_tiles(hand),
        "turn_phase": PHASES[(meta >> 1) & 7],
        "game_over": bool((meta >> 4) & 1),
        "winner": winner,
        "final_scores": [_i16(w[W_SCORES]), _i16(w[W_SCORES] >> 16)],
        "rng_key": w[W_KEYLO] | (w[W_KEYHI] << 32),
        "rng_event": w[W_EVENT],
        "moves": w[W_MOVES],
    }


KEY_EXACT, KEY_REFERENCE = 0, 1


def canon_words(words):
    """The 23 words that carry get_canonical_tuple's content (harmonies_engine.py:81-110)."""
    w = np.array(np.asarray(words, dtype=np.uint32).reshape(-1)[:CANON_WORDS], dtype=np.uint32)
    w[W_BAG1META] &= np.uint32(0x0FFFFFFF)
    return w


def _py_int_hash(x):
    return -2 if x == -1 else x  # CPython: hash(-1) == hash(-2) == -2


def ref_key_words(words):
    """Normal form under the identity MCTS.py really uses: Python's hash() of the canonical
    tuple (MCTS.py:14,177,185).  Board items at coordinates that differ only by -1 vs -2
    hash alike, so each board is replaced by the leftmost embedding of its sorted
    (alias(q), alias(r), stack) sequence (see HZ_KEY_REFERENCE in harmonies_b200.h)."""
    w = canon_words(words)
    for base in (W_BOARD0, W_BOARD1):
        planes = [int(x) for x in w[base : base + 9]]
        occ = planes[0] | planes[1] | planes[2]
        out = [0] * 9
        nxt = 0
        for i in range(NUM_HEXES):
            if not (occ >> i) & 1:
                continue
            qi, ri = sorted_coords[i]
            j = nxt
            while (_py_int_hash(sorted_coords[j][0]), _py_int_hash(sorted_coords[j][1])) != (
                _py_int_hash(qi),
                _py_int_hash(ri),
            ):
                j += 1
            for k in range(9):
                out[k] |= ((planes[k] >> i) & 1) << j
            nxt = j + 1
        w[base : base + 9] = np.array(out, dtype=np.uint32)
    return w


def _hash23(w):
    h = 0x9E3779B97F4A7C15
    for x in w:
        h = ((h ^ int(x)) * 0x9FB21C651E98DF25) & M64
        h ^= h >> 32
    return mix(h)


def canon_hash(words, mode=KEY_EXACT):
    """64-bit node key; same function as hz_canon_hash (csrc) and the C oracle."""
    return _hash23(canon_words(words) if mode == KEY_EXACT else ref_key_words(words))


def fake_eval(h):
    """Synthetic evaluator keyed by the canonical hash (hz_tree_fake_eval): exact dyadic
    rationals, so every implementation agrees bit-for-bit."""
    p = np.empty(143, dtype=np.float32)
    for a in range(143):
        p[a] = np.float32((mix(h ^ (a + 1)) >> 40) * 2.0**-24)
    v = (mix(h ^ 0x5EED) >> 40) * 2.0**-23 - 1.0
    return p, float(v)


# ---- actions -----------------------------------------------------------------------
def action_to_move(a):
    """Flat action index -> reference move (int pile index or (tile_type, (q, r)))."""
    a = int(a)
    if a < 5:
        return a
    t, i = divmod(a - 5, NUM_HEXES)
    return (TILE_TYPES[t], sorted_coords[i])


def mask_to_actions(mask_words):
    m = 0
    for k, x in enumerate(np.asarray(mask_words, dtype=np.uint32).reshape(-1)[:MASK_WORDS]):
        m |= int(x) << (32 * k)
    return [a for a in range(143) if (m >> a) & 1]


def actions_to_mask(actions):
    out = np.zeros(MASK_WORDS, dtype=np.uint32)
    for a in actions:
        out[a >> 5] |= np.uint32(1 << (a & 31))
    return out


INITIAL_BAG_COUNTS = list(INITIAL_BAG_BY_TYPE)
