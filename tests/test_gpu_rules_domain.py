"""GPU: the engine's closed-form rules (csrc/hz_core.cuh, csrc/hz_engine.cu) over their whole domains, against the C
oracle.

Random games seldom reach the edges these rules are written for: rings of exactly six field hexes, 4-hex claws next to
4-hex paths, water components of 9 and more hexes in resolve_water, a building whose neighbours show exactly 2 + 2 top
types, the alias moves of the reference key, the last partial warp of k_legal and ties across the lanes of k_greedy.
So each rule is run on every input of its domain, or on a structured family that contains every shape:

- tests/probe_rules.cu runs the neighbour expansion and the six direction pulls on all 2^23 masks, and score_board with
  every large water component scored in place and, separately, through a queue that cannot overflow;
- hz_score, hz_canon_hash, hz_legal_mask, hz_random_actions and hz_greedy_actions run through the public entry points.

The oracle's big sweeps run chunked on a thread pool (ctypes releases the GIL) and once per module.
"""

import ctypes as C
import itertools
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from harmonies_alphazero_b200 import packed as pk
from harmonies_alphazero_b200.constants import NEIGHBOR_MASKS, sorted_coords

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
N_RECS, REC_WORDS = 16, 32
VALID = 0x7FFFFF
ALL_MASKS = 1 << 23
# axial directions in the order of the probe's pulls: E, W, S, N, NE, SW
DIRECTIONS = [(1, 0), (-1, 0), (0, 1), (0, -1), (1, -1), (-1, 1)]
WATER, PLANT, WOOD, STONE, BUILDING, FIELD = range(6)
STACKS = [()] + [s for n in (1, 2, 3) for s in itertools.product(range(6), repeat=n)]   # every stack of height 0-3
SLICE = 1 << 21                                               # records per GPU launch of the 2^23 sweeps


# ---- fixtures and helpers --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    """tests/probe_rules.cu built with the library's flags (and HZ_NVCC_EXTRA, so a -DHZ_DEBUG_BOUNDS run covers it)"""
    from harmonies_alphazero_b200 import build

    so = str(tmp_path_factory.mktemp("probe") / "probe_rules.so")
    extra = os.environ.get("HZ_NVCC_EXTRA", "").split()
    cmd = [build._nvcc()] + build.NVCC_FLAGS + extra + ["-shared", "-o", so, os.path.join(HERE, "probe_rules.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    torch.cuda.init()
    return C.CDLL(so)


@pytest.fixture(scope="module")
def hb():
    from harmonies_alphazero_b200 import batched

    batched._lib.load()
    return batched


@pytest.fixture(scope="module")
def orc(oracle):
    oracle.score(np.zeros((1, 32), dtype=np.uint32))            # the oracle's geometry, set up before any thread runs
    return oracle


def _pool_map(fn, recs, chunks=64):
    """fn over chunks of recs on a thread pool; the results (arrays or tuples of arrays) concatenated in order"""
    parts = np.array_split(recs, min(chunks, max(1, len(recs))))
    with ThreadPoolExecutor(os.cpu_count() or 8) as ex:
        res = list(ex.map(fn, parts))
    if isinstance(res[0], tuple):
        return tuple(np.concatenate(r) for r in zip(*res))
    return np.concatenate(res)


def _call(fn, *args):
    """fn(*args) with torch tensors passed as device pointers: args holds them until fn has returned"""
    return fn(*(C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args))


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check(fn, what, *args):
    """run a checking launcher (its last argument is the mismatch buffer) and assert no mismatch"""
    out = torch.zeros(REC_WORDS * (1 + N_RECS), dtype=torch.int32, device="cuda")
    assert _call(fn, *args, out) == 0, f"{what}: CUDA error"
    o = out.cpu().numpy().view(np.uint32)
    n = int(o[0])
    for r in o[REC_WORDS:].reshape(N_RECS, REC_WORDS)[: min(n, N_RECS)]:
        print(what, [hex(int(x)) for x in r[:6]])
    assert n == 0, f"{what}: {n} mismatches, first ones printed above"


def _popc(a):
    return np.bitwise_count(np.asarray(a, dtype=np.uint32)).astype(np.int64)


def _stack_planes(occ, stacks):
    """the 9 planes of a board holding stacks[h] at every hex h of the masks occ (uint32[n]) -> uint32[n, 9]"""
    occ = np.asarray(occ, dtype=np.uint32)
    out = np.zeros((len(occ), 9), dtype=np.uint32)
    for level in range(3):
        for b in range(3):
            pm = sum(1 << h for h, st in enumerate(stacks) if len(st) > level and ((st[level] + 1) >> b) & 1)
            out[:, 3 * level + b] = occ & np.uint32(pm)
    return out


def _records(n):
    return np.zeros((n, 32), dtype=np.uint32)


def _set_meta(recs, player, phase, n_piles=0):
    recs[:, pk.W_BAG1META] = (recs[:, pk.W_BAG1META] & np.uint32(0xFFFF)) | (np.asarray(n_piles, dtype=np.uint32) << 16) | \
        ((np.asarray(player, dtype=np.uint32) | (np.asarray(phase, dtype=np.uint32) << 1)) << 24)


def _set_keys(recs, rng):
    keys = rng.integers(0, 2**63, size=len(recs), dtype=np.uint64) * 2 + rng.integers(0, 2, size=len(recs), dtype=np.uint64)
    recs[:, pk.W_KEYLO] = (keys & 0xFFFFFFFF).astype(np.uint32)
    recs[:, pk.W_KEYHI] = (keys >> 32).astype(np.uint32)
    recs[:, pk.W_MOVES] = rng.integers(0, 2**32, size=len(recs), dtype=np.uint64).astype(np.uint32)
    recs[:, pk.W_EVENT] = rng.integers(0, 2**32, size=len(recs), dtype=np.uint64).astype(np.uint32)


# ---- 1. neighbour expansion and direction pulls ----------------------------------------------------------------------
def _direction_table():
    """hex i's neighbour in each direction (or -1), from the axial coordinates"""
    index = {c: i for i, c in enumerate(sorted_coords)}
    return [[index.get((q + dq, r + dr), -1) for (q, r) in sorted_coords] for dq, dr in DIRECTIONS]


def test_direction_table_partitions_every_neighbour_set():
    table = _direction_table()
    for i in range(23):
        per_dir = [1 << table[d][i] if table[d][i] >= 0 else 0 for d in range(6)]
        assert sum(per_dir) == NEIGHBOR_MASKS[i]                  # disjoint (distinct bits) and complete
        assert len({x for x in per_dir if x}) == bin(NEIGHBOR_MASKS[i]).count("1")
        for d, (dq, dr) in enumerate(DIRECTIONS):                 # opposite directions are inverse maps
            j = table[d][i]
            if j >= 0:
                assert table[DIRECTIONS.index((-dq, -dr))][j] == i


def test_neighbour_expansion_and_pulls_on_every_mask(probe):
    """nbr_alu, the shared-memory LUT and pull_E/W/S/N/NE/SW on all 2^23 masks"""
    table = np.array(_direction_table(), dtype=np.int32)
    _check(probe.probe_nbr_sweep, "nbr", _cuda(np.array(NEIGHBOR_MASKS, dtype=np.uint32).view(np.int32)), _cuda(table))


# ---- scoring: every way of running score_board ----------------------------------------------------------------------
def _gpu_terms(hb, probe, recs):
    """[(way, terms int16[n, 2, 5], block pushes or None)] for hz_score and the probe's two queue modes"""
    st = hb.states_from_numpy(recs)
    sc, tm = hb.score(st, with_terms=True)
    tm = tm.cpu().numpy()
    assert np.array_equal(sc.cpu().numpy(), tm.sum(axis=2, dtype=np.int16))
    out = [("hz_score", tm, None)]
    nb = (len(recs) + 127) // 128
    for queue in (0, 1):
        terms = torch.zeros((len(recs), 2, 5), dtype=torch.int16, device="cuda")
        pushes = torch.zeros(nb, dtype=torch.int32, device="cuda")
        assert _call(probe.probe_score, st, C.c_int64(len(recs)), C.c_int(queue), terms, pushes) == 0
        out.append((("in place", "queue")[queue], terms.cpu().numpy(), pushes.cpu().numpy()))
    return out


def _assert_terms(got, want, recs, what):
    bad = np.nonzero((got != want).any(axis=(1, 2)))[0]
    assert len(bad) == 0, (what, len(bad), recs[bad[0]].tolist(), got[bad[0]].tolist(), want[bad[0]].tolist())


def _score_everywhere(hb, probe, recs, want, what):
    """all three ways against the oracle's terms; returns the queue run's pushes per 128-record block"""
    pushes = None
    for way, tm, p in _gpu_terms(hb, probe, recs):
        _assert_terms(tm, want, recs, f"{what}, {way}")
        if way == "queue":
            pushes = p
    return pushes


# ---- 2 + 3. water, fields and mountains on every top mask ------------------------------------------------------------
# Record m: board 0 holds height-1 water on m and stones on the complement (heights 1-3 by pattern A), board 1
# height-1 fields on m and stones on the complement (pattern B).  So every mask is the water and the field mask of one
# record and the stone mask of both boards of another.
HEIGHT_A = [1 + h % 3 for h in range(23)]
HEIGHT_B = [1 + (h // 2 + 1) % 3 for h in range(23)]


def _terrain(lo, hi):
    m = np.arange(lo, hi, dtype=np.uint32)
    c = ~m & np.uint32(VALID)
    recs = _records(hi - lo)
    recs[:, 0:9] = _stack_planes(m, [(WATER,)] * 23) | _stack_planes(c, [(STONE,) * k for k in HEIGHT_A])
    recs[:, 9:18] = _stack_planes(m, [(FIELD,)] * 23) | _stack_planes(c, [(STONE,) * k for k in HEIGHT_B])
    return recs


@pytest.fixture(scope="module")
def terrain_terms(orc):
    parts = [_pool_map(lambda r: orc.score(r)[1], _terrain(lo, lo + SLICE)) for lo in range(0, ALL_MASKS, SLICE)]
    return np.concatenate(parts)


def test_water_fields_and_mountains_on_every_mask(hb, probe, terrain_terms):
    assert len(terrain_terms) == ALL_MASKS == 8_388_608
    pushes = []
    for lo in range(0, ALL_MASKS, SLICE):
        recs = _terrain(lo, lo + SLICE)
        pushes.append(_score_everywhere(hb, probe, recs, terrain_terms[lo: lo + SLICE], f"terrain from {lo}"))
    pushes = np.concatenate(pushes)
    # the queue run scored every component of >= 5 hexes through resolve_water; hz_score's queue holds 256 of a
    # block's 128 records (same layout), so some of its blocks overflowed and scored the rest in place, and some not
    assert pushes.sum() > 10**6 and pushes.max() <= 8 * 128
    assert (pushes > 256).any() and (pushes <= 256).any()
    w = terrain_terms[:, 0, 4]
    assert w[VALID] == 15 + (7 - 6) * 4                            # the whole board: one river of diameter 6 (7 hexes long)
    f = terrain_terms[:, 1, 2]
    ring = sum(1 << h for h in range(23) if (NEIGHBOR_MASKS[11] >> h) & 1)   # the six hexes around hex 11
    assert f[ring] == 5 and f[ring | (1 << 11)] == 5


# ---- 4. every stack on every hex ----------------------------------------------------------------------------------------
def _every_stack_records():
    """board 0: stack s alone on hex h; board 1: stack s on all 23 hexes.  259 x 23 records"""
    recs = _records(len(STACKS) * 23)
    for s, st in enumerate(STACKS):
        all_hexes = _stack_planes([VALID], [st] * 23)[0]
        for h in range(23):
            recs[s * 23 + h, 0:9] = _stack_planes([1 << h], [st] * 23)[0]
            recs[s * 23 + h, 9:18] = all_hexes
    return recs


def test_every_stack_on_every_hex(hb, probe, orc):
    recs = _every_stack_records()
    assert len(STACKS) == 259 and len(recs) == 5_957
    _, want = orc.score(recs)
    _score_everywhere(hb, probe, recs, want, "every stack")
    assert want[:, :, 0].max() == want[:, :, 1].max() == 23 * 7    # plant on wood-wood, mountains 3 high: everywhere


# ---- 5. every building neighbourhood -----------------------------------------------------------------------------------
def _neighbourhood_records():
    """a building on a height-2 stack at hex c (board 0) and the same building at height 1 or 3 (board 1), times every
    assignment of {empty, the six top types} to c's neighbours; neighbour stacks 1-3 high by the assignment's index"""
    out = []
    for c in range(23):
        nb = [h for h in range(23) if (NEIGHBOR_MASKS[c] >> h) & 1]
        a = np.arange(7 ** len(nb), dtype=np.int64)
        planes = np.zeros((len(a), 9), dtype=np.uint32)
        for j, h in enumerate(nb):
            v = (a // 7 ** j) % 7                                 # 0 empty, else top type v - 1
            height = np.where(v > 0, 1 + (a + j) % 3, 0)
            for level in range(3):
                top = level == height - 1
                code = np.where(top, v, (a + level + j) % 6 + 1)  # tiles below the top: any type
                code = np.where(level < height, code, 0)
                for b in range(3):
                    planes[:, 3 * level + b] |= (((code >> b) & 1) << h).astype(np.uint32)
        recs = _records(len(a))
        recs[:, 0:9] = planes
        recs[:, 9:18] = planes
        bit = np.uint32(1 << c)
        under = np.array([WOOD, STONE, BUILDING])[a % 3] + 1      # what a building may be placed on
        for b in range(3):
            recs[:, b] |= ((under >> b) & 1).astype(np.uint32) * bit
            recs[:, 3 + b] |= np.uint32(((BUILDING + 1) >> b) & 1) * bit
        # board 1: the building alone (height 1) or on two tiles (height 3)
        h3 = (a % 2 == 1)
        for b in range(3):
            recs[:, 9 + b] |= np.where(h3, ((under >> b) & 1), ((BUILDING + 1) >> b) & 1).astype(np.uint32) * bit
            recs[:, 12 + b] |= np.where(h3, ((under >> b) & 1), 0).astype(np.uint32) * bit
            recs[:, 15 + b] |= np.where(h3, ((BUILDING + 1) >> b) & 1, 0).astype(np.uint32) * bit
        out.append(recs)
    return np.concatenate(out)


@pytest.fixture(scope="module")
def neighbourhoods(orc):
    recs = _neighbourhood_records()
    return recs, _pool_map(lambda r: orc.score(r)[1], recs)


def test_every_building_neighbourhood(hb, probe, neighbourhoods):
    recs, want = neighbourhoods
    assert len(recs) == sum(7 ** bin(m).count("1") for m in NEIGHBOR_MASKS) == 906_059
    _score_everywhere(hb, probe, recs, want, "building neighbourhoods")
    # the centre scores on board 0 exactly when its neighbours show >= 3 top types, including exactly 2 + 2 types
    # split between {water, plant, wood} and {stone, building, field}
    assert (want[:, 0, 3] >= 5).sum() > 10**5 and (want[:, 0, 3] == 0).any()


# ---- 6. canonical keys -----------------------------------------------------------------------------------------------
# a distinct stack on every hex (board 1 another set), so that a stack on the wrong hex changes the key
KEY_STACKS = [[STACKS[1 + (7 * h + 3 * p) % 258] for h in range(23)] for p in (0, 1)]


def _key_records(lo, hi):
    m = np.arange(lo, hi, dtype=np.uint32)
    recs = _records(hi - lo)
    recs[:, 0:9] = _stack_planes(m, KEY_STACKS[0])
    recs[:, 9:18] = _stack_planes(m ^ np.uint32(0x555555), KEY_STACKS[1])
    # piles, hand and bag as a record can hold them: piles of 1-3 tiles up to n_piles (0 behind), a hand of 0-3 tiles
    rng = np.random.default_rng(lo + 1)
    n_piles = rng.integers(0, 6, size=hi - lo)
    codes = [np.where(k < n_piles, _multisets(rng, hi - lo, 1), 0) for k in range(5)] + [_multisets(rng, hi - lo, 0)]
    recs[:, pk.W_PILES01] = codes[0] | codes[1] << 16
    recs[:, pk.W_PILES23] = codes[2] | codes[3] << 16
    recs[:, pk.W_PILE4H] = codes[4] | codes[5] << 16
    recs[:, pk.W_BAG0] = rng.integers(0, 2**32, size=hi - lo, dtype=np.uint64).astype(np.uint32)
    recs[:, pk.W_BAG1META] = rng.integers(0, 2**16, size=hi - lo, dtype=np.uint64).astype(np.uint32)
    _set_meta(recs, rng.integers(0, 2, size=hi - lo), rng.integers(0, 5, size=hi - lo), n_piles)
    return recs


def _multisets(rng, n, least):
    """n multiset codes of least..3 tiles"""
    size = rng.integers(least, 4, size=n)
    tiles = rng.integers(0, 6, size=(n, 3)).astype(np.uint32)
    return sum(np.where(j < size, np.uint32(1) << (2 * tiles[:, j]), 0) for j in range(3)).astype(np.uint32)


def _alias(x):
    return -2 if x == -1 else x


def _leftmost_embedding(planes, occ):
    """the board moved to the leftmost embedding of its (alias class, stack) sequence (the oracle's ref_key_words),
    with numpy over records; and whether a stack moved"""
    cls = [(_alias(q), _alias(r)) for q, r in sorted_coords]
    cand = [[j for j in range(23) if cls[j] == cls[i]] for i in range(23)]
    nxt = np.zeros(len(occ), dtype=np.int64)
    out = planes.copy()
    moved = np.zeros(len(occ), dtype=bool)
    for i in range(23):
        on = ((occ >> np.uint32(i)) & np.uint32(1)).astype(bool)
        j = np.full(len(occ), i, dtype=np.int64)
        for c in reversed(cand[i]):
            if c < i:
                j = np.where(c >= nxt, c, j)
        nxt = np.where(on, j + 1, nxt)
        for c in cand[i]:                                          # the stack at i moves down to c
            if c < i:
                mv = on & (j == c)
                moved |= mv
                for k in range(9):
                    bit = (out[:, k] >> np.uint32(i)) & np.uint32(1) & mv.astype(np.uint32)
                    out[:, k] = (out[:, k] & ~(bit << np.uint32(i))) | (bit << np.uint32(c))
    return out, moved


@pytest.fixture(scope="module")
def key_hashes(orc):
    out = {}
    for mode in (pk.KEY_EXACT, pk.KEY_REFERENCE):
        out[mode] = np.concatenate([_pool_map(lambda r, md=mode: orc.canon_hash(r, md), _key_records(lo, lo + SLICE))
                                    for lo in range(0, ALL_MASKS, SLICE)])
    return out


def _gpu_hash(hb, recs, mode):
    return hb.canon_hash(hb.states_from_numpy(recs), mode).cpu().numpy().view(np.uint64)


def test_canonical_keys_on_every_occupancy(hb, key_hashes):
    assert all(len(h) == ALL_MASKS for h in key_hashes.values())
    for lo in range(0, ALL_MASKS, SLICE):
        recs = _key_records(lo, lo + SLICE)
        for mode in (pk.KEY_EXACT, pk.KEY_REFERENCE):
            got = _gpu_hash(hb, recs, mode)
            bad = np.nonzero(got != key_hashes[mode][lo: lo + SLICE])[0]
            assert len(bad) == 0, (mode, len(bad), recs[bad[0]].tolist())


def test_leftmost_embedding_keys(hb, key_hashes):
    """the same reference key for a board and its leftmost embedding, a different exact key wherever a stack moved.
    Only hexes 1-10, 14, 15, 19 and 20 take part in an alias move, so the records of masks 0 .. 2^21 - 1 hold every
    occupancy of them on both boards."""
    recs = _key_records(0, SLICE)
    emb = recs.copy()
    moved = np.zeros(len(recs), dtype=bool)
    for p in (0, 1):
        occ = recs[:, 9 * p] | recs[:, 9 * p + 1] | recs[:, 9 * p + 2]
        emb[:, 9 * p: 9 * p + 9], mv = _leftmost_embedding(recs[:, 9 * p: 9 * p + 9], occ)
        moved |= mv
    assert np.array_equal(_gpu_hash(hb, emb, pk.KEY_REFERENCE), key_hashes[pk.KEY_REFERENCE][:SLICE])
    assert np.array_equal(_gpu_hash(hb, emb, pk.KEY_EXACT) == key_hashes[pk.KEY_EXACT][:SLICE], ~moved)
    assert moved.sum() > SLICE // 2 and (~moved).sum() > 10**4


def test_key_ignores_words_outside_the_key(hb):
    rng = np.random.default_rng(77)
    recs = _key_records(0, 1 << 20)[rng.permutation(1 << 20)]
    dirty = recs.copy()
    dirty[:, 22] |= rng.integers(0, 16, size=len(recs), dtype=np.uint64).astype(np.uint32) << 28
    dirty[:, 23:32] = rng.integers(0, 2**32, size=(len(recs), 9), dtype=np.uint64).astype(np.uint32)
    for mode in (pk.KEY_EXACT, pk.KEY_REFERENCE):
        assert np.array_equal(_gpu_hash(hb, dirty, mode), _gpu_hash(hb, recs, mode))
        flipped = recs.copy()                                       # one bit inside the key changes it
        flipped[:, 21] ^= np.uint32(1) << rng.integers(0, 32, size=len(recs), dtype=np.uint64).astype(np.uint32)
        assert (_gpu_hash(hb, flipped, mode) != _gpu_hash(hb, recs, mode)).all()


# ---- 7. legal masks and random actions ----------------------------------------------------------------------------------
def _rotation_boards():
    """board i holds STACKS[(i + h) % 259] on hex h: every stack on every hex once over the 259 boards"""
    return np.array([_stack_planes([VALID], [STACKS[(i + h) % 259] for h in range(23)])[0] for i in range(259)])


def _place_boards():
    """the rotation boards, and the same boards with about three hexes in four emptied (many legal placements)"""
    rot = _rotation_boards()
    thin = np.array([sum(1 << h for h in range(23) if (5 * h + i) % 4 == 0) for i in range(259)], dtype=np.uint32)
    return np.concatenate([rot, rot & thin[:, None]])


def _place_records():
    """518 boards x all 4,096 hand codes, the mover's board one of them, the other player's board another; phases
    place_tile_1..3 and the player by record"""
    boards = _place_boards()
    nb = len(boards)
    n = nb * 4096
    idx = np.arange(n)
    bi, hand = idx // 4096, (idx % 4096).astype(np.uint32)
    player = (idx // 3) % 2
    recs = _records(n)
    mover, other = boards[bi], boards[(bi + 101) % nb]
    recs[:, 0:9] = np.where(player[:, None] == 0, mover, other)
    recs[:, 9:18] = np.where(player[:, None] == 0, other, mover)
    recs[:, pk.W_PILES01] = 0x0015_0101
    recs[:, pk.W_PILES23] = 0x0540_0090
    recs[:, pk.W_PILE4H] = hand << 16 | 0x0111
    recs[:, pk.W_BAG0] = 0x05060708
    _set_meta(recs, player, 1 + idx % 3, 3 + idx % 3)
    _set_keys(recs, np.random.default_rng(5))
    return recs, bi, hand


def _tiles(hand):
    return sum((np.asarray(hand, dtype=np.int64) >> (2 * t)) & 3 for t in range(6))


@pytest.fixture(scope="module")
def place_set(orc):
    return _place_set(orc)


def _place_set(orc):
    """records, and the legal masks they must have: the union over the types in hand of the oracle's mask for a hand
    of that one type (the oracle's hand holds at most three tiles; the kernels take any 2-bit counts)"""
    recs, bi, hand = _place_records()
    boards = _place_boards()
    single = _records(len(boards) * 6)
    single[:, 0:9] = np.repeat(boards, 6, axis=0)
    single[:, pk.W_PILE4H] = (np.uint32(1) << (2 * np.tile(np.arange(6, dtype=np.uint32), len(boards)))) << 16
    _set_meta(single, 0, 1)
    type_masks = orc.legal_mask(single).reshape(len(boards), 6, 5)
    want = np.zeros((len(recs), 5), dtype=np.uint32)
    for t in range(6):
        has = ((hand >> (2 * t)) & 3) != 0
        want |= np.where(has[:, None], type_masks[bi, t], 0).astype(np.uint32)
    small = _tiles(hand) <= 3                                     # hands the oracle holds as they are
    return recs, want, small


def _want_random(recs, want):
    """the uniform policy's action from the masks: the k-th legal action, k = (rand >> 32) * n >> 32"""
    key = (recs[:, pk.W_KEYLO].astype(np.uint64) | (recs[:, pk.W_KEYHI].astype(np.uint64) << np.uint64(32))) ^ \
        np.uint64(pk.PLAYOUT_SALT)
    r = _mix(key ^ _mix(recs[:, pk.W_MOVES].astype(np.uint64) + np.uint64(0x9E3779B97F4A7C15)))
    n = _popc(want).sum(axis=1)
    k = (((r >> np.uint64(32)) * n.astype(np.uint64)) >> np.uint64(32)).astype(np.int64)
    act = np.full(len(recs), -1, dtype=np.int64)
    below = np.zeros(len(recs), dtype=np.int64)
    for w in range(5):                                            # the word holding the k-th set bit, then the bit
        c = _popc(want[:, w])
        here = (act < 0) & (k < below + c) & (n > 0)
        bits = ((want[:, w, None] >> np.arange(32, dtype=np.uint32)) & np.uint32(1)).astype(np.int16)
        cum = np.cumsum(bits, axis=1, dtype=np.int16)
        pos = np.argmax(cum > (k - below)[:, None], axis=1)
        act = np.where(here, 32 * w + pos, act)
        below += c
    return act


def _mix(z):
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def test_legal_masks_and_random_actions_every_stack_and_hand(hb, orc, place_set):
    recs, want, small = place_set
    assert len(recs) == 2 * 259 * 4096 == 2_121_728 and small.sum() == 2 * 259 * 84
    st = hb.states_from_numpy(recs)
    got = hb.legal_mask(st).cpu().numpy().view(np.uint32)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), recs[bad[0]].tolist(), got[bad[0]].tolist(), want[bad[0]].tolist())
    assert np.array_equal(orc.legal_mask(recs[small]), want[small])
    act = hb.random_actions(st).cpu().numpy().astype(np.int64)
    assert np.array_equal(act, _want_random(recs, want))
    assert np.array_equal(act[small], _pool_map(orc.random_actions, recs[small]).astype(np.int64))
    n = _popc(want).sum(axis=1)
    assert (n == 0).any() and n.max() >= 60 and len(np.unique(act)) == 143 - 5 + 1   # every placement, and none


def test_choose_and_over_phases(hb, orc):
    """0-5 piles in the choose phase (every key and move counter picks its own pile), and game_over"""
    rng = np.random.default_rng(11)
    boards = _rotation_boards()
    recs = _records(6 * 4096 + 512)
    recs[:, 0:9] = boards[rng.integers(0, 259, size=len(recs))]
    recs[:, 9:18] = boards[rng.integers(0, 259, size=len(recs))]
    recs[:, pk.W_PILE4H] = rng.integers(0, 4096, size=len(recs), dtype=np.uint64).astype(np.uint32) << 16
    _set_keys(recs, rng)
    n_piles = np.arange(len(recs)) % 6
    phase = np.where(np.arange(len(recs)) < 6 * 4096, 0, 4)
    _set_meta(recs, rng.integers(0, 2, size=len(recs)), phase, n_piles)
    assert len(recs) == 25_088
    st = hb.states_from_numpy(recs)
    assert np.array_equal(hb.legal_mask(st).cpu().numpy().view(np.uint32), orc.legal_mask(recs))
    act = hb.random_actions(st).cpu().numpy()
    assert np.array_equal(act, orc.random_actions(recs))
    for p in range(1, 6):                                          # every pile is picked
        assert set(act[(phase == 0) & (n_piles == p)].tolist()) == set(range(p))


@pytest.mark.parametrize("n", [1, 31, 32, 33, 127, 129, 4097])
def test_legal_mask_row_counts_and_output_views(hb, place_set, n):
    """rows past n stay untouched in a sentinel-filled buffer; words 23..31 of a record do not change its mask"""
    recs, want, _ = place_set
    rng = np.random.default_rng(n)
    pick = rng.choice(len(recs), size=n, replace=False)
    r = recs[pick].copy()
    r[:, 23:32] = rng.integers(0, 2**32, size=(n, 9), dtype=np.uint64).astype(np.uint32)
    buf = torch.full((n + 70, 5), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    out = buf[3: 3 + n]
    assert out.is_contiguous() and out.data_ptr() != buf.data_ptr()
    hb.legal_mask(hb.states_from_numpy(r), out=out)
    b = buf.cpu().numpy().view(np.uint32)
    assert np.array_equal(b[3: 3 + n], want[pick])
    assert (b[:3] == 0x5A5A5A5A).all() and (b[3 + n:] == 0x5A5A5A5A).all()


# ---- 8. greedy ---------------------------------------------------------------------------------------------------------
def _sparse_records(rng, n):
    """boards with 0-12 tiles (random stacks) and hands of three distinct types: 33-69 legal placements, many ties"""
    recs = _records(n)
    rot = _rotation_boards()
    for i in range(n):
        stacks = [()] * 23
        for h in rng.choice(23, size=int(rng.integers(0, 13) if i % 3 else rng.integers(0, 2)), replace=False):
            stacks[int(h)] = STACKS[int(rng.integers(1, 259))]
        p = i % 2
        recs[i, 9 * p: 9 * p + 9] = _stack_planes([VALID], stacks)[0]
        recs[i, 9 * (1 - p): 9 * (1 - p) + 9] = rot[i % 259] if i % 7 == 0 else 0
        types = rng.choice(6, size=3 if i % 4 else 2, replace=False)
        recs[i, pk.W_PILE4H] = int(sum(1 << (2 * int(t)) for t in types)) << 16
        _set_meta(recs[i: i + 1], p, 1 + i % 3)
    return recs


def _tie_records():
    """every placement scores the same, so the first legal action must win: empty boards and hands that score
    nothing alone (wood, building at height 1, an isolated field)"""
    recs = _records(4)
    hands = [0x410, 0x510, 0x500, 0x110]                           # {wood, field}, {wood, building, field}, ...
    for i, hand in enumerate(hands):
        recs[i, pk.W_PILE4H] = hand << 16
        p = i % 2
        recs[i, 9 * (1 - p): 9 * (1 - p) + 9] = _stack_planes([VALID], [(WATER,)] * 23)[0]
        _set_meta(recs[i: i + 1], p, 1 + i % 3)
    return recs


def _placement_scores(orc, recs):
    """per record, the mover's score after each legal action in ascending order, by oracle.apply + oracle.score"""
    masks = orc.legal_mask(recs)
    acts = [pk.mask_to_actions(m) for m in masks]
    rows = np.repeat(np.arange(len(recs)), [len(a) for a in acts])
    flat = np.concatenate([np.asarray(a, dtype=np.int16) for a in acts])
    after, status = orc.apply(recs[rows], flat)
    assert (status == 0).all()
    sc, _ = orc.score(after)
    mover = (recs[rows, pk.W_BAG1META] >> 24) & 1
    per = np.split(sc[np.arange(len(rows)), mover].astype(np.int64), np.cumsum([len(a) for a in acts])[:-1])
    return acts, per


def test_greedy_against_the_oracle(hb, orc, neighbourhoods, place_set):
    rng = np.random.default_rng(29)
    parts = []
    s4 = _every_stack_records()[rng.choice(5_957, size=3000, replace=False)]
    s5 = neighbourhoods[0][rng.choice(906_059, size=20_000, replace=False)]
    for s in (s4, s5):                                             # the scoring records' boards, player 0 or 1 to place
        r = s.copy()
        r[:, pk.W_PILE4H] = np.array([sum(1 << (2 * int(t)) for t in rng.choice(6, size=int(rng.integers(1, 4))))
                                      for _ in range(len(r))], dtype=np.uint32) << 16
        _set_meta(r, rng.integers(0, 2, size=len(r)), rng.integers(1, 4, size=len(r)))
        parts.append(r)
    recs7, _, small = place_set                                    # hands the oracle holds: <= 3 tiles
    parts.append(recs7[rng.choice(np.nonzero(small)[0], size=20_000, replace=False)])
    sparse = _sparse_records(rng, 1200)
    ties = _tie_records()
    parts += [sparse, ties]
    recs = np.concatenate(parts)
    assert len(recs) == 3_000 + 20_000 + 20_000 + 1_200 + 4 == 44_204
    got = hb.greedy_actions(hb.states_from_numpy(recs)).cpu().numpy()
    want = _pool_map(orc.greedy_actions, recs)
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, (len(bad), recs[bad[0]].tolist(), int(got[bad[0]]), int(want[bad[0]]))
    n_legal = _popc(orc.legal_mask(recs)).sum(axis=1)
    assert ((n_legal > 32) & (n_legal <= 64)).sum() >= 100 and (n_legal > 64).sum() >= 100

    # the designed sets, action by action: the first maximum wins, with ties on different lanes and loop rounds
    acts, per = _placement_scores(orc, np.concatenate([sparse, ties]))
    first = np.array([a[int(np.argmax(s))] if len(a) else -1 for a, s in zip(acts, per)])
    assert np.array_equal(got[-len(first):], first)
    lanes = rounds = 0
    for s in per:
        k = np.nonzero(s == s.max())[0] if len(s) else []
        if len(k) > 1:
            lanes += len({int(x) % 32 for x in k}) > 1
            rounds += len({int(x) // 32 for x in k}) > 1
    assert lanes > 100 and rounds > 100
    tie_scores = per[-len(ties):]
    assert all(len(s) > 32 and (s == s[0]).all() for s in tie_scores)
    assert all(len(s) > 64 for s in tie_scores[1:2])
