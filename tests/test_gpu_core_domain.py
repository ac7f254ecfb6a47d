"""GPU: the fused playout's bit-sliced building blocks (csrc/hz_core.cuh) over their whole input ranges, and the edges
of those ranges through the public entry points.

Games drawn by random play never go near the edges these primitives are written for: bag totals past 127 (a record
may carry up to 255 tiles of each type), every hand code, boards with no or one legal hex, move and event counters at
the rand table's end and at the 32-bit wrap, and a block's water queue overflowing at the final scoring.  So:

- tests/probe_core.cu runs nth_set_bit, bag_total / draw_pile / draw_pile3, place_random and playout_round directly,
  next to naive references that are themselves checked against the host specification (packed.draw_pile, the
  oracle's legal set and random action);
- hz_playout and hz_tree_rollout_eval play records with those counters, and records whose last placement scores many
  large rivers in full 64-game blocks, against the C oracle.
"""

import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest
import torch

from harmonies_alphazero_b200 import packed as pk
from harmonies_alphazero_b200.constants import NEIGHBOR_MASKS

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
INIT_BAG = [23, 19, 21, 23, 15, 19]
N_RECS, REC_WORDS = 16, 32


# ---- fixtures --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    """tests/probe_core.cu built with the library's flags (and HZ_NVCC_EXTRA, so a -DHZ_DEBUG_BOUNDS run covers it)"""
    from harmonies_alphazero_b200 import build

    so = str(tmp_path_factory.mktemp("probe") / "probe_core.so")
    extra = os.environ.get("HZ_NVCC_EXTRA", "").split()
    cmd = [build._nvcc()] + build.NVCC_FLAGS + extra + ["-shared", "-o", so, os.path.join(HERE, "probe_core.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    torch.cuda.init()
    return C.CDLL(so)


@pytest.fixture(scope="module")
def hb():
    from harmonies_alphazero_b200 import batched

    batched._lib.load()
    return batched


def _call(fn, *args):
    """fn(*args) with torch tensors passed as device pointers: args holds them until fn has returned"""
    return fn(*(C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args))


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _u64(a):
    return _cuda(np.asarray(a, dtype=np.uint64).view(np.int64))


def _u32(a):
    return _cuda(np.asarray(a, dtype=np.uint32).view(np.int32))


def _out():
    return torch.zeros(REC_WORDS * (1 + N_RECS), dtype=torch.int32, device="cuda")


def _check(fn, out, what, *args):
    """run a checking launcher; assert no mismatch, printing the first records (word 0: which comparison failed)"""
    assert _call(fn, *args) == 0, f"{what}: CUDA error"
    o = out.cpu().numpy().view(np.uint32)
    n = int(o[0])
    recs = o[REC_WORDS:].reshape(N_RECS, REC_WORDS)[: min(n, N_RECS)]
    for r in recs:
        print(what, [hex(int(x)) for x in r[:12]])
    assert n == 0, f"{what}: {n} mismatches, first ones printed above"


# ---- nth_set_bit ---------------------------------------------------------------------------------------------------
def test_nth_set_bit_every_mask_and_rank(probe):
    """all 2^23 masks, every k < popc(m): 9.6e7 pairs against a bit loop"""
    out = _out()
    _check(probe.probe_nth_sweep, out, "nth_set_bit", out)


def test_nth_reference_is_the_specification(probe):
    rng = np.random.default_rng(1)
    m = rng.integers(1, 1 << 23, size=100_000, dtype=np.uint32)
    pc = np.array([bin(int(x)).count("1") for x in m])
    k = (rng.random(len(m)) * pc).astype(np.int32)
    pos = torch.zeros(len(m), dtype=torch.int32, device="cuda")
    assert _call(probe.probe_ref_nth, _u32(m), _cuda(k), C.c_int64(len(m)), pos) == 0
    want = [[i for i in range(23) if (int(x) >> i) & 1][int(j)] for x, j in zip(m, k)]
    assert pos.cpu().numpy().tolist() == want


# ---- draws ------------------------------------------------------------------------------------------------------
def _bag_word(b):
    return sum(int(c) << (8 * t) for t, c in enumerate(b))


def _draw_list(probe, bags, zs, what):
    out = _out()
    _check(probe.probe_draw_list, out, what, _u64([_bag_word(b) for b in bags]), _u64(zs),
           C.c_int64(len(bags)), out)


def test_draws_every_composition_of_the_initial_bag(probe):
    """bag_total, draw_pile and draw_pile3 on all 8.1e7 bags inside [23, 19, 21, 23, 15, 19], three draws each"""
    out = _out()
    _check(probe.probe_draw_sweep, out, "draw sweep", C.c_uint64(0xD2A5), C.c_int(3), out)


def _boundary_zs(total, rng):
    """for each slot j = 0..2 and each r < total - j: z whose slot j holds the smallest and the largest 21-bit x with
    (x * (total - j)) >> 21 == r, the other slots random"""
    zs = []
    for j in range(3):
        t = total - j
        if t <= 0:
            break
        for r in range(t):
            for x in (-(-(r << 21) // t), -(-((r + 1) << 21) // t) - 1):
                z = int(rng.integers(0, 2**63, dtype=np.uint64)) & ~(0x1FFFFF << (21 * j))
                zs.append(z | (x << (21 * j)))
    return zs


def _family():
    """bags of total <= 6, every one-type bag, the initial bag, and bags of total 121..255"""
    rng = np.random.default_rng(7)
    bags = [b for b in itertools.product(range(7), repeat=6) if sum(b) <= 6]
    bags += [[c if u == t else 0 for u in range(6)] for t in range(6) for c in range(1, 256)]
    bags.append(INIT_BAG)
    for total in range(121, 256):
        for _ in range(2):
            bags.append(rng.multinomial(total, [1 / 6] * 6).tolist())
    return bags


def test_draws_at_every_boundary_of_r(probe):
    rng = np.random.default_rng(3)
    bags, zs = [], []
    for b in _family():
        z = _boundary_zs(sum(b), rng) or [int(rng.integers(0, 2**63, dtype=np.uint64))]
        bags += [b] * len(z)
        zs += z
    _draw_list(probe, bags, zs, "draw boundaries")


def test_draws_from_bags_past_127_tiles(probe):
    """totals 128..1530: up to the 255 per type that pack_fields accepts"""
    rng = np.random.default_rng(5)
    bags = [[100, 50, 0, 0, 0, 0], [23, 19, 21, 23, 15, 28], [255] * 6, [0, 0, 0, 0, 255, 255], [128, 0, 0, 0, 0, 0]]
    bags += rng.integers(0, 256, size=(4000, 6)).tolist()
    bags += [rng.multinomial(int(t), [1 / 6] * 6).tolist() for t in rng.integers(128, 256, size=4000)]
    bags = [b for b in bags if max(b) <= 255 and sum(b) >= 128]
    reps = 64
    zs = rng.integers(0, 2**63, size=len(bags) * reps, dtype=np.uint64) * 2 + rng.integers(0, 2, size=len(bags) * reps, dtype=np.uint64)
    _draw_list(probe, [b for b in bags for _ in range(reps)], zs, "large bags")


def test_draw_reference_is_packed_draw_pile(probe):
    rng = np.random.default_rng(9)
    n = 100_000
    bags = np.concatenate([rng.integers(0, 24, size=(n // 2, 6)), rng.integers(0, 256, size=(n // 2, 6))])
    bags[::17] = 0
    bags[1::17, 1:] = 0
    zs = rng.integers(0, 2**63, size=n, dtype=np.uint64) * 2 + 1
    codes = torch.zeros(n, dtype=torch.int32, device="cuda")
    after = torch.zeros(n, dtype=torch.int64, device="cuda")
    assert _call(probe.probe_ref_draw, _u64([_bag_word(b) for b in bags]), _u64(zs), C.c_int64(n), codes,
                                after) == 0
    codes = codes.cpu().numpy().view(np.uint32)
    after = after.cpu().numpy().view(np.uint64)
    for i in range(n):
        b = bags[i].tolist()
        tiles = pk.draw_pile(b, int(zs[i]))
        assert int(codes[i]) == pk.multiset_code(tiles) and int(after[i]) == _bag_word(b), i


# ---- place_random -------------------------------------------------------------------------------------------------
def _planes(stacks):
    """23 stacks (tuples of type indices, bottom first) -> the 9 planes of a board"""
    p = [0] * 9
    for h, st in enumerate(stacks):
        for level, t in enumerate(st):
            for b in range(3):
                if ((t + 1) >> b) & 1:
                    p[3 * level + b] |= 1 << h
    return p


def _place_boards():
    stacks = [()] + [s for n in (1, 2, 3) for s in itertools.product(range(6), repeat=n)]
    assert len(stacks) == 259
    boards = [_planes([stacks[(i + h) % 259] for h in range(23)]) for i in range(259)]
    rng = np.random.default_rng(13)
    for _ in range(2000):
        heights = rng.choice(4, size=23, p=rng.dirichlet([1, 1, 1, 1]))
        boards.append(_planes([tuple(rng.integers(0, 6, size=int(h)).tolist()) for h in heights]))
    field, wood, full = (5,), (2,), (3, 3, 3)
    for empty in range(23):                                       # one empty hex among fields: one legal hex
        boards.append(_planes([() if h == empty else field for h in range(23)]))
        boards.append(_planes([wood if h == empty else field for h in range(23)]))     # plant / building only
    boards.append(_planes([field] * 23))                          # nothing legal
    boards.append(_planes([full] * 23))
    return np.array(boards, dtype=np.uint32)


def _type_masks(oracle, boards):
    """per board, the six types' legal hex masks: oracle.legal_mask on player 0 in place_tile_1 holding every type (as
    two hands of three: the packed hand holds at most three tiles)"""
    n = len(boards)
    rec = np.zeros((2 * n, 32), dtype=np.uint32)
    rec[:, :9] = np.repeat(boards, 2, axis=0)
    rec[0::2, pk.W_PILE4H] = 0x015 << 16
    rec[1::2, pk.W_PILE4H] = 0x540 << 16
    rec[:, pk.W_BAG1META] = pk.PHASE_INDEX["place_tile_1"] << 25
    lm = oracle.legal_mask(rec)
    masks = np.zeros((n, 6), dtype=np.uint32)
    for i in range(n):
        for half in (0, 1):
            acts = pk.mask_to_actions(lm[2 * i + half])
            for a in acts:
                t, h = divmod(a - 5, 23)
                masks[i, t] |= np.uint32(1 << h)
    return masks


@pytest.fixture(scope="module")
def place_set(oracle):
    boards = _place_boards()
    return boards, _type_masks(oracle, boards)


def test_place_random_every_hand_and_draw_edge(probe, place_set):
    """2,307 gap-free boards x all 4,096 hand codes x both edges of the policy draw for every k < n (n <= 138)"""
    boards, masks = place_set
    out = _out()
    evals = torch.zeros(1, dtype=torch.int64, device="cuda")
    _check(probe.probe_place_sweep, out, "place_random", _u32(boards), _u32(masks), C.c_int(len(boards)),
           out, evals)
    assert int(evals.item()) > 10**8
    assert (np.array([sum(bin(int(x)).count("1") for x in m) for m in masks]) <= 1).sum() >= 40


def test_place_reference_is_the_oracles_random_move(probe, oracle, place_set):
    """the device reference against oracle.random_actions + oracle.apply on 10^5 (board, hand, key, moves)"""
    boards, masks = place_set
    rng = np.random.default_rng(17)
    n = 100_000
    bi = rng.integers(0, len(boards), size=n)
    hands = np.zeros(n, dtype=np.uint32)
    for i, k in enumerate(rng.integers(1, 4, size=n)):
        for t in rng.integers(0, 6, size=k):
            hands[i] += np.uint32(1 << (2 * int(t)))
    rec = np.zeros((n, 32), dtype=np.uint32)
    rec[:, :9] = boards[bi]
    rec[:, pk.W_PILE4H] = hands << 16
    rec[:, pk.W_BAG1META] = 1 << 25                               # player 0, place_tile_1
    keys = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    rec[:, pk.W_KEYLO] = keys & 0xFFFFFFFF
    rec[:, pk.W_KEYHI] = keys >> 32
    rec[:, pk.W_MOVES] = rng.integers(0, 2**32, size=n, dtype=np.uint64).astype(np.uint32)
    rhs = np.array([pk.rand(int(k) ^ pk.PLAYOUT_SALT, int(m)) >> 32 for k, m in zip(keys, rec[:, pk.W_MOVES])], dtype=np.uint32)
    res = torch.zeros((n, 11), dtype=torch.int32, device="cuda")
    assert _call(probe.probe_ref_place, _u32(boards[bi]), _u32(masks[bi]), _u32(hands), _u32(rhs),
                                 C.c_int64(n), res) == 0
    res = res.cpu().numpy().view(np.uint32)
    acts = oracle.random_actions(rec)
    after, status = oracle.apply(rec, acts)
    moved = acts >= 0
    assert moved.mean() > 0.5 and (~moved).any()
    assert (status[moved] == 0).all()
    assert np.array_equal(res[:, :9], after[:, :9])
    assert np.array_equal(res[:, 9], after[:, pk.W_PILE4H] >> 16)
    assert np.array_equal(res[:, 10] != 0, moved)
    assert np.array_equal(res[moved, 10], np.uint32(1) << ((acts[moved] - 5) % 23).astype(np.uint32))


# ---- playout_round ------------------------------------------------------------------------------------------------
def _set_bag(rec, bag):
    rec[pk.W_BAG0] = bag[0] | (bag[1] << 8) | (bag[2] << 16) | (bag[3] << 24)
    rec[pk.W_BAG1META] = (int(rec[pk.W_BAG1META]) & 0xFFFF0000) | bag[4] | (bag[5] << 8)


def _cover_with_fields(rec, player, n, rng):
    for h in rng.choice(23, size=n, replace=False):
        rec[9 * player + 1] |= np.uint32(1 << int(h))
        rec[9 * player + 2] |= np.uint32(1 << int(h))


def test_playout_round_equals_eight_steps(probe, oracle):
    """round starts of real games, with bags of 0..11 and 120..255+ tiles, boards where a placement finds no legal
    hex, and move / event counters up to the largest that round_ready admits (and one past)"""
    rng = np.random.default_rng(23)
    parts = [oracle.playout(oracle.init_states(1024, seed=300 + r), max_steps=8 * r)[0] for r in range(8)]
    base = np.concatenate(parts)
    recs = [base.copy()]
    v = base.copy()                                               # bags around the round's limits
    totals = rng.choice([0, 3, 5, 6, 7, 11, 120, 126, 127, 128, 129, 200, 255, 600, 1530], size=len(v))
    for i, t in enumerate(totals):
        bag = rng.multinomial(int(t), [1 / 6] * 6) if t <= 255 else np.minimum(rng.multinomial(int(t), [1 / 6] * 6), 255)
        _set_bag(v[i], [int(x) for x in bag])
    recs.append(v)
    v = base.copy()                                               # no legal hex at some placement
    for i in range(len(v)):
        _cover_with_fields(v[i], int(rng.integers(0, 2)), int(rng.integers(19, 24)), rng)
    recs.append(v)
    v = base.copy()                                               # counters at the rand table's end
    v[:, pk.W_MOVES] = rng.integers(496, 506, size=len(v))
    v[:, pk.W_EVENT] = rng.integers(56, 64, size=len(v))
    recs.append(v)
    recs = np.concatenate(recs)
    out = _out()
    flags = torch.zeros(len(recs), dtype=torch.int32, device="cuda")
    _check(probe.probe_round, out, "playout_round", _u32(recs), C.c_int64(len(recs)), out, flags)
    f = flags.cpu().numpy()
    ready, ok = (f & 1) != 0, (f & 2) != 0
    meta = recs[:, pk.W_BAG1META] >> 24
    start = ((meta & 0x1F) == 0) & (((recs[:, pk.W_BAG1META] >> 16) & 0xFF) == 5)
    want_ready = start & (recs[:, pk.W_MOVES] <= 504) & (recs[:, pk.W_EVENT] <= 62)
    assert np.array_equal(ready, want_ready)
    total = np.array([sum((int(w) >> (8 * t)) & 0xFF for t in range(4)) + (int(x) & 0xFF) + ((int(x) >> 8) & 0xFF)
                      for w, x in zip(recs[:, pk.W_BAG0], recs[:, pk.W_BAG1META])])
    assert not ok[ready & ((total < 6) | (total > 127))].any()
    assert ok[ready & (total == 6)].any() and ok[ready & (total == 127)].any()
    assert (ready & ~ok & (total >= 6) & (total <= 127)).any()   # a placement without a legal hex
    assert ok[ready & (recs[:, pk.W_MOVES] == 504) & (recs[:, pk.W_EVENT] == 62)].any()


# ---- counters at the rand table's end and at the 32-bit wrap, through the entry points -------------------------
MOVES = [503, 504, 505, 511, 512, 513] + list(range(2**32 - 9, 2**32))
EVENTS = [61, 62, 63, 64, 2**32 - 1]


def _mid_games(oracle, n, seed):
    parts = [oracle.playout(oracle.init_states(n, seed=seed + d), max_steps=d)[0] for d in (0, 6, 31, 52)]
    return np.concatenate(parts)


def _with_counters(games):
    out = []
    for mv, ev in itertools.product(MOVES, EVENTS):
        g = games.copy()
        g[:, pk.W_MOVES] = mv
        g[:, pk.W_EVENT] = ev
        out.append(g)
    return np.concatenate(out)


def _playout_vs_oracle(hb, oracle, init, max_steps):
    st = hb.states_from_numpy(init)
    steps, total = hb.playout(st, max_steps=max_steps)
    ref, rsteps, rtotal = oracle.playout(init, max_steps=max_steps, n_threads=8)
    got = st.cpu().numpy().view(np.uint32)
    bad = np.nonzero((got != ref).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), init[bad[0]].tolist())
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), rsteps)
    assert int(total.item()) == rtotal
    return ref


@pytest.mark.parametrize("max_steps", [1, 8, 9, 1000])
def test_playout_counters_past_the_rand_table_and_at_the_wrap(hb, oracle, max_steps):
    init = _with_counters(_mid_games(oracle, 16, 1000 + max_steps))
    ref = _playout_vs_oracle(hb, oracle, init, max_steps)
    if max_steps == 1000:
        assert (ref[:, pk.W_MOVES] < 512).any() and (ref[:, pk.W_EVENT] < 64).any()   # wrapped back into the table


def _roots_rollout_eval(hb, roots, R, seed):
    from harmonies_alphazero_b200 import tree as tr
    from tests.test_gpu_rollout_eval import _host_rollout_eval

    n = len(roots)
    skeys = np.random.default_rng(seed).integers(0, 2**63, size=n, dtype=np.uint64)
    t = tr.BatchedMCTS(n, 4, key_mode=pk.KEY_EXACT)
    t.reset(hb.states_from_numpy(roots), tr.search_keys_tensor(skeys))
    leaf = torch.empty((n, 32), dtype=torch.int32, device="cuda")
    t.select(2.0, leaf_states=leaf)
    policy = torch.full((n, 143), float("nan"), device="cuda")
    value = torch.full((n,), float("nan"), device="cuda")
    total = torch.zeros(1, dtype=torch.int64, device="cuda")
    t.rollout_eval(policy, value, R, total)
    leaves = leaf.cpu().numpy().view(np.uint32)
    assert np.array_equal(leaves, roots)                          # the unexpanded roots are the leaves
    return leaves, skeys, policy, value, total, _host_rollout_eval


@pytest.mark.parametrize("R", [1, 32, 64])
def test_rollout_eval_roots_with_those_counters(hb, oracle, R):
    roots = _with_counters(_mid_games(oracle, 2, 2000 + R))
    roots = roots[(roots[:, pk.W_BAG1META] >> 25 & 7) != 4]
    leaves, skeys, policy, value, total, host = _roots_rollout_eval(hb, roots, R, R)
    hp, hv, hsteps = host(oracle, leaves, skeys, R)
    assert np.array_equal(policy.cpu().numpy().view(np.uint32), hp.view(np.uint32))
    assert np.array_equal(value.cpu().numpy().view(np.uint32), hv.view(np.uint32))
    assert int(total.item()) == hsteps


# ---- the fused kernels' final scoring with the block's water queue overflowing -----------------------------------
def _components(mask):
    comps, rem = [], mask
    while rem:
        comp = rem & -rem
        while True:
            grow = comp
            for h in range(23):
                if (comp >> h) & 1:
                    grow |= NEIGHBOR_MASKS[h] & rem
            if grow == comp:
                break
            comp = grow
        comps.append(comp)
        rem &= ~comp
    return comps


def _rivers(rng, max_size, tries):
    """a water mask of up to four separate rivers of >= 5 hexes (sizes up to max_size), not touching each other: the
    one of `tries` random attempts with the most of them"""
    best = 0
    for _ in range(tries):
        water, banned = 0, 0
        for _ in range(4):
            free = [h for h in range(23) if not ((water | banned) >> h) & 1]
            if not free:
                break
            comp = 1 << int(rng.choice(free))
            size = int(rng.integers(5, max_size + 1))
            while bin(comp).count("1") < size:
                grow = [h for h in range(23) if not ((comp | water | banned) >> h) & 1
                        and NEIGHBOR_MASKS[h] & comp]
                if not grow:
                    break
                comp |= 1 << int(rng.choice(grow))
            if bin(comp).count("1") < 5:
                break
            water |= comp
            for h in range(23):
                if (comp >> h) & 1:
                    banned |= NEIGHBOR_MASKS[h]
        if sum(bin(c).count("1") >= 5 for c in _components(water)) > sum(bin(c).count("1") >= 5 for c in _components(best)):
            best = water
    return best


OTHER_STACKS = [(5,), (3,), (3, 3), (2, 1), (2, 4), (3, 4), (1,)]   # field, stone, mountain, tree, buildings, plant


def _endgame_records(n, seed):
    """player 1 to place the last tile of the game (the ending flag is set): both boards full of rivers of >= 5 hexes,
    the other hexes other tiles, player 1's board with free hexes for the last tile"""
    rng = np.random.default_rng(seed)
    recs = np.zeros((n, 32), dtype=np.uint32)
    for i in range(n):
        for p in (0, 1):
            water = _rivers(rng, 21, 1) if i % 8 == 0 else _rivers(rng, 9, 40)
            stacks = []
            free = set(rng.choice([h for h in range(23) if not (water >> h) & 1], size=2, replace=False).tolist()) if p else set()
            for h in range(23):
                if (water >> h) & 1:
                    stacks.append((0,) if rng.random() < 0.7 else (2, 0) if rng.random() < 0.5 else (3, 3, 0))
                elif h in free:
                    stacks.append(())
                else:
                    stacks.append(OTHER_STACKS[rng.choice(len(OTHER_STACKS), p=[.3, .15, .1, .15, .1, .1, .1])])
            recs[i, 9 * p: 9 * p + 9] = _planes(stacks)
        hand = 1 << (2 * int(rng.choice([0, 0, 1, 5])))
        recs[i, pk.W_PILES01] = 0x15 | (0x90 << 16)
        recs[i, pk.W_PILES23] = 0x111 | (0x501 << 16)
        recs[i, pk.W_PILE4H] = hand << 16
        _set_bag(recs[i], [int(x) for x in rng.integers(0, 6, size=6)])
        recs[i, pk.W_BAG1META] |= (4 << 16) | ((1 | (3 << 1) | (1 << 4)) << 24)   # 4 piles; player 1, place_tile_3, ending
        key = int(rng.integers(0, 2**63, dtype=np.uint64))
        recs[i, pk.W_KEYLO], recs[i, pk.W_KEYHI] = key & 0xFFFFFFFF, key >> 32
        recs[i, pk.W_EVENT] = int(rng.integers(20, 40))
        recs[i, pk.W_MOVES] = int(rng.integers(150, 250))
    return recs


def _water_top(rec, p):
    b = [int(x) for x in rec[9 * p: 9 * p + 9]]
    occ1, occ2 = b[3] | b[4] | b[5], b[6] | b[7] | b[8]
    t0 = b[6] | (b[3] & ~occ2) | (b[0] & ~occ1)
    t1 = b[7] | (b[4] & ~occ2) | (b[1] & ~occ1)
    t2 = b[8] | (b[5] & ~occ2) | (b[2] & ~occ1)
    return t0 & ~t1 & ~t2 & 0x7FFFFF


def _large_rivers(rec):
    """water components of >= 5 hexes on both boards: what score_board pushes to the block's queue"""
    return sum(bin(c).count("1") >= 5 for p in (0, 1) for c in _components(_water_top(rec, p)))


@pytest.fixture(scope="module")
def endgames():
    return _endgame_records(64 * 6, 41)


@pytest.mark.parametrize("max_steps", [1, 1000])
def test_playout_final_scoring_overflows_the_water_queue(hb, oracle, endgames, max_steps):
    ref = _playout_vs_oracle(hb, oracle, endgames, max_steps)
    over, _ = oracle.outcome(ref)
    assert over.all()
    sc, _ = oracle.score(ref)
    assert np.array_equal(ref[:, pk.W_SCORES], (sc[:, 0].astype(np.uint32) & 0xFFFF) | ((sc[:, 1].astype(np.uint32) & 0xFFFF) << 16))
    pushes = np.array([_large_rivers(r) for r in ref]).reshape(-1, 64).sum(axis=1)
    assert (pushes > 128).all(), pushes                          # k_playout's queue: WaterQueue<128, 128> per 64 games
    sizes = [bin(c).count("1") for r in ref for p in (0, 1) for c in _components(_water_top(r, p))]
    assert max(sizes) >= 15


def test_rollout_eval_final_scoring_overflows_the_water_queue(hb, oracle, endgames):
    roots = np.array([r for r in endgames if _large_rivers(r) >= 4][:24])
    leaves, skeys, policy, value, total, host = _roots_rollout_eval(hb, roots, 64, 5)
    hp, hv, hsteps = host(oracle, leaves, skeys, 64)
    assert np.array_equal(policy.cpu().numpy().view(np.uint32), hp.view(np.uint32))
    assert np.array_equal(value.cpu().numpy().view(np.uint32), hv.view(np.uint32))
    assert int(total.item()) == hsteps == 64 * len(roots)
    # one root's 64 rollouts share a block, and each pushes the rivers of both final boards: the last tile joins two
    # rivers at most
    assert len(roots) == 24 and all((_large_rivers(r) - 1) * 64 > 128 for r in roots)


# ---- the object API with bags past 127 tiles -----------------------------------------------------------------------
@pytest.mark.parametrize("bag", [[23, 19, 21, 23, 15, 28], [100, 50, 0, 0, 0, 50]])
def test_object_api_draws_from_large_bags(oracle, bag):
    from harmonies_alphazero_b200 import harmonies_engine as eng

    eng._dev().device()
    bag_d = dict(zip(eng.TILE_TYPES, bag))
    key = 0x1234_5678_9ABC_DEF1
    base = {"player_boards": [{}, {}], "tile_bag": dict(bag_d), "available_piles": [["water"], ["plant", "wood"]],
            "current_player": 0, "tiles_in_hand": ["stone"], "turn_phase": "place_tile_3", "game_over": False,
            "winner": None, "final_scores": [0, 0], "_rng_key": key, "_rng_event": 7, "_moves": 30}

    def spec(counts, event, n_draws):
        """pk.draw_pile's tiles for draw event `event`: draw k of the event uses z = rand(key, event * 8 + k)"""
        out = []
        for k in range(n_draws):
            out.append(pk.draw_pile(counts, pk.rand(key, event * 8 + k)))
        return out

    s = eng.HarmoniesGameState(dict(base, tile_bag=dict(bag_d)))
    tiles = s._draw_tiles(12)
    counts = list(bag)
    want = [t for p in spec(counts, 7, 4) for t in p]
    assert tiles == [eng.TILE_TYPES[t] for t in want]
    assert [s.tile_bag[t] for t in eng.TILE_TYPES] == counts

    s = eng.HarmoniesGameState(dict(base, tile_bag=dict(bag_d)))
    s._replenish_piles()
    counts = list(bag)
    piles = spec(counts, 7, 3)
    assert [sorted(p) for p in s.available_piles[2:]] == [sorted(eng.TILE_TYPES[t] for t in p) for p in piles]
    assert [s.tile_bag[t] for t in eng.TILE_TYPES] == counts

    s = eng.HarmoniesGameState(dict(base, tile_bag=dict(bag_d)))
    n = s.apply_move(("stone", (0, 0)))
    ref, status = oracle.apply(s._pack()[None], np.array([5 + 23 * 3 + pk.coordinate_to_index_map[(0, 0)]], dtype=np.int16))
    assert status[0] == 0
    assert np.array_equal(n._pack(), ref[0])
    counts = list(bag)
    piles = spec(counts, 7, 3)
    assert [sorted(p) for p in n.available_piles[2:]] == [sorted(eng.TILE_TYPES[t] for t in p) for p in piles]
    assert n.current_player == 1 and [n.tile_bag[t] for t in eng.TILE_TYPES] == counts
