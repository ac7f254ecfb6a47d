"""The fused playout's placement pick (place_random: the legal-set counts, the type covering the draw, the k-th legal hex
of that type) against the C oracle on synthetic mid-turn records.

Hands hold one to three tile types with repeats; boards carry random gap-free stacks up to height three, so that the
stacking sets of plants (on wood), stones (on stone) and buildings (on a height-1 wood, stone or building) are non-empty
next to the empty hexes; some boards leave a single legal hex.  max_steps = 1, 2 and 3 compare every placement of the
turn on its own; then the records are played to the end."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W_PILE4H, W_BAG1META = 20, 22
N = 8192


@pytest.fixture(scope="module")
def hb():
    from harmonies_alphazero_b200 import batched

    batched._lib.load()
    return batched


def stack(board, hex_, codes):
    """tiles `codes` (bottom first) on hex_ of a 9-word board"""
    for level, code in enumerate(codes):
        for q in range(3):
            if (code >> q) & 1:
                board[3 * level + q] |= 1 << hex_


def mid_turn_records(oracle, seed):
    rng = np.random.default_rng(seed)
    init = oracle.init_states(N, seed=seed)
    for i in range(N):
        player, phase = int(rng.integers(0, 2)), int(rng.integers(1, 4))
        for p in range(2):
            board = np.zeros(9, dtype=np.uint32)
            if i % 8 == 7:
                # one legal hex at most: every other hex under a field (nothing stacks on it), the last one empty or a
                # wood / stone / building of height 1
                last = int(rng.integers(0, 23))
                for h in range(23):
                    stack(board, h, [6] if h != last else [int(c) for c in rng.choice([3, 4, 5], size=int(rng.integers(0, 2)))])
            else:
                for h in range(23):
                    height = int(rng.choice(4, p=[0.35, 0.3, 0.2, 0.15]))
                    stack(board, h, [int(c) for c in rng.choice([3, 4, 5, 2, 1, 6], size=height, p=[.3, .3, .2, .1, .05, .05])])
            init[i, 9 * p:9 * p + 9] = board
        # the tiles left for the turn (three on every fourth record), from all six types or, on every third record, from
        # the three that stack
        types = rng.choice([1, 3, 4] if i % 3 == 0 else 6, size=3 if i % 4 == 0 else 4 - phase)
        hand = sum(1 << (2 * int(t)) for t in types)   # two-bit counts, at most 3 of a type
        init[i, W_PILE4H] = (init[i, W_PILE4H] & 0xFFFF) | (hand << 16)
        init[i, W_BAG1META] = (init[i, W_BAG1META] & 0x00FFFFFF) | ((player | (phase << 1)) << 24)
    return init


def check_vs_oracle(hb, oracle, init, max_steps):
    st = hb.states_from_numpy(init)
    steps, total = hb.playout(st, max_steps=max_steps)
    ref, rsteps, rtotal = oracle.playout(init, max_steps=max_steps, n_threads=8)
    assert np.array_equal(st.cpu().numpy().view(np.uint32), ref)
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), rsteps)
    assert int(total.item()) == rtotal
    return rsteps


@pytest.mark.parametrize("max_steps", [1, 2, 3, 1000])
def test_mid_turn_picks(hb, oracle, max_steps):
    init = mid_turn_records(oracle, seed=70 + max_steps % 7)
    steps = check_vs_oracle(hb, oracle, init, max_steps)
    assert (steps == min(max_steps, 3)).any() and (steps < min(max_steps, 3)).any()   # full turns and stuck placements
