"""The fused playout's round path (playout_round: a whole round of eight actions per loop iteration, both players'
placements interleaved) against the C oracle, which plays one action at a time.

The kernel takes a round whole only from (player 0, choose, not ending, 5 piles) when 8 more actions fit in
max_steps, and falls back to single steps for anything irregular (no legal hex, a top-up from a bag of fewer than
three tiles).  These cases put rounds at every cut-off and start offset and force each fallback."""

import numpy as np
import pytest
import torch

from tests.conftest import load_golden

pytestmark = pytest.mark.gpu

W_BAG0, W_BAG1META, W_MOVES = 21, 22, 27


@pytest.fixture(scope="module")
def hb():
    from harmonies_alphazero_b200 import batched

    batched._lib.load()
    return batched


def host(states):
    return states.cpu().numpy().view(np.uint32)


def check_vs_oracle(hb, oracle, init, max_steps=1000):
    st = hb.states_from_numpy(init)
    steps, total = hb.playout(st, max_steps=max_steps)
    ref, rsteps, rtotal = oracle.playout(init, max_steps=max_steps, n_threads=8)
    assert np.array_equal(host(st), ref)
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), rsteps)
    assert int(total.item()) == rtotal
    return rsteps


@pytest.mark.parametrize("max_steps", list(range(1, 18)) + list(range(63, 74)))
def test_rounds_cut_by_max_steps(hb, oracle, max_steps):
    init = oracle.init_states(2048, seed=900 + max_steps)
    check_vs_oracle(hb, oracle, init, max_steps)


@pytest.mark.parametrize("offset", range(8))
def test_starts_inside_a_round(hb, oracle, offset):
    """games `offset` actions into their first, fourth and seventh round (advanced by the oracle), played to the end"""
    parts = []
    for r in (0, 3, 6):
        fresh = oracle.init_states(1024, seed=40 + 8 * r + offset)
        parts.append(oracle.playout(fresh, max_steps=8 * r + offset)[0])
    init = np.concatenate(parts)
    assert (init[:, W_MOVES] % 8 == offset).all()
    check_vs_oracle(hb, oracle, init)


def test_nearly_empty_bags(hb, oracle):
    """bags of 0..11 tiles: top-ups of fewer than three tiles, partial piles, the bag running out mid-game"""
    rng = np.random.default_rng(3)
    init = oracle.init_states(4096, seed=5)
    for i in range(len(init)):
        counts = np.zeros(6, dtype=np.uint32)
        for t in rng.integers(0, 6, size=i % 12):
            counts[t] += 1
        init[i, W_BAG0] = counts[0] | (counts[1] << 8) | (counts[2] << 16) | (counts[3] << 24)
        init[i, W_BAG1META] = (init[i, W_BAG1META] & 0xFFFF0000) | counts[4] | (counts[5] << 8)
    steps = check_vs_oracle(hb, oracle, init)
    assert len(set(steps.tolist())) > 3


def fields(init, player, n_occupied, rng):
    """n_occupied[i] random hexes of game i's board `player` covered by a field (code 6: nothing stacks on it)"""
    for i, m in enumerate(n_occupied):
        mask = 0
        for h in rng.choice(23, size=int(m), replace=False):
            mask |= 1 << int(h)
        init[i, 9 * player + 1] |= mask
        init[i, 9 * player + 2] |= mask


def test_near_full_boards_and_no_legal_hex(hb, oracle):
    """boards with 15..23 hexes taken: player 0 ends a turn with <= 2 empty hexes (the game ends after player 1's
    turn), player 1 does, or a player has no legal hex at the first, second or third placement of a round (player 1's:
    after player 0's three placements of the same round went through)"""
    rng = np.random.default_rng(11)
    n = 4096
    init = oracle.init_states(n, seed=17)
    fields(init, 0, rng.integers(15, 24, size=n), rng)
    fields(init, 1, rng.integers(0, 24, size=n), rng)
    steps = check_vs_oracle(hb, oracle, init)
    assert (steps % 8 != 0).any() and (steps % 8 == 0).any()
    # player 0 free, player 1 blocked at some point of the first round
    init = oracle.init_states(n, seed=18)
    fields(init, 1, rng.integers(20, 24, size=n), rng)
    steps = check_vs_oracle(hb, oracle, init)
    assert ((steps > 4) & (steps < 8)).any()


@pytest.mark.parametrize("which", ["states", "after"])
def test_weird_goldens_to_the_end(hb, oracle, which):
    """the reference's non-standard states (ragged piles, leftover hands, nearly empty bags, stray flags)"""
    init = np.ascontiguousarray(load_golden("weird")[which].view(np.uint32))
    check_vs_oracle(hb, oracle, init)


def test_playout_keys_equals_playout(hb):
    n = 20000
    keys = torch.randint(0, 2**62, (n,), dtype=torch.int64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    res, total = hb.playout_keys(keys)
    st = hb.init_states(n, keys=keys.cpu().numpy().view(np.uint64))
    steps, total2 = hb.playout(st)
    w = host(st)
    r = res.cpu().numpy().view(np.uint32)
    assert np.array_equal(r[:, 0], w[:, W_BAG1META])
    assert np.array_equal(r[:, 1], w[:, 23])
    assert np.array_equal(r[:, 2], w[:, W_MOVES])
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), w[:, W_MOVES])
    assert int(total.item()) == int(total2.item())
