"""GPU: the object-level drop-in API (harmonies_engine / process_game_state / MCTS modules of
this package) — the same cases as the reference's tests/test_harmonies_engine.py (value
semantics of apply_move, phase/pile/hand bookkeeping, hash/eq sensitivity), plus the search
entry point and the trainer hook."""

import random
from collections import deque

import numpy as np
import pytest
import torch

from harmonies_alphazero_b200 import packed as pk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from harmonies_alphazero_b200 import harmonies_engine

    harmonies_engine._dev().device()
    return harmonies_engine


# ---- reference tests/test_harmonies_engine.py:5-74 ------------------------------------------
def test_apply_move_returns_new_object_and_keeps_original(eng):
    s = eng.HarmoniesGameState()
    keep = s.clone()
    n = s.apply_move(0)
    assert n is not s
    assert (s.current_player, s.turn_phase, s.tiles_in_hand, len(s.available_piles)) == (
        keep.current_player, keep.turn_phase, keep.tiles_in_hand, len(keep.available_piles))
    assert n.turn_phase == "place_tile_1" and s.turn_phase == "choose_pile" and s.current_player == 0


def test_choose_pile_moves_pile_to_hand_and_leaves_bag_and_boards(eng):
    s = eng.HarmoniesGameState()
    chosen = list(s.available_piles[0])
    bag, b0, b1 = s.tile_bag.copy(), s.player_boards[0].copy(), s.player_boards[1].copy()
    n = s.apply_move(0)
    assert len(n.available_piles) == len(s.available_piles) - 1 == 4
    assert len(n.tiles_in_hand) == eng.PILE_SIZE and sorted(n.tiles_in_hand) == sorted(chosen)
    assert len(s.available_piles) == 5 and s.tiles_in_hand == []
    assert n.tile_bag == bag and n.player_boards[0] == b0 and n.player_boards[1] == b1
    assert sum(n.tile_bag.values()) == 120 - 15


# ---- reference tests/test_harmonies_engine.py:76-169 ------------------------------------------
def test_hash_and_eq_follow_every_field(eng):
    s1 = eng.HarmoniesGameState()
    s2 = s1.clone()
    assert s1 == s2 and hash(s1) == hash(s2)
    for mutate in (
        lambda s: setattr(s, "current_player", 1 - s.current_player),
        lambda s: setattr(s, "turn_phase", "place_tile_1"),
        lambda s: setattr(s, "tiles_in_hand", ["water"]),
        lambda s: setattr(s, "available_piles", [["a", "b", "c"]]),     # arbitrary names, as the reference test
        lambda s: s.tile_bag.__setitem__("water", s.tile_bag["water"] - 1),
        lambda s: s.player_boards[0].__setitem__((0, 0), ["water"]),
    ):
        t = s1.clone()
        mutate(t)
        assert t != s1 and hash(t) != hash(s1)
    a, b = s1.clone(), s1.clone()
    a.player_boards[0][(0, 0)] = ["water"]
    b.player_boards[0][(0, 0)] = ["stone"]
    assert a != b and hash(a) != hash(b)
    assert (s1 == 5) is False


# ---- behaviour of the rules through the object API vs the oracle ---------------------------
def test_full_game_through_object_api_matches_oracle(eng, oracle):
    random.seed(7)
    s = eng.HarmoniesGameState()
    w = s._pack()
    steps = 0
    while not s.is_game_over():
        moves = s.get_legal_moves()
        acts = pk.mask_to_actions(oracle.legal_mask(w[None])[0])
        assert [pk.action_to_move(a) for a in acts] == moves and moves
        assert s.get_game_outcome() is None
        mv = moves[random.randrange(len(moves))]
        from harmonies_alphazero_b200.process_game_state import get_action_index

        w2, st = oracle.apply(w[None], [get_action_index(mv)])
        s2 = s.apply_move(mv)
        assert st[0] == 0 and np.array_equal(s2._pack()[:28], w2[0][:28])
        s, w = s2, w2[0]
        steps += 1
    assert 56 <= steps <= 160 and s.turn_phase == "game_over" and s.get_game_outcome() in (1, -1, 0)
    sc = oracle.score(w[None])[0][0]
    assert [s.calculate_score_for_player(0), s.calculate_score_for_player(1)] == sc.tolist() == s.final_scores
    assert s.get_legal_moves() == []                        # :205-208
    with pytest.raises(ValueError):
        s.apply_move(0)                                     # :296


def test_apply_move_value_errors(eng):
    s = eng.HarmoniesGameState()
    for bad in (5, -1, "0", (0, 0), 1.0):
        with pytest.raises(ValueError):
            s.apply_move(bad)                               # :220
    p = s.apply_move(1)
    hand = p.tiles_in_hand
    missing = [t for t in eng.TILE_TYPES if t not in hand][0]
    for bad in (0, ("lava", (0, 0)), (hand[0], (9, 9)), (missing, (0, 0)), [hand[0], (0, 0)]):
        with pytest.raises(ValueError):
            p.apply_move(bad)                               # :234,242,246
    q = eng.HarmoniesGameState(initial_state={
        "player_boards": [{(0, 0): ["water"]}, {}], "tile_bag": {t: 5 for t in eng.TILE_TYPES},
        "available_piles": [], "current_player": 0, "tiles_in_hand": ["water", "plant", "wood"],
        "turn_phase": "place_tile_1", "game_over": False, "winner": None, "final_scores": [0, 0]})
    for t in ("water", "plant", "wood"):
        with pytest.raises(ValueError):
            q.apply_move((t, (0, 0)))                       # :281
    assert q.player_boards[0] == {(0, 0): ["water"]} and q.tiles_in_hand == ["water", "plant", "wood"]


def test_state_tensors_and_action_index(eng, oracle):
    from harmonies_alphazero_b200.process_game_state import create_state_tensors, get_action_index

    random.seed(3)
    s = eng.HarmoniesGameState()
    for _ in range(11):
        m = s.get_legal_moves()
        s = s.apply_move(m[random.randrange(len(m))])
    b, g = create_state_tensors(s)
    assert b.shape == (38, 5, 7) and g.shape == (42,) and b.dtype == g.dtype == torch.float32 and not b.is_cuda
    ob, og = oracle.encode(s._pack()[None])
    assert np.array_equal(b.numpy(), ob[0]) and np.array_equal(g.numpy(), og[0])
    assert get_action_index(3) == 3 and get_action_index(("field", (3, -2))) == 5 + 23 * 5 + 22
    for bad in (5, ("lava", (0, 0)), ("water", (7, 7)), "x"):
        with pytest.raises(ValueError):
            get_action_index(bad)


class _FakeManager:
    """ModelManager.predict stand-in keyed by the state tensors' content (exactly computable)."""

    def __init__(self):
        self.calls = 0

    def predict(self, board, glob):
        self.calls += 1
        assert board.shape == (38, 5, 7) and glob.shape == (42,)
        h = int(board.sum().item() * 1000 + glob.sum().item() * 7919) & 0xFFFFFFFF
        p, v = pk.fake_eval(pk.mix(h))
        return p, v


def test_get_best_action_and_pi_matches_oracle(eng, oracle):
    from harmonies_alphazero_b200 import MCTS
    from harmonies_alphazero_b200.process_game_state import get_action_index

    cfg = {"num_simulations": 30, "cpuct": 2, "dirichlet_alpha": 0.4, "dirichlet_epsilon": 0.25,
           "turns_until_tau0": 15, "action_size": 143, "testing": True}
    random.seed(21)
    s = eng.HarmoniesGameState()
    for move_no in range(6):
        mgr = _FakeManager()
        st = random.getstate()
        mv, pi = MCTS.get_best_action_and_pi(s.clone(), mgr, cfg, move_no)
        random.setstate(st)
        skey = random.getrandbits(64)          # the key the search drew
        assert mgr.calls == 30 and pi.shape == (143,) and pi.dtype == np.float64

        def ev(w):
            b, g = oracle.encode(w[None])
            h = int(torch.from_numpy(b[0]).sum().item() * 1000 + torch.from_numpy(g[0]).sum().item() * 7919) & 0xFFFFFFFF
            return pk.fake_eval(pk.mix(h))

        r = oracle.search(s._pack(), skey, 30, 2.0, eval_fn=ev)
        assert np.abs(pi - r["N"] / r["N"].sum()).max() <= 1e-6
        assert get_action_index(mv) == int(np.argmax(r["N"]))
        s = s.apply_move(mv)
    # exploratory mode samples a visited move; terminal root returns (None, zeros)
    cfg2 = dict(cfg, testing=False)
    mv, pi = MCTS.get_best_action_and_pi(s.clone(), _FakeManager(), cfg2, 0)
    assert pi[get_action_index(mv)] > 0 and abs(pi.sum() - 1) < 1e-9
    while not s.is_game_over():
        m = s.get_legal_moves()
        s = s.apply_move(m[0])
    mv, pi = MCTS.get_best_action_and_pi(s.clone(), _FakeManager(), cfg, 70)
    assert mv is None and pi.sum() == 0


def test_trainer_hook_fills_replay_buffer(eng):
    from harmonies_alphazero_b200 import net, trainer_hooks

    class Manager:
        model = net.AlphaZeroNet.from_config(net.TEST_MODEL_CONFIG)

    class FakeTrainer:
        self_play_config = {"num_games_per_iter": 6}
        mcts_config = {"num_simulations": 5, "cpuct": 1.0, "dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.0,
                       "turns_until_tau0": 0, "action_size": 143, "testing": True}
        replay_buffer = deque(maxlen=10000)

    t = FakeTrainer()
    stats = trainer_hooks.execute_self_play_phase(t, Manager(), n_slots=4)
    assert stats["games"] == 6 and len(t.replay_buffer) == stats["examples"] >= 6 * 56
    b, g, p, z = t.replay_buffer[0]
    assert b.shape == (38, 5, 7) and g.shape == (42,) and p.shape == (143,) and z.shape == (1,)
    assert abs(float(p.sum()) - 1.0) < 1e-5
    one = trainer_hooks.self_play_worker((Manager.model.state_dict(), net.TEST_MODEL_CONFIG, {}, FakeTrainer.mcts_config, "cpu"))
    assert len(one) >= 56 and one[0][0].shape == (38, 5, 7)

    # arena hook (trainer.py:293-431): match + the reference's promotion rule
    calls = []

    class EvalManager:
        def __init__(self, seed):
            torch.manual_seed(seed)
            self.model = net.AlphaZeroNet.from_config(net.TEST_MODEL_CONFIG)

        def save_checkpoint(self, folder, filename, iteration):
            calls.append(("save", folder, filename, iteration))

        def load_checkpoint(self, folder, filename):
            calls.append(("load", folder, filename))

    class EvalTrainer(FakeTrainer):
        self_play_config = {"eval_episodes": 6, "eval_win_rate_threshold": -1.0, "checkpoint_folder": "ckpt", "num_iterations": 9}
        best_model_filename = "best.pth"

    et = EvalTrainer()
    et.model_manager, et.best_model_manager = EvalManager(1), EvalManager(2)
    cfg_eval = {"num_simulations": 6, "cpuct": 1.0, "testing": True}
    res = trainer_hooks.evaluate_model(et, eval_config=cfg_eval)
    assert res["candidate_wins"] + res["best_wins"] + res["draws"] == 6 and res["promoted"]
    assert calls == [("save", "ckpt", "best.pth", 9), ("load", "ckpt", "best.pth")]
    et.self_play_config = dict(et.self_play_config, eval_win_rate_threshold=2.0)
    calls.clear()
    assert not trainer_hooks.evaluate_model(et, eval_config=cfg_eval)["promoted"] and calls == []


def test_trainer_hook_with_the_test_run_buffer(eng):
    """The self-play outcome tests/ref_dropin_runner.py checks on the reference's Trainer, on the hook alone: six games into
    test_run.py's deque(maxlen=100) (config.py:160) leave its last 100 examples, and a second phase plays new games."""
    from harmonies_alphazero_b200 import net, trainer_hooks

    class Manager:
        model = net.AlphaZeroNet.from_config(net.TEST_MODEL_CONFIG)

    class Trainer:
        self_play_config = {"num_games_per_iter": 6}
        mcts_config = {"num_simulations": 4, "cpuct": 1.0, "dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.25,
                       "turns_until_tau0": 15, "action_size": 143, "testing": True}
        replay_buffer = deque(maxlen=100)

    t = Trainer()
    assert trainer_hooks.execute_self_play_phase(t, Manager(), n_slots=4)["games"] == 6
    assert len(t.replay_buffer) == 100
    assert [tuple(x.shape) for x in t.replay_buffer[-1]] == [(38, 5, 7), (42,), (143,), (1,)]
    first = torch.stack([e[0] for e in t.replay_buffer])
    trainer_hooks.execute_self_play_phase(t, Manager(), n_slots=4)
    assert len(t.replay_buffer) == 100
    assert not torch.equal(torch.stack([e[0] for e in t.replay_buffer]), first)


# ---- the reference's private helpers (harmonies_engine.py:120-143,301-354,369-523) -------------
def test_end_turn_actions_equals_the_tail_of_apply_move(eng):
    """apply_move of a third placement = place the tile, then _end_turn_actions (harmonies_engine.py:
    283-292,301-329): doing the placement on the attributes and calling the private helper must give
    the state apply_move gives (same draw stream, same event) — through turn switches, the end
    trigger, player 1's last turn and the final scoring."""
    random.seed(11)
    s = eng.HarmoniesGameState()
    checked = ended = 0
    while not s.is_game_over():
        moves = s.get_legal_moves()
        mv = moves[random.randrange(len(moves))]
        nxt = s.apply_move(mv)
        if s.turn_phase == "place_tile_3":
            t = s.clone()
            tile, coord = mv
            t.player_boards[t.current_player].setdefault(coord, []).append(tile)
            t.tiles_in_hand.remove(tile)
            t._end_turn_actions()
            assert t == nxt and (t.game_over, t.winner, t.final_scores) == (nxt.game_over, nxt.winner, nxt.final_scores)
            assert t.turn_phase == nxt.turn_phase and t.current_player == nxt.current_player
            checked += 1
            ended += nxt.is_game_over()
        s = nxt
    assert checked >= 15 and ended == 1


def test_draw_and_replenish_helpers(eng):
    random.seed(5)
    s = eng.HarmoniesGameState()
    bag0 = dict(s.tile_bag)
    tiles = s._draw_tiles(3)
    assert len(tiles) == 3 and all(t in eng.TILE_TYPES for t in tiles)
    for t in eng.TILE_TYPES:
        assert s.tile_bag[t] == bag0[t] - tiles.count(t)
    more = s._draw_tiles(7)
    assert len(more) == 7 and sum(s.tile_bag.values()) == 105 - 10
    s.available_piles = s.available_piles[:2]
    before = sum(s.tile_bag.values())
    s._replenish_piles()
    assert len(s.available_piles) == 5 and all(len(p) == 3 for p in s.available_piles)
    assert sum(s.tile_bag.values()) == before - 9
    # an empty bag gives no tiles and no piles (harmonies_engine.py:123-124,135-136)
    e = eng.HarmoniesGameState()
    e.tile_bag = {t: 0 for t in eng.TILE_TYPES}
    e.available_piles = []
    assert e._draw_tiles(3) == []
    e._replenish_piles()
    assert e.available_piles == []
    # a nearly empty bag gives a partial pile (:125)
    e.tile_bag["stone"] = 2
    assert e._draw_tiles(3) == ["stone", "stone"] and e.tile_bag["stone"] == 0
    assert e._get_top_tile({(0, 0): ["wood", "plant"]}, (0, 0)) == "plant" and e._get_top_tile({}, (0, 0)) is None


def test_score_term_helpers_match_the_reference(eng):
    """_score_grass/_mountains/_fields/_buildings/_water on boards of the reference-generated golden
    scoring set (per-term values recorded from harmonies_engine.py:369-523)."""
    from tests.conftest import load_golden

    g = load_golden("scoring")
    s = eng.HarmoniesGameState()
    for i in range(0, 6000, 401):
        f = pk.unpack_fields(g["states"][i])
        for p in (0, 1):
            board = f["player_boards"][p]
            got = [s._score_grass(board, p), s._score_mountains(board, p), s._score_fields(board, p),
                   s._score_buildings(board, p), s._score_water(board, p)]
            assert got == g["terms"][i, p].tolist()
    t = eng.HarmoniesGameState({**pk.unpack_fields(g["states"][7]), "rng_key": 0})
    t._calculate_final_scores()
    t._determine_winner()
    assert t.final_scores == g["totals"][7].tolist()
    assert t.winner == (0 if t.final_scores[0] > t.final_scores[1] else 1 if t.final_scores[1] > t.final_scores[0] else -1)


def test_search_entry_point_edge_cases_follow_the_reference(eng):
    """MCTS.py:297 (terminal leaves are not sent to the network), :420-423 (greedy choice with an
    unvisited root takes the first root edge), :386-392 (the uniform fallback is written into an int
    array and truncates to zero)."""
    from harmonies_alphazero_b200 import MCTS

    cfg = {"num_simulations": 1, "cpuct": 2, "dirichlet_alpha": 0.4, "dirichlet_epsilon": 0.25,
           "turns_until_tau0": 15, "action_size": 143, "testing": True}
    random.seed(3)
    s = eng.HarmoniesGameState()
    mv, pi = MCTS.get_best_action_and_pi(s.clone(), _FakeManager(), cfg, 0)
    assert mv == s.get_legal_moves()[0] and pi.sum() == 0 and pi.dtype.kind == "i"
    # exploratory phase with an unvisited root: random legal move (MCTS.py:425-433)
    mv, pi = MCTS.get_best_action_and_pi(s.clone(), _FakeManager(), dict(cfg, testing=False), 0)
    assert mv in s.get_legal_moves() and pi.sum() == 0
    # play to the last turn: searches from there reach terminal leaves, which must not be evaluated
    while True:
        nxt = s.apply_move(s.get_legal_moves()[0])
        if nxt.is_game_over():
            break
        s = nxt
    mgr = _FakeManager()
    mv, pi = MCTS.get_best_action_and_pi(s.clone(), mgr, dict(cfg, num_simulations=12), 60)
    assert mv is not None and 1 <= mgr.calls < 12
