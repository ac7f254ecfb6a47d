"""The Gumbel search on the GPU (BatchedMCTS.set_gumbel / gumbel_root, include/harmonies_b200.h "Gumbel search").

- Whole trees against the C restatement (tests/gumbel_oracle.c), node for node and edge for edge, plus the root's policy
  target and played action.  CUDA's and glibc's double exp/log need not agree in the last bit, so a search may differ
  only where the oracle saw a decision whose winner led another candidate by less than 1e-9; such searches are counted
  and must stay at or below 1 %.  (The device also sums the per-node reductions in warp order, the oracle in edge
  order: the last bits of those fp64 sums may differ too.)
- PUCT is unchanged after the mode was on, the mode composes with the eval cache and the symmetry frames, and it
  refuses Dirichlet noise.
"""

import numpy as np
import pytest
import torch

from harmonies_alphazero_b200 import _lib
from tests import gumbel_oracle as go
from tests.conftest import load_golden
from tests.test_gpu_eval_cache import ElementwiseNet, _default_net, _Searcher
from tests.test_gpu_search_limits import _oracle_fn, check_invariants, compare_tree, ev_row, layout, read_tree

pytestmark = pytest.mark.gpu
NEAR_TIE = 1e-9


@pytest.fixture(scope="module")
def mods():
    from harmonies_alphazero_b200 import batched, tree

    batched._lib.load()
    return batched, tree


def _roots(hb, n, seed):
    """a third fresh, a third mid-game, a third from the weird goldens"""
    k = n // 3
    st = hb.init_states(n - k, seed=seed)
    mid = st[k:].clone()
    hb.playout(mid, max_steps=37)
    st[k:] = mid
    weird = load_golden("weird")["states"].view(np.uint32)
    weird = weird[(seed * 7919 + 131 * np.arange(k)) % len(weird)]
    return np.concatenate([st.cpu().numpy().view(np.uint32), weird])


def _run(mods, roots, skeys, sims, g, evals=None):
    hb, tr = mods
    n = len(roots)
    t = tr.BatchedMCTS(n, sims)
    t.set_gumbel(num_sims=sims, **g)
    t.reset(hb.states_from_numpy(roots), tr.search_keys_tensor(skeys))
    policy = torch.empty((n, 143), dtype=torch.float32, device="cuda")
    value = torch.empty(n, dtype=torch.float32, device="cuda")
    leaf = torch.empty((n, 32), dtype=torch.int32, device="cuda")
    for _ in range(sims):
        t.select(2.0, leaf_states=leaf)
        if evals is None:
            t.fake_eval(policy, value)
        else:
            p, v = evals(leaf.cpu().numpy().view(np.uint32))
            policy.copy_(torch.from_numpy(p))
            value.copy_(torch.from_numpy(v))
        t.expand_backup(policy, value)
    return t


def _parity(mods, oracle, sims, m, ev):
    """(searches, searches that differ at a near-tie of the oracle) of one configuration; any other difference raises"""
    n = 24 if sims <= 64 else 12
    roots = _roots(mods[0], n, 11 * sims + m)
    skeys = np.random.default_rng(sims * 100 + m).integers(0, 2**63, size=n, dtype=np.uint64)
    g = dict(m=m, c_visit=50.0, c_scale=0.1, scale=1.0)
    f = None if ev is None else ev_row(oracle, ev)
    t = _run(mods, roots, skeys, sims, g, f)
    gd = read_tree(t, layout(n, sims, 0, 1))
    pol, act, rv = (x.cpu().numpy() for x in t.gumbel_root())
    near = 0
    for i in range(n):
        r = go.search(roots[i], skeys[i], sims, g, eval_fn=None if f is None else _oracle_fn(f), tree=True)
        assert r["rc"] == 0 and gd["status"][i] == 0
        try:
            compare_tree(gd, i, r)
            check_invariants(gd, i, layout(n, sims, 0, 1))
            assert np.abs(pol[i] - r["policy"]).max() <= 1e-6, "policy target"
            assert int(act[i]) == r["action"], "action"
            assert rv[i] == np.float32(r["root_value"]), "root value"
        except AssertionError as e:
            if r["gap"] < NEAR_TIE:
                near += 1
                continue
            raise AssertionError(f"tree {i}, {sims} simulations, m = {m}, evaluator {ev}, gap {r['gap']}: {e}") from e
    return n, near


def test_trees_match_the_oracle(mods, oracle):
    """every (n, m, evaluator) configuration; at most 1 % of all searches may differ, each at an oracle near-tie"""
    searches = near = 0
    for sims in (1, 2, 15, 16, 17, 64, 100):
        for m in (1, 4, 16):
            for ev in (None, "equal", "stair"):
                a, b = _parity(mods, oracle, sims, m, ev)
                searches, near = searches + a, near + b
    assert near <= searches // 100, (near, searches)


def test_played_action_is_legal_and_policy_sums_to_one(mods):
    hb, tr = mods
    n, sims = 256, 32
    roots = _roots(hb, n, 5)
    t = _run(mods, roots, np.arange(n, dtype=np.uint64) + 9, sims, dict(m=16))
    pol, act, _ = t.gumbel_root()
    child = t.root_edges()[3].cpu().numpy()
    legal = hb.legal_mask(hb.states_from_numpy(roots)).cpu().numpy().view(np.uint32)
    pol, act = pol.cpu().numpy(), act.cpu().numpy()
    for i in range(n):
        edges = child[i] >= 0
        if not edges.any():                 # terminal root, or no legal move
            assert act[i] == -1 and not pol[i].any(), i
            continue
        bits = np.array([(legal[i, a >> 5] >> (a & 31)) & 1 for a in range(143)], bool)
        assert 0 <= act[i] < 143 and bits[act[i]] and edges[act[i]], (i, int(act[i]))
        assert abs(float(pol[i].sum()) - 1.0) < 1e-5 and not pol[i][~bits].any(), i


def _puct(mods, roots, t=None, sims=40):
    hb, tr = mods
    n = roots.shape[0]
    t = t or tr.BatchedMCTS(n, sims)
    t.reset(roots, tr.search_keys_tensor(np.arange(n, dtype=np.uint64) + 3))
    noise = torch.rand((n, 143), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)).add_(1e-3)
    policy = torch.empty((n, 143), dtype=torch.float32, device="cuda")
    value = torch.empty(n, dtype=torch.float32, device="cuda")
    for _ in range(sims):
        t.select(2.0)
        t.fake_eval(policy, value)
        t.expand_backup(policy, value, noise=noise, eps=0.25)
    N, W, P, child = t.root_edges()
    return t, (N, W.view(torch.int64), P.view(torch.int32), child, t.choose())


def test_puct_unchanged_after_gumbel(mods):
    hb, tr = mods
    roots = hb.init_states(64, seed=21)
    hb.playout(roots[32:], max_steps=30)
    _, ref = _puct(mods, roots)
    t = tr.BatchedMCTS(64, 40)
    t.set_gumbel(m=16)
    t.reset(roots)
    policy = torch.empty((64, 143), dtype=torch.float32, device="cuda")
    value = torch.empty(64, dtype=torch.float32, device="cuda")
    for _ in range(10):
        t.select(2.0)
        t.fake_eval(policy, value)
        with pytest.raises(_lib.HarmoniesLibraryError):
            t.expand_backup(policy, value, noise=torch.ones((64, 143), device="cuda"), eps=0.25)   # Dirichlet refused
        t.expand_backup(policy, value)
    t.set_gumbel(None)
    _, got = _puct(mods, roots, t)
    for a, b in zip(ref, got):
        assert torch.equal(a, b)


def _gumbel_chain(mods, ev, kind, sym, entries, n=32, sims=16, moves=24, seed=4):
    """(root edges, gumbel_root) of every search along real games, network evaluator, cache on or off"""
    hb, tr = mods
    import harmonies_alphazero_b200.net as net

    s = _Searcher((hb, net, None, tr, None), ev, kind, n, sims, hb.KEY_EXACT, 1, sym, entries)
    s.t.set_gumbel(m=8, num_sims=sims)
    roots = hb.init_states(n, seed=seed)
    out = []
    for _ in range(moves):
        s.search(roots, None)
        N, W, _, _ = s.t.root_edges()
        pol, act, rv = s.t.gumbel_root()
        out.append((N, W.view(torch.int64), pol.view(torch.int32), act, rv.view(torch.int32)))
        over, _ = hb.outcome(roots)
        a = torch.where(act < 0, hb.random_actions(roots), act)
        hb.apply(roots, torch.where(over.bool(), torch.full_like(a, -1), a))
    s.t.check_status()
    return out


@pytest.mark.parametrize("kind,sym", [("tiles", None), ("tiles", "board"), ("nhwc40", "full")])
def test_gumbel_identical_with_eval_cache(mods, kind, sym):
    import harmonies_alphazero_b200.net as net

    ev = _default_net(net, "random", seed=2) if kind == "tiles" else ElementwiseNet()    # one evaluator for both runs
    a = _gumbel_chain(mods, ev, kind, sym, 0)
    b = _gumbel_chain(mods, ev, kind, sym, 1 << 16)
    for mv, (x, y) in enumerate(zip(a, b)):
        for u, v in zip(x, y):
            assert torch.equal(u, v), f"move {mv}"


@pytest.mark.parametrize("sym", ["board", "full"])
def test_gumbel_identical_with_symmetry_under_synthetic_evaluator(mods, sym):
    hb, tr = mods
    roots = hb.init_states(48, seed=8)
    hb.playout(roots[24:], max_steps=25)
    res = []
    for mode in (None, sym):
        t = tr.BatchedMCTS(48, 24)
        t.set_symmetry(mode)
        t.set_gumbel(m=16)
        t.reset(roots)
        t.run_synthetic(24, 2.0)
        N, W, _, _ = t.root_edges()
        pol, act, _ = t.gumbel_root()
        res.append((N, W.view(torch.int64), pol.view(torch.int32), act))
    for u, v in zip(*res):
        assert torch.equal(u, v)


def test_graph_replay_equals_eager(mods):
    hb, tr = mods
    n, sims = 64, 20
    roots = hb.init_states(n, seed=12)
    hb.playout(roots[32:], max_steps=50)
    policy = torch.empty((n, 143), dtype=torch.float32, device="cuda")
    value = torch.empty(n, dtype=torch.float32, device="cuda")

    def step(t):
        t.select(2.0)
        t.fake_eval(policy, value)
        t.expand_backup(policy, value)

    eager = tr.BatchedMCTS(n, sims)
    eager.set_gumbel(m=16)
    eager.reset(roots)
    for _ in range(sims):
        step(eager)
    g = tr.BatchedMCTS(n, sims)
    g.set_gumbel(m=16)
    g.reset(roots)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step(g)                                         # warm-up step, then capture one step and replay it
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            step(g)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(sims - 1):
        graph.replay()
    torch.cuda.synchronize()
    a, b = eager.gumbel_root(), g.gumbel_root()
    assert torch.equal(eager.root_edges()[0], g.root_edges()[0])
    for u, v in zip(a, b):
        assert torch.equal(u, v)


# ---- self-play, replay and arena ------------------------------------------------------------------------------------
def _selfplay(net, games=48, slots=32, sims=16, **kw):
    from harmonies_alphazero_b200 import selfplay as sp

    cfg = sp.SelfPlayConfig(n_slots=slots, num_simulations=sims, search="gumbel", gumbel_m=8, seed=5, **kw)
    return sp.BatchedSelfPlay(net, cfg).play(games)


def _same_traj(a, b):
    for f in ("states", "visits", "z", "game_id", "move_no"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    assert torch.equal(a.policy.view(torch.int32), b.policy.view(torch.int32))


def test_selfplay_output(mods):
    from harmonies_alphazero_b200 import selfplay as sp

    hb, _ = mods
    tr = _selfplay(sp.SyntheticEvaluator())
    assert tr.policy is not None and tr.policy.shape == (len(tr), 143) and tr.stats["games"] == 48
    legal = hb.legal_mask(tr.states.contiguous()).cpu().numpy().view(np.uint32)
    bits = ((legal[:, np.arange(143) >> 5] >> (np.arange(143) & 31).astype(np.uint32)) & 1).astype(bool)
    pol = tr.policy.cpu().numpy()
    has = pol.sum(axis=1) > 0
    assert has.mean() > 0.9                                   # rows without a search (one-move roots) may be empty
    assert np.abs(pol[has].sum(axis=1) - 1.0).max() < 1e-5 and not pol[~bits].any()
    assert torch.equal(tr.pi(), tr.policy)
    ex = tr.to_reference_examples(last=10)
    assert len(ex) == 10 and torch.equal(ex[-1][2], tr.policy[-1].cpu())
    assert int(tr.visits.to(torch.int64).sum()) > 0         # the visit counts are still recorded


def test_selfplay_graph_compaction_and_symmetry_identical(mods):
    from harmonies_alphazero_b200 import selfplay as sp

    ref = _selfplay(sp.SyntheticEvaluator())
    _same_traj(ref, _selfplay(sp.SyntheticEvaluator(), use_cuda_graph=False))
    _same_traj(ref, _selfplay(sp.SyntheticEvaluator(), compact_live=False))
    _same_traj(ref, _selfplay(sp.SyntheticEvaluator(), eval_symmetry="full"))


def test_selfplay_identical_with_eval_cache(mods):
    import harmonies_alphazero_b200.net as net

    ev = _default_net(net, "random", seed=3)
    _same_traj(_selfplay(ev, games=40), _selfplay(ev, games=40, eval_cache=1 << 15))


def test_selfplay_rollout_evaluator_and_rejections(mods):
    from harmonies_alphazero_b200 import selfplay as sp

    tr = _selfplay(sp.RolloutEvaluator(4), games=16, slots=16, sims=8)
    assert tr.stats["games"] == 16 and tr.policy is not None
    with pytest.raises(ValueError):
        _selfplay(sp.SyntheticEvaluator(), leaves_per_step=2)
    with pytest.raises(ValueError):
        sp.BatchedSelfPlay(sp.SyntheticEvaluator(), sp.SelfPlayConfig(n_slots=4, search="mcts"))
    cfg = sp.SelfPlayConfig.from_mcts_config({"num_simulations": 16, "cpuct": 2.0, "search": "gumbel", "gumbel_m": 4,
                                              "gumbel_c_visit": 20, "gumbel_c_scale": 0.5})
    assert (cfg.search, cfg.gumbel_m, cfg.gumbel_c_visit, cfg.gumbel_c_scale) == ("gumbel", 4, 20.0, 0.5)


def test_replay_ring_policy_targets(mods):
    from harmonies_alphazero_b200 import selfplay as sp
    from harmonies_alphazero_b200.replay import ReplayRing

    tr = _selfplay(sp.SyntheticEvaluator())
    ring = ReplayRing(4096)
    ring.extend(tr)
    n = len(tr)
    idx = torch.arange(n, device="cuda")
    _, _, pi, _ = ring._batch(idx)
    assert torch.equal(pi, tr.policy)
    sym = torch.randint(0, 480, (n,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    board, glob, pi, z = ring._batch(idx, sym=sym)
    want = tr.transform(sym)
    assert torch.equal(pi, want.policy)
    b2, g2 = want.encode()
    assert torch.equal(board, b2) and torch.equal(glob, g2)
    board, glob, pi, z = ring.sample(64, augment="full", generator=torch.Generator(device="cuda").manual_seed(1))
    assert pi.shape == (64, 143)
    other = ReplayRing(4096)
    other.load_state_dict(ring.state_dict())
    assert torch.equal(other._batch(idx)[2], tr.policy)
    puct = sp.BatchedSelfPlay(sp.SyntheticEvaluator(), sp.SelfPlayConfig(n_slots=16, num_simulations=8, seed=1)).play(8)
    with pytest.raises(ValueError):
        ring.extend(puct)                                       # a ring holds one kind of target
    r = ReplayRing(64)
    r.extend(puct)
    with pytest.raises(ValueError):
        r.extend(tr)


def test_gumbel_root_respects_active_prefix(mods):
    hb, tr = mods
    t = tr.BatchedMCTS(16, 8)
    t.set_gumbel(m=4)
    t.reset(hb.init_states(16, seed=1))
    t.run_synthetic(8, 2.0)
    t.set_active(torch.tensor([10], dtype=torch.int32, device="cuda"))
    pol, act, rv = t.gumbel_root()
    assert (act[10:] == -1).all() and not pol[10:].any() and not rv[10:].any()
    assert (act[:10] >= 0).all()


def test_arena_mixed_search(mods):
    from harmonies_alphazero_b200 import arena
    from harmonies_alphazero_b200.selfplay import RolloutEvaluator

    cfg = {"num_simulations": 8, "cpuct": 2.0, "gumbel_m": 4}
    r = arena.play_match(RolloutEvaluator(4), RolloutEvaluator(4), 6, cfg, search=("gumbel", "puct"))
    assert r["candidate_wins"] + r["best_wins"] + r["draws"] == 6 and r["games"] == 6
    r = arena.play_match(RolloutEvaluator(4), arena.GREEDY, 4, cfg, search="gumbel")
    assert r["candidate_wins"] + r["best_wins"] + r["draws"] == 4
    with pytest.raises(ValueError):
        arena.play_match(RolloutEvaluator(4), RolloutEvaluator(4), 2, cfg, search="alphabeta")
