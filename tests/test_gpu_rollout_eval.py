"""GPU: the rollout evaluator (hz_tree_rollout_eval) — network-free leaf values from fused random playouts.

Every leaf row is restated on the host from the header's specification: rollout keys from pk.rand and the exact
canonical hash, the R re-keyed copies played out by the C oracle, value = the mover's mean outcome, priors uniform
over the legal moves.  The GPU must reproduce policy and value bits and the step total; whole searches driven by it
must match oracle.search with that restatement as its evaluator.
"""

import numpy as np
import pytest
import torch

from harmonies_alphazero_b200 import packed as pk
from tests.conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    from harmonies_alphazero_b200 import batched, selfplay, tree

    batched._lib.load()
    return batched, tree, selfplay


def _host_rollout_eval(oracle, leaves, skeys, R):
    """(policy [n,143] f32, value [n] f32, total steps) of the leaf rows, restated on the host."""
    leaves = np.ascontiguousarray(leaves, dtype=np.uint32).reshape(-1, 32)
    n = len(leaves)
    over, _ = oracle.outcome(leaves)
    legal = oracle.legal_mask(leaves)
    hashes = oracle.canon_hash(leaves, pk.KEY_EXACT)
    policy = np.zeros((n, 143), dtype=np.float32)
    copies = np.repeat(leaves, R, axis=0)
    for i in range(n):
        acts = pk.mask_to_actions(legal[i])
        if not over[i] and acts:
            policy[i, acts] = np.float32(1.0) / np.float32(len(acts))
        base = pk.rand(int(skeys[i]) ^ pk.ROLLOUT_SALT, int(hashes[i]))
        for r in range(R):
            k = pk.rand(base, r)
            copies[i * R + r, pk.W_KEYLO] = k & 0xFFFFFFFF
            copies[i * R + r, pk.W_KEYHI] = k >> 32
    live = np.repeat(over == 0, R)
    final, steps, _ = oracle.playout(copies[live], max_steps=1000)
    _, oc = oracle.outcome(final)
    o = np.zeros(n * R, dtype=np.int64)
    o[live] = oc
    sigma = np.where((leaves[:, 22] >> 24) & 1, -1, 1)
    value = (sigma * o.reshape(n, R).sum(axis=1)).astype(np.float32) / np.float32(R)
    return policy, value, int(steps.astype(np.int64).sum())


def _mixed_roots(hb, n, seed):
    """n roots at game depths 0/6/31/52/60 (the split of test_many_roots_vs_oracle)."""
    st = hb.init_states(n, seed=seed)
    cuts = [0, n // 4, n // 2, 3 * n // 4, 7 * n // 8, n]
    for (lo, hi), d in zip(zip(cuts[:-1], cuts[1:]), [0, 6, 31, 52, 60]):
        sl = st[lo:hi].clone()
        hb.playout(sl, max_steps=d)
        st[lo:hi] = sl
    return st.cpu().numpy().view(np.uint32)


def _weird_roots():
    """distinct positions of the weird goldens: terminal ones and stuck ones (no legal move, not over) included"""
    return np.unique(load_golden("weird")["states"], axis=0)


@pytest.mark.parametrize("R", [1, 2, 8, 32, 64])
def test_leaf_values_and_priors_match_the_oracle(mods, oracle, R):
    hb, tr, _ = mods
    roots = np.concatenate([_mixed_roots(hb, 512, 555), _weird_roots()])
    n = len(roots)
    skeys = np.random.default_rng(R).integers(0, 2**63, size=n, dtype=np.uint64)
    t = tr.BatchedMCTS(n, 8, key_mode=pk.KEY_EXACT)
    t.reset(hb.states_from_numpy(roots), tr.search_keys_tensor(skeys))
    t.run_synthetic(3, 2.0)                                      # grow the trees a little: leaves below the roots
    leaf = torch.empty((n, 32), dtype=torch.int32, device="cuda")
    t.select(2.0, leaf_states=leaf)
    policy = torch.full((n, 143), float("nan"), device="cuda")
    value = torch.full((n,), float("nan"), device="cuda")
    total = torch.zeros(1, dtype=torch.int64, device="cuda")
    t.rollout_eval(policy, value, R, total)
    leaves = leaf.cpu().numpy().view(np.uint32)
    hp, hv, hsteps = _host_rollout_eval(oracle, leaves, skeys, R)
    assert np.array_equal(policy.cpu().numpy().view(np.uint32), hp.view(np.uint32))
    assert np.array_equal(value.cpu().numpy().view(np.uint32), hv.view(np.uint32))
    assert int(total.item()) == hsteps
    # the row set covers what the specification singles out
    over, _ = oracle.outcome(leaves)
    stuck = (oracle.legal_mask(leaves) == 0).all(axis=1) & (over == 0)
    assert over.any() and stuck.any() and (np.abs(hv) < 1).any()


def _gpu_search(mods, roots, skeys, sims, R, key_mode, leaves, noise, eps):
    hb, tr, _ = mods
    n = len(roots)
    t = tr.BatchedMCTS(n, sims, key_mode=key_mode, leaves=leaves)
    t.reset(hb.states_from_numpy(roots), tr.search_keys_tensor(skeys))
    policy = torch.empty((t.rows, 143), device="cuda")
    value = torch.empty(t.rows, device="cuda")
    nz = torch.from_numpy(noise).cuda()
    for _ in range(sims // leaves):
        t.select(2.0)
        t.rollout_eval(policy, value, R)
        t.expand_backup(policy, value, is_logits=False, noise=nz, eps=eps)
    t.check_status()
    return t


@pytest.mark.parametrize("key_mode", [0, 1])
@pytest.mark.parametrize("leaves", [1, 4])
def test_whole_searches_match_oracle_search(mods, oracle, key_mode, leaves):
    hb, _, _ = mods
    n, sims, R, eps = 64, 32, 8, 0.25
    roots = _mixed_roots(hb, n, 77 + key_mode)
    rng = np.random.default_rng(10 * key_mode + leaves)
    skeys = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    noise = rng.gamma(0.4, size=(n, 143)).astype(np.float32) + np.float32(1e-6)
    t = _gpu_search(mods, roots, skeys, sims, R, key_mode, leaves, noise, eps)
    N, W, P, _ = (x.cpu().numpy() for x in t.root_edges())
    nn, ne, _ = (x.cpu().numpy() for x in t.stats())
    for i in range(n):
        def eval_fn(w, sk=skeys[i]):
            p, v, _ = _host_rollout_eval(oracle, np.array(w, dtype=np.uint32), [sk], R)
            return p[0], float(v[0])

        r = oracle.search(roots[i], skeys[i], sims, 2.0, noise[i], eps, eval_fn=eval_fn, key_mode=key_mode, leaves=leaves)
        assert np.array_equal(N[i], r["N"]), i
        assert np.array_equal(W[i], r["W"]), i
        assert np.array_equal(P[i].view(np.uint32), r["P"].view(np.uint32)), i
        assert nn[i] == r["n_nodes"] and ne[i] == r["n_edges"], i


def test_terminal_and_stuck_roots(mods, oracle):
    """A root that is over gets a zero row and value 0 and no rollout; a root whose mover has no legal hex gets a zero
    row and value 0 (its rollouts end at once)."""
    hb, tr, _ = mods
    w = _weird_roots()
    over, _ = oracle.outcome(w)
    phase = (w[:, 22] >> 25) & 7
    stuck = (oracle.legal_mask(w) == 0).all(axis=1) & (over == 0) & (phase >= 1) & (phase <= 3)
    roots = np.concatenate([w[over == 1][:32], w[stuck][:32]])
    assert (over == 1).sum() >= 1 and stuck.sum() >= 1
    n = len(roots)
    t = tr.BatchedMCTS(n, 4)
    t.reset(hb.states_from_numpy(roots))
    t.select(2.0)
    policy = torch.full((n, 143), 5.0, device="cuda")
    value = torch.full((n,), 5.0, device="cuda")
    total = torch.zeros(1, dtype=torch.int64, device="cuda")
    t.rollout_eval(policy, value, 16, total)
    assert (policy == 0).all() and (value == 0).all() and int(total.item()) == 0
    t.expand_backup(policy, value)
    t.check_status()
    assert (t.root_policy()[0] == 0).all()


def test_active_prefix_rows_keep_their_sentinel(mods):
    hb, tr, _ = mods
    n, K, R = 64, 2, 4
    st = hb.init_states(n, seed=31)
    hb.playout(st, max_steps=7)
    a, b = tr.BatchedMCTS(n, 8, leaves=K), tr.BatchedMCTS(n, 8, leaves=K)
    out = []
    for t, active in ((a, None), (b, 24)):
        if active is not None:
            t.set_active(torch.tensor([active], dtype=torch.int32, device="cuda"))
        t.reset(st)
        t.run_synthetic(4, 2.0)
        t.select(2.0)
        policy = torch.full((n * K, 143), -3.0, device="cuda")
        value = torch.full((n * K,), -3.0, device="cuda")
        t.rollout_eval(policy, value, R)
        out.append((policy, value))
    (pa, va), (pb, vb) = out
    assert torch.equal(pb[:24 * K], pa[:24 * K]) and torch.equal(vb[:24 * K], va[:24 * K])
    assert (pb[24 * K:] == -3.0).all() and (vb[24 * K:] == -3.0).all()


def test_rollout_counts_outside_the_powers_of_two_up_to_64_are_rejected(mods):
    hb, tr, sp = mods
    from harmonies_alphazero_b200 import _lib

    t = tr.BatchedMCTS(4, 4)
    t.reset(hb.init_states(4, seed=1))
    t.select(2.0)
    policy = torch.empty((4, 143), device="cuda")
    value = torch.empty(4, device="cuda")
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    for R in (0, -1, 3, 6, 48, 128):
        assert lib.hz_tree_rollout_eval(t.handle, R, policy.data_ptr(), value.data_ptr(), None, stream) == -1   # HZ_ERR_ARG
        with pytest.raises(_lib.HarmoniesLibraryError):
            t.rollout_eval(policy, value, R)
        with pytest.raises(ValueError):
            sp.RolloutEvaluator(R)
    assert lib.hz_tree_rollout_eval(None, 8, policy.data_ptr(), value.data_ptr(), None, stream) == -1
    assert lib.hz_tree_rollout_eval(t.handle, 8, None, value.data_ptr(), None, stream) == -1


def test_rollout_selfplay_is_the_same_with_and_without_graph_and_compaction(mods, oracle):
    hb, _, sp = mods
    sims, games = 32, 64
    out = []
    for graph, compact in ((True, True), (False, True), (True, False), (False, False)):
        cfg = sp.SelfPlayConfig(n_slots=32, num_simulations=sims, testing=True, seed=17, use_cuda_graph=graph,
                                compact_live=compact)
        t = sp.BatchedSelfPlay(sp.RolloutEvaluator(8), cfg).play(games)
        assert t.stats["games"] == games
        order = torch.argsort(t.game_id * 1000 + t.move_no.to(torch.int64))
        out.append(tuple(x[order].cpu() for x in (t.states, t.visits, t.z, t.game_id, t.move_no)))
    for other in out[1:]:
        assert all(torch.equal(x, y) for x, y in zip(out[0], other))
    S, V, Z, G, M = (x.numpy() for x in out[0])
    S = S.view(np.uint32)
    assert sorted(set(G.tolist())) == list(range(games))
    assert (V.sum(axis=1) == sims - 1).all()                        # sum N = S - 1 (MCTS.py:355-381)
    legal = oracle.legal_mask(S)
    for i in range(0, len(S), 17):
        assert set(np.nonzero(V[i])[0].tolist()) <= set(pk.mask_to_actions(legal[i]))
    # z = the game's outcome from the mover's view: replay each game's last recorded move to its end
    for g in range(0, games, 5):
        idx = np.nonzero(G == g)[0]
        assert M[idx].tolist() == list(range(len(idx)))
        last = idx[-1]
        acts = pk.mask_to_actions(legal[last])
        nxt, _ = oracle.apply(np.repeat(S[last][None], len(acts), 0), np.array(acts, dtype=np.int16))
        over, oc = oracle.outcome(nxt)
        mover = (S[idx, 22] >> 24) & 1
        want = {int(oc[k]) for k in range(len(acts)) if over[k]}     # the game ended with the last move
        assert want and any(np.array_equal(Z[idx], c * (1.0 - 2.0 * mover).astype(np.float32)) for c in want), g


def test_rollout_selfplay_with_root_noise(mods):
    hb, _, sp = mods
    torch.manual_seed(3)
    cfg = sp.SelfPlayConfig(n_slots=24, num_simulations=16, seed=5)
    t = sp.BatchedSelfPlay(sp.RolloutEvaluator(4), cfg).play(30)
    assert t.stats["games"] == 30 and (t.visits.sum(dim=1) == 15).all()
    assert set(torch.unique(t.z.abs()).tolist()) <= {0.0, 1.0}


def test_arena_with_rollout_players(mods):
    from harmonies_alphazero_b200 import arena, net

    cfg = {"num_simulations": 16, "cpuct": 2, "dirichlet_alpha": 0.1, "dirichlet_epsilon": 0,
           "turns_until_tau0": 0, "action_size": 143, "testing": True}
    ro = mods[2].RolloutEvaluator(8)
    torch.manual_seed(0)
    m = net.AlphaZeroNet.from_config(net.TEST_MODEL_CONFIG).eval()
    inf = net.InferenceNet(m, device="cuda", dtype=torch.bfloat16)
    for cand, best, games, seed in ((ro, arena.GREEDY, 8, 3), (inf, ro, 6, 5), (ro, mods[2].RolloutEvaluator(2), 5, 1)):
        r = arena.play_match(cand, best, games, cfg, seed=seed)
        assert r["games"] == games and r["candidate_wins"] + r["best_wins"] + r["draws"] == games
        assert 0.0 <= r["win_rate"] <= 1.0
        assert arena.play_match(cand, best, games, cfg, seed=seed) == r            # deterministic
