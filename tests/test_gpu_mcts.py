"""GPU parity tests of the search-tree kernels through the C ABI.

Contract (BASELINE.json north_star): given identical priors and values, visit counts are
identical to the reference's and policy targets agree within 1e-6 fp32.  Anchors: the
committed reference searches (tests/golden/mcts.npz, produced by MCTS.py itself) and the C
oracle on many more seeded roots.
"""

import numpy as np
import pytest
import torch

from tests.conftest import load_golden
from harmonies_alphazero_b200 import packed as pk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    from harmonies_alphazero_b200 import batched, tree

    batched._lib.load()
    return batched, tree


def _run_group(mods, roots, skeys, sims, cpuct, noise, eps, key_mode=1):
    hb, tr = mods
    n = len(roots)
    t = tr.BatchedMCTS(n, sims, key_mode=key_mode)
    t.reset(hb.states_from_numpy(roots), tr.search_keys_tensor(skeys))
    nz = None if noise is None else torch.from_numpy(np.ascontiguousarray(noise, dtype=np.float32)).cuda()
    t.run_synthetic(sims, cpuct, noise=nz, eps=eps)
    t.check_status()
    return t


def test_golden_reference_searches(mods):
    """84 searches run by the reference's own MCTS.py: N, W, P, node/edge counts, pi, move."""
    g = load_golden("mcts")
    groups = {}
    for i in range(len(g["sims"])):
        k = (int(g["sims"][i]), float(g["cpuct"][i]), bool(g["testing"][i]), float(g["eps"][i]))
        groups.setdefault(k, []).append(i)
    for (sims, cpuct, testing, eps), idx in groups.items():
        idx = np.array(idx)
        t = _run_group(mods, g["root"][idx], g["skey"][idx], sims, cpuct, None if testing else g["noise"][idx], eps)
        N, W, P, _ = (x.cpu().numpy() for x in t.root_edges())
        assert np.array_equal(N, g["N"][idx])
        assert np.array_equal(W, g["W"][idx])
        assert np.array_equal(P.view(np.uint32), g["P"][idx].view(np.uint32))
        nn, ne, _ = (x.cpu().numpy() for x in t.stats())
        assert np.array_equal(nn, g["n_nodes"][idx]) and np.array_equal(ne, g["n_edges"][idx])
        visits, pi = (x.cpu().numpy() for x in t.root_policy())
        assert np.array_equal(visits, g["N"][idx])
        assert np.abs(pi.astype(np.float64) - g["pi"][idx]).max() <= 1e-6   # tolerance of north_star
        expl = ((g["testing"][idx] == 0) & (g["move_no"][idx] < g["tau0"][idx])).astype(np.uint8)
        a = t.choose(torch.from_numpy(g["choice_u"][idx]).cuda(), torch.from_numpy(expl).cuda()).cpu().numpy()
        assert np.array_equal(a, g["action"][idx])
        greedy = t.choose().cpu().numpy()
        want = np.where(g["N"][idx].sum(1) > 0, g["N"][idx].argmax(1), -1)
        assert np.array_equal(greedy, want)


@pytest.mark.parametrize("key_mode", [0, 1])
def test_many_roots_vs_oracle(mods, oracle, key_mode):
    """512 roots at mixed game depths x 64 simulations, both key modes, with root noise."""
    hb, _ = mods
    n, sims, cpuct, eps = 512, 64, 2.0, 0.25
    st = hb.init_states(n, seed=555)
    for lo, hi, d in [(0, 128, 0), (128, 256, 6), (256, 384, 31), (384, 448, 52), (448, 512, 60)]:
        sl = st[lo:hi].clone()
        hb.playout(sl, max_steps=d)
        st[lo:hi] = sl
    roots = st.cpu().numpy().view(np.uint32)
    rng = np.random.default_rng(8)
    skeys = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    noise = rng.gamma(0.4, size=(n, 143)).astype(np.float32) + np.float32(1e-6)
    t = _run_group(mods, roots, skeys, sims, cpuct, noise, eps, key_mode=key_mode)
    N, W, P, _ = (x.cpu().numpy() for x in t.root_edges())
    nn, ne, _ = (x.cpu().numpy() for x in t.stats())
    for i in range(n):
        r = oracle.search(roots[i], skeys[i], sims, cpuct, noise[i], eps, key_mode=key_mode)
        assert np.array_equal(N[i], r["N"]), i
        assert np.array_equal(W[i], r["W"]), i
        assert np.array_equal(P[i].view(np.uint32), r["P"].view(np.uint32)), i
        assert nn[i] == r["n_nodes"] and ne[i] == r["n_edges"], i


def test_full_size_config3_properties_and_oracle_subsample(mods, oracle):
    """BASELINE.json configs[3] sizes: 4,096 trees x 100 simulations (synthetic evaluator).
    Size-independent properties on all trees, identical visit counts vs the oracle on a
    192-tree subsample, default (derived) search keys."""
    hb, tr = mods
    n, sims = 4096, 100
    st = hb.init_states(n, seed=4040)
    hb.playout(st, max_steps=10)
    t = tr.BatchedMCTS(n, sims)
    t.reset(st)                                   # keys = rand(game key ^ SEARCH_SALT, moves)
    t.run_synthetic(sims, 2.0)
    t.check_status()
    N, W, P, child = (x.cpu().numpy() for x in t.root_edges())
    nn, ne, _ = (x.cpu().numpy() for x in t.stats())
    assert (N.sum(axis=1) == sims - 1).all()                       # MCTS.py:355-381: sum N = S - 1
    legal = hb.legal_mask(st).cpu().numpy().view(np.uint32)
    for i in range(0, n, 97):
        acts = pk.mask_to_actions(legal[i])
        assert set(np.nonzero(child[i] >= 0)[0].tolist()) == set(acts)     # one root edge per legal move
        assert set(np.nonzero(N[i])[0].tolist()) <= set(acts)
    assert (np.abs(W) <= N + 1e-9).all() and (nn <= 1 + 69 * sims).all() and (ne >= nn - 1).all()
    words = st.cpu().numpy().view(np.uint32)
    for i in range(0, n, 22)[:192]:
        f = pk.unpack_fields(words[i])
        skey = pk.rand(f["rng_key"] ^ pk.SEARCH_SALT, f["moves"])
        r = oracle.search(words[i], skey, sims, 2.0)
        assert np.array_equal(N[i], r["N"]) and np.array_equal(W[i], r["W"]), i
        assert nn[i] == r["n_nodes"] and ne[i] == r["n_edges"], i


@pytest.mark.parametrize("leaves", [2, 4, 8])
def test_virtual_loss_mode_matches_oracle(mods, oracle, leaves):
    """throughput mode (north_star: select/expand/backup "using virtual loss"): K simulations in
    flight per tree and step.  Oracle = the reference's search restated with the same
    virtual-loss schedule (hzo_search_vl; leaves=1 is the pinned sequential search)."""
    hb, tr = mods
    n, sims, cpuct, eps = 256, 64, 2.0, 0.25
    st = hb.init_states(n, seed=909)
    for lo, hi, d in [(0, 64, 0), (64, 128, 5), (128, 192, 30), (192, 256, 58)]:
        sl = st[lo:hi].clone()
        hb.playout(sl, max_steps=d)
        st[lo:hi] = sl
    roots = st.cpu().numpy().view(np.uint32)
    rng = np.random.default_rng(leaves)
    skeys = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    noise = rng.gamma(0.4, size=(n, 143)).astype(np.float32) + np.float32(1e-6)
    t = tr.BatchedMCTS(n, sims, leaves=leaves)
    t.reset(hb.states_from_numpy(roots), tr.search_keys_tensor(skeys))
    t.run_synthetic(sims, cpuct, noise=torch.from_numpy(noise).cuda(), eps=eps)
    t.check_status()
    N, W, P, _ = (x.cpu().numpy() for x in t.root_edges())
    nn, ne, _ = (x.cpu().numpy() for x in t.stats())
    # every in-flight visit has landed: total visits = sims minus the ones that ended at the root
    for i in range(n):
        r = oracle.search(roots[i], skeys[i], sims, cpuct, noise[i], eps, leaves=leaves)
        assert np.array_equal(N[i], r["N"]), i
        assert np.array_equal(W[i], r["W"]), i
        assert np.array_equal(P[i].view(np.uint32), r["P"].view(np.uint32)), i
        assert nn[i] == r["n_nodes"] and ne[i] == r["n_edges"], i


def test_select_outputs_leaf_encoding(mods, oracle):
    """the tensors handed to the network are create_state_tensors(leaf) (MCTS.py:299)"""
    hb, tr = mods
    n, sims = 256, 12
    st = hb.init_states(n, seed=99)
    hb.playout(st, max_steps=9)
    t = tr.BatchedMCTS(n, sims)
    t.reset(st, tr.search_keys_tensor(np.arange(n, dtype=np.uint64)))
    policy = torch.empty((n, 143), device="cuda")
    value = torch.empty(n, device="cuda")
    leaf = torch.empty((n, 32), dtype=torch.int32, device="cuda")
    for s in range(sims):
        # every (dtype, layout) but T16K (test_leaf_encoder_writes_the_stem_image); pad40 is the 40-channel NHWC
        # layout (channels 38 and 39 written as zero) that the self-play stem reads
        for dtype in (torch.float32, torch.bfloat16):
            for cl, pad40 in ((False, False), (True, False), (True, True)):
                board = torch.full((n, 40 if pad40 else 38, 5, 7), 7.0, dtype=dtype, device="cuda").contiguous(
                    memory_format=torch.channels_last if cl else torch.contiguous_format)
                glob = torch.empty((n, 42), dtype=dtype, device="cuda")
                t.select(2.0, board, glob, leaf, dtype=dtype, channels_last=cl, pad40=pad40)
                b2, g2 = hb.encode(leaf, dtype=dtype, channels_last=cl)
                assert torch.equal(board[:, :38], b2) and (board[:, 38:] == 0).all() and torch.equal(glob, g2)
                if dtype == torch.float32:
                    ob, og = oracle.encode(leaf.cpu().numpy().view(np.uint32))
                    assert np.array_equal(board[:, :38].cpu().numpy(), ob) and np.array_equal(glob.cpu().numpy(), og)
        t.fake_eval(policy, value)
        # synthetic evaluator == packed.fake_eval of the leaf's exact hash
        if s == 3:
            w = leaf[7].cpu().numpy().view(np.uint32)
            p, v = pk.fake_eval(pk.canon_hash(w))
            assert np.array_equal(policy[7].cpu().numpy(), p) and float(value[7]) == v
        t.expand_backup(policy, value)
    t.check_status()


def test_fused_softmax_path(mods):
    """is_logits=1: priors = softmax(logits) inside the expand kernel (model.py:104)"""
    hb, tr = mods
    n, sims = 128, 20
    st = hb.init_states(n, seed=4)
    keys = tr.search_keys_tensor(np.arange(n, dtype=np.uint64) + 17)
    torch.manual_seed(0)
    logits = torch.randn((sims, n, 143), device="cuda")
    values = torch.tanh(torch.randn((sims, n), device="cuda"))
    res = []
    for fused in (False, True):
        t = tr.BatchedMCTS(n, sims)
        t.reset(st, keys)
        for s in range(sims):
            t.select(2.0)
            if fused:
                t.expand_backup(logits[s], values[s], is_logits=True)
            else:
                t.expand_backup(torch.softmax(logits[s], dim=1).contiguous(), values[s])
        res.append(t.root_edges())
    # softmax rounding differs in the last ulp; visit counts only flip on exact near-ties
    same = (res[0][0] == res[1][0]).all(dim=1).float().mean().item()
    assert same > 0.9
    assert torch.allclose(res[0][2], res[1][2], rtol=1e-5, atol=1e-7)


def test_golden_searches_with_the_reference_models_priors(mods):
    """16 searches x 100 simulations run by the reference's MCTS.py with the reference's default-size
    AlphaZeroModel behind ModelManager.predict (real fp32 softmax priors: W sums round, priors are not
    dyadic).  The GPU trees are fed the recorded (priors, value) table in the reference's call order
    (terminal leaves are not evaluated, MCTS.py:297) and must reproduce N, W, P, the node / edge counts,
    pi within 1e-6 and the chosen move."""
    hb, tr = mods
    g = load_golden("mcts_real")
    sims = int(g["sims"])
    for testing in (0, 1):
        idx = np.nonzero(g["testing"] == testing)[0]
        n = len(idx)
        t = tr.BatchedMCTS(n, sims)
        t.reset(hb.states_from_numpy(g["root"][idx]), tr.search_keys_tensor(g["skey"][idx]))
        noise = None if testing else torch.from_numpy(np.ascontiguousarray(g["noise"][idx])).cuda()
        eps = float(g["eps"][idx][0])
        assert (g["eps"][idx] == eps).all()
        table_p, table_v = torch.from_numpy(g["table_p"][idx]).cuda(), torch.from_numpy(g["table_v"][idx]).cuda()
        used = torch.zeros(n, dtype=torch.int64, device="cuda")
        leaf = torch.empty((n, 32), dtype=torch.int32, device="cuda")
        rows = torch.arange(n, device="cuda")
        for _ in range(sims):
            t.select(float(g["cpuct"][idx][0]), leaf_states=leaf)
            live = ((leaf[:, 22] >> 29) & 3) == 0                  # is_game_over <=> winner bits set
            k = used.clamp_max(sims - 1)
            t.expand_backup(table_p[rows, k].contiguous(), table_v[rows, k].contiguous(), noise=noise, eps=eps)
            used += live.to(torch.int64)
        t.check_status()
        assert np.array_equal(used.cpu().numpy(), g["n_eval"][idx])          # same number of network calls
        N, W, P, _ = (x.cpu().numpy() for x in t.root_edges())
        assert np.array_equal(N, g["N"][idx])
        assert np.array_equal(W, g["W"][idx])
        assert np.array_equal(P.view(np.uint32), g["P"][idx].view(np.uint32))
        nn, ne, _ = (x.cpu().numpy() for x in t.stats())
        assert np.array_equal(nn, g["n_nodes"][idx]) and np.array_equal(ne, g["n_edges"][idx])
        _, pi = (x.cpu().numpy() for x in t.root_policy())
        assert np.abs(pi.astype(np.float64) - g["pi"][idx]).max() <= 1e-6
        expl = ((g["testing"][idx] == 0) & (g["move_no"][idx] < g["tau0"][idx])).astype(np.uint8)
        a = t.choose(torch.from_numpy(g["choice_u"][idx]).cuda(), torch.from_numpy(expl).cuda()).cpu().numpy()
        assert np.array_equal(a, g["action"][idx])


def test_arena_overflow_is_reported(mods):
    hb, tr = mods
    n = 8
    st = hb.init_states(n, seed=1)
    t = tr.BatchedMCTS(n, 50, max_nodes=40)
    t.reset(st, tr.search_keys_tensor(np.arange(n, dtype=np.uint64)))
    t.run_synthetic(50, 2.0)
    with pytest.raises(RuntimeError):
        t.check_status()


def test_overflow_survives_reset(mods):
    """hz_tree_reset starts a new search but keeps the record of a truncated one (sticky high
    nibble): a caller that checks only every few searches still sees it."""
    hb, tr = mods
    n = 8
    st = hb.init_states(n, seed=1)
    t = tr.BatchedMCTS(n, 50, max_nodes=40)
    t.reset(st, tr.search_keys_tensor(np.arange(n, dtype=np.uint64)))
    t.run_synthetic(50, 2.0)
    t.reset(st, tr.search_keys_tensor(np.arange(n, dtype=np.uint64)))
    t.run_synthetic(1, 2.0)                      # a tiny search that fits (the root expansion: <= 5 children)
    status = t.stats()[2].cpu().numpy()
    assert (status & 0x0F == 0).all() and (status & 0xF0 != 0).any()
    with pytest.raises(RuntimeError):
        t.check_status()


def test_terminal_root(mods):
    hb, tr = mods
    st = hb.init_states(4, seed=3)
    hb.playout(st)
    t = tr.BatchedMCTS(4, 10)
    t.reset(st, tr.search_keys_tensor(np.arange(4, dtype=np.uint64)))
    t.run_synthetic(10, 2.0)
    visits, pi = t.root_policy()
    assert (visits == 0).all() and (pi == 0).all()
    assert (t.choose() == -1).all()   # MCTS.py:439: (None, pi)


def test_active_prefix_leaves_other_trees_untouched(mods):
    """hz_tree_set_active: trees beyond the device-side count keep their previous search bit for bit,
    the active ones search exactly as without the switch."""
    hb, tree = mods[0], mods[-1]
    st = hb.init_states(64, seed=21)
    hb.playout(st, max_steps=9)
    a = tree.BatchedMCTS(64, 32)
    b = tree.BatchedMCTS(64, 32)
    a.reset(st); a.run_synthetic(20, 2.0)
    b.reset(st); b.run_synthetic(20, 2.0)
    st2 = st.clone()
    hb.playout(st2, max_steps=3)
    na = torch.tensor([24], dtype=torch.int32, device="cuda")
    b.set_active(na)
    b.reset(st2); b.run_synthetic(32, 2.0)
    c = tree.BatchedMCTS(64, 32)
    c.reset(st2); c.run_synthetic(32, 2.0)
    Nb, Wb, Pb, _ = b.root_edges(); Na, Wa, Pa, _ = a.root_edges(); Nc, Wc, Pc, _ = c.root_edges()
    assert torch.equal(Nb[:24], Nc[:24]) and torch.equal(Wb[:24], Wc[:24]) and torch.equal(Pb[:24], Pc[:24])
    assert torch.equal(Nb[24:], Na[24:]) and torch.equal(Wb[24:], Wa[24:])
    b.set_active(None)
    b.reset(st2); b.run_synthetic(32, 2.0)
    Nb, Wb, _, _ = b.root_edges()
    assert torch.equal(Nb, Nc) and torch.equal(Wb, Wc)
