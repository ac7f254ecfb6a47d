"""Whole search trees of the GPU kernels against the C oracle, node for node and edge for edge,
at the limits that ordinary searches never reach:

- paths deeper than a warp (back_fill of path edges 32 and beyond, with and without virtual loss);
- wide virtual loss (K = 3, 20, 32, 64);
- degenerate PUCT inputs: zero and subnormal priors, cpuct * P overflowing to inf, cpuct = 0,
  exact ties at every level, values of +-1, -0.0 and inexact decimals, root noise with eps 0 and 1;
- an arena that the search fills exactly (max_nodes);
- hz_tree_root_policy and hz_tree_choose at the boundaries of the sampling threshold.

The device arenas are read straight from BatchedMCTS.workspace through a restatement of
hz_mcts.cu's layout_for; the reader checks itself against hz_tree_workspace_bytes,
hz_tree_root_edges and hz_tree_stats before any comparison uses it.  Besides the oracle's tree,
each comparison checks what the root statistics cannot show: no in-flight visit left on an
edge, the child cache (edge_cinfo) agreeing with the child's node arrays, and the hash table
holding every node exactly once where linear probing finds it.
"""

import numpy as np
import pytest
import torch

from harmonies_alphazero_b200 import packed as pk

ACTIONS = np.arange(143)


@pytest.fixture(scope="module")
def mods():
    from harmonies_alphazero_b200 import batched, tree

    batched._lib.load()
    return batched, tree


# ---- the device arenas (hz_mcts.cu layout_for, restated) ------------------------------------------------------------
_ARRAYS = [   # (name, bytes per element, per: n = node, e = edge, s = table slot, p = path entry, r = row (tree, leaf), t = tree)
    ("node_state", 128, "n"), ("node_hash", 8, "n"), ("node_edge0", 4, "n"), ("node_info", 4, "n"),
    ("edge_child", 4, "e"), ("edge_N", 4, "e"), ("edge_W", 8, "e"), ("edge_P", 4, "e"), ("edge_am", 2, "e"),
    ("table", 4, "s"), ("path", 4, "p"), ("depth", 4, "r"), ("leaf", 4, "r"), ("sim", 4, "t"), ("n_nodes", 4, "t"),
    ("n_edges", 4, "t"), ("status", 1, "t"), ("search_key", 8, "t"), ("edge_V", 4, "e"), ("table_hash", 8, "s"),
    ("edge_cinfo", 4, "e"),
]
_NP = {"node_state": np.uint32, "node_hash": np.uint64, "node_edge0": np.uint32, "node_info": np.uint32,
       "edge_child": np.uint32, "edge_N": np.int32, "edge_W": np.float64, "edge_P": np.float32, "edge_am": np.uint16,
       "table": np.uint32, "table_hash": np.uint64, "edge_V": np.int32, "edge_cinfo": np.uint32}


def layout(n_trees, max_sims, max_nodes, leaves):
    """dict(max_nodes, max_edges, table_size, off = {name: (byte offset, elements per tree, bytes per element)}, total)"""
    mn = max_nodes if max_nodes > 0 else 1 + 69 * max_sims
    me = 69 * max_sims + 32
    ts = 64
    while ts < 2 * mn:
        ts <<= 1
    per = {"n": mn, "e": me, "s": ts, "p": leaves * (max_sims + 1), "r": leaves, "t": 1}
    off, o = {}, 0
    for name, b, k in _ARRAYS:
        off[name] = (o, per[k], b)
        o += (n_trees * per[k] * b + 255) & ~255
    return {"max_nodes": mn, "max_edges": me, "table_size": ts, "off": off, "total": o}


def _device_array(t, L, name):
    """[n_trees, elements * bytes] uint8 view of one array of the workspace (device)"""
    o, per, b = L["off"][name]
    return t.workspace[o : o + t.n * per * b].view(t.n, per * b)


def read_tree(t, L):
    """Host copy of every tree (node arrays up to the largest n_nodes, edge arrays up to the largest n_edges), checked
    against the library's own accessors."""
    nn, ne, st = (x.cpu().numpy() for x in t.stats())
    mn, me = max(int(nn.max()), 1), max(int(ne.max()), 1)
    g = {"n_nodes": nn, "n_edges": ne, "status": st}
    for name, _, k in _ARRAYS:
        if name not in _NP:
            continue
        b = L["off"][name][2]
        lim = {"n": mn, "e": me, "s": L["table_size"]}[k]
        g[name] = _device_array(t, L, name)[:, : lim * b].cpu().numpy().copy().view(_NP[name])
    g["node_state"] = g["node_state"].reshape(t.n, mn, 32)
    for name in ("n_nodes", "n_edges"):    # the counters as the arena holds them
        assert np.array_equal(_device_array(t, L, name).cpu().numpy().view(np.int32)[:, 0], g[name])
    # root edges as hz_tree_root_edges reports them
    N, W, P, child = (x.cpu().numpy() for x in t.root_edges())
    for i in range(t.n):
        e0, k = int(g["node_edge0"][i, 0]), int(g["node_info"][i, 0] & 0xFF)
        a = g["edge_am"][i, e0 : e0 + k] & 0xFF
        want = {"N": np.zeros(143, np.int32), "W": np.zeros(143), "P": np.zeros(143, np.float32), "c": np.full(143, -1, np.int32)}
        want["N"][a], want["W"][a], want["P"][a] = g["edge_N"][i, e0 : e0 + k], g["edge_W"][i, e0 : e0 + k], g["edge_P"][i, e0 : e0 + k]
        want["c"][a] = g["edge_child"][i, e0 : e0 + k]
        assert np.array_equal(want["N"], N[i]) and np.array_equal(want["c"], child[i]), i
        assert np.array_equal(want["W"].view(np.uint64), W[i].view(np.uint64)), i
        assert np.array_equal(want["P"].view(np.uint32), P[i].view(np.uint32)), i
    return g


def check_invariants(g, i, L):
    """What a finished step must leave in tree i, whatever the search did."""
    nn, ne = int(g["n_nodes"][i]), int(g["n_edges"][i])
    info, e0 = g["node_info"][i, :nn], g["node_edge0"][i, :nn]
    assert (g["edge_V"][i, :ne] == 0).all(), "in-flight visits left on edges"
    child = g["edge_child"][i, :ne]
    assert (child < nn).all()
    ci = g["edge_cinfo"][i, :ne]
    known = ci != 0
    assert np.array_equal(ci[known], e0[child[known]] | ((info[child[known]] & 0xFF) << 24)), "stale child cache"
    # the hash table: each node once, under its own key, reachable from key & mask without an empty slot on the way
    tab, th = g["table"][i], g["table_hash"][i]
    ts = L["table_size"]
    slots = np.nonzero(tab)[0]
    ids = tab[slots].astype(np.int64) - 1
    assert np.array_equal(np.sort(ids), np.arange(nn)), "table does not list every node exactly once"
    keys = g["node_hash"][i, ids]
    assert np.array_equal(th[slots], keys)
    home = (keys & np.uint64(ts - 1)).astype(np.int64)
    dist = (slots - home) & (ts - 1)
    occ = np.concatenate([tab != 0, tab != 0])
    idx = np.arange(2 * ts)
    last_empty = np.maximum.accumulate(np.where(occ, -1, idx))[ts:]   # at or before slot s (cyclic): s + ts - run
    run = np.arange(ts, 2 * ts) - last_empty                         # occupied slots ending at s
    assert (dist < run[slots]).all(), "a node the linear probe cannot reach"


def compare_tree(g, i, r):
    """tree i of the device == the oracle's dump r (oracle.search(..., tree=True))"""
    o = r["tree"]
    nn, ne = int(g["n_nodes"][i]), int(g["n_edges"][i])
    assert (nn, ne) == (r["n_nodes"], r["n_edges"]), (nn, ne, r["n_nodes"], r["n_edges"])
    assert np.array_equal(g["node_state"][i, :nn], o["words"]), "node words"
    assert np.array_equal(g["node_hash"][i, :nn], o["hash"]), "node keys"
    info = g["node_info"][i, :nn]
    assert np.array_equal(g["node_edge0"][i, :nn], o["first_edge"].astype(np.uint32)), "first edges"
    assert np.array_equal(info & 0xFF, o["n_edges"].astype(np.uint32)), "edge counts"
    assert np.array_equal(info >> 8, o["player"].astype(np.uint32)), "players"
    assert np.array_equal(g["edge_child"][i, :ne], o["child"].astype(np.uint32)), "edge children"
    assert np.array_equal(g["edge_N"][i, :ne], o["N"]), "edge N"
    assert np.array_equal(g["edge_W"][i, :ne].view(np.uint64), o["W"].view(np.uint64)), "edge W bits"
    assert np.array_equal(g["edge_P"][i, :ne].view(np.uint32), o["P"].view(np.uint32)), "edge P bits"
    am = g["edge_am"][i, :ne]
    assert np.array_equal(am & 0xFF, o["action"].astype(np.uint16)), "edge actions"
    assert np.array_equal(am >> 8, o["mover"].astype(np.uint16)), "edge movers"
    assert (o["V"] == 0).all()


def test_layout_restatement_matches_the_library():
    from harmonies_alphazero_b200 import _lib

    lib = _lib.load()
    for n in (1, 3, 64, 1000):
        for sims in (1, 2, 33, 100, 2560):
            for mn in (0, 1, 40, 1000, 4097):
                for k in (1, 3, 8, 20, 64):
                    assert lib.hz_tree_workspace_bytes(n, sims, mn, k) == layout(n, sims, mn, k)["total"], (n, sims, mn, k)


# ---- evaluators: functions of the leaf's words only, so the oracle's call order does not matter ----------------------
def _legal_bits(oracle, w):
    m = oracle.legal_mask(w)
    return ((m[:, ACTIONS >> 5] >> (ACTIONS & 31).astype(np.uint32)) & 1).astype(bool)


def ev_chain(oracle):
    """one-hot prior on the highest legal action, value 0: the search walks one line to the end of the game"""
    def f(w):
        legal = _legal_bits(oracle, w)
        p = np.zeros((len(w), 143), np.float32)
        hi = 142 - np.argmax(legal[:, ::-1], axis=1)
        rows = np.nonzero(legal.any(axis=1))[0]
        p[rows, hi[rows]] = 1.0
        return p, np.zeros(len(w), np.float32)
    return f


STAIR = np.ldexp(np.ones(143, np.float32), -8 * (142 - ACTIONS))   # 2^-8(142-a): normals, subnormals (a = 124..126), zeros
ROWS = {"stair": STAIR, "zeros": np.zeros(143, np.float32), "equal": np.full(143, 2.0, np.float32)}
VALUES = np.array([1.0, -1.0, -0.0, 0.1, 0.0, -0.7], np.float32)


def ev_row(oracle, kind):
    """a constant prior row; value +-1, -0.0, 0.1f, 0 or -0.7f by the leaf's exact key"""
    def f(w):
        h = oracle.canon_hash(w, pk.KEY_EXACT)
        return np.repeat(ROWS[kind][None], len(w), axis=0), VALUES[(h % np.uint64(len(VALUES))).astype(np.int64)]
    return f


def _oracle_fn(f):
    def g(w):
        p, v = f(np.asarray(w, dtype=np.uint32)[None])
        return p[0], float(v[0])
    return g


# ---- one batch of searches, compared at checkpoints ------------------------------------------------------------------
def run_and_compare(mods, oracle, roots, skeys, sims, cpuct, *, leaves=1, key_mode=1, evals=None, noise=None, eps=0.0,
                    checkpoints=(), max_nodes=0, compare=None):
    """Runs len(roots) GPU searches of `sims` simulations, K = leaves per step.  evals: None (the synthetic evaluator on
    both sides) or one host evaluator per tree.  At each checkpoint s (and at the end) every tree i with compare[i] is
    compared with oracle.search(sims = s).  Returns (handle, last read of the arenas, longest path seen, the oracle's
    results of the final comparison by tree)."""
    hb, tr = mods
    n, K = len(roots), leaves
    assert sims % K == 0 and all(s % K == 0 for s in checkpoints)
    t = tr.BatchedMCTS(n, sims, key_mode=key_mode, leaves=K, max_nodes=max_nodes)
    L = layout(n, sims, max_nodes, K)
    assert t.workspace_bytes == L["total"]
    t.reset(hb.states_from_numpy(roots), tr.search_keys_tensor(skeys))
    nz = None if noise is None else torch.from_numpy(np.ascontiguousarray(noise, dtype=np.float32)).cuda()
    policy = torch.empty((t.rows, 143), dtype=torch.float32, device="cuda")
    value = torch.empty(t.rows, dtype=torch.float32, device="cuda")
    leaf = torch.empty((t.rows, 32), dtype=torch.int32, device="cuda")
    depth = _device_array(t, L, "depth").view(torch.int32)
    deepest = torch.zeros((), dtype=torch.int32, device="cuda")
    groups = None
    if evals is not None:
        groups = {}
        for i, f in enumerate(evals):
            groups.setdefault(f, []).append(i)
        groups = [(f, (np.array(ix)[:, None] * K + np.arange(K)).ravel()) for f, ix in groups.items()]
    compare = np.ones(n, bool) if compare is None else compare
    results = {}
    stops = sorted(set(checkpoints) | {sims})
    for step in range(sims // K):
        t.select(cpuct, leaf_states=leaf)
        deepest = torch.maximum(deepest, depth.max())
        if groups is None:
            t.fake_eval(policy, value)
        else:
            w = leaf.cpu().numpy().view(np.uint32)
            p = np.empty((t.rows, 143), np.float32)
            v = np.empty(t.rows, np.float32)
            for f, rows in groups:
                p[rows], v[rows] = f(w[rows])
            policy.copy_(torch.from_numpy(p))
            value.copy_(torch.from_numpy(v))
        t.expand_backup(policy, value, noise=nz, eps=eps)
        s = (step + 1) * K
        if s not in stops:
            continue
        g = read_tree(t, L)
        for i in range(n):
            if not compare[i]:
                continue
            r = oracle.search(roots[i], skeys[i], s, cpuct, None if noise is None else noise[i], eps,
                              eval_fn=None if evals is None else _oracle_fn(evals[i]), key_mode=key_mode, leaves=K, tree=True)
            assert r["rc"] == 0
            try:
                assert g["status"][i] == 0
                compare_tree(g, i, r)
                check_invariants(g, i, L)
            except AssertionError as e:
                raise AssertionError(f"tree {i} after {s} simulations (K = {K}, key mode {key_mode}, cpuct {cpuct}): {e}") from e
            results[i] = r
    return t, g, int(deepest.item()), results


def _mixed_roots(hb, n, seed, depths=(0, 6, 31, 52, 60)):
    st = hb.init_states(n, seed=seed)
    cuts = np.linspace(0, n, len(depths) + 1).astype(int)
    for lo, hi, d in zip(cuts[:-1], cuts[1:], depths):
        sl = st[lo:hi].clone()
        hb.playout(sl, max_steps=d)
        st[lo:hi] = sl
    return st.cpu().numpy().view(np.uint32).copy()


def _noise(rng, n):
    return rng.gamma(0.4, size=(n, 143)).astype(np.float32) + np.float32(1e-6)


CHECKS = (1, 2, 31, 32, 33, 64, 65)


@pytest.mark.gpu
@pytest.mark.parametrize("key_mode", [0, 1])
def test_ordinary_searches_node_for_node(mods, oracle, key_mode):
    """the synthetic evaluator on mixed-depth roots with root noise: today's scenario, every node and edge"""
    hb, _ = mods
    n = 128
    roots = _mixed_roots(hb, n, 300 + key_mode)
    rng = np.random.default_rng(key_mode)
    skeys = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    run_and_compare(mods, oracle, roots, skeys, 66, 2.0, key_mode=key_mode, noise=_noise(rng, n), eps=0.25, checkpoints=CHECKS)


@pytest.mark.gpu
@pytest.mark.parametrize("key_mode", [0, 1])
def test_deep_chains_back_up_past_the_warp(mods, oracle, key_mode):
    """one line of play to the end of the game: back_fill runs with depth >= 65 (edges 32.. and 64.. of the path take
    the loop after the warp-wide update)"""
    hb, _ = mods
    n = 16
    roots = _mixed_roots(hb, n, 410 + key_mode, depths=(0, 0, 0, 6))
    skeys = np.arange(n, dtype=np.uint64) + 5000
    f = ev_chain(oracle)
    _, _, deepest, _ = run_and_compare(mods, oracle, roots, skeys, 160, 2.0, key_mode=key_mode, evals=[f] * n,
                                       checkpoints=CHECKS + (96, 127, 128, 129))
    assert deepest >= 65, deepest


@pytest.mark.gpu
@pytest.mark.parametrize("leaves", [8, 64])
def test_deep_chains_under_virtual_loss(mods, oracle, leaves):
    """K in-flight descents per step follow the same line (cpuct 1e4 outweighs the virtual loss): paths past 32 edges
    with in-flight visits to land on every edge"""
    hb, _ = mods
    n = 8
    roots = _mixed_roots(hb, n, 420 + leaves, depths=(0, 0, 0, 4))
    skeys = np.arange(n, dtype=np.uint64) * 7 + 11
    sims = 40 * leaves
    f = ev_chain(oracle)
    _, _, deepest, _ = run_and_compare(mods, oracle, roots, skeys, sims, 1e4, leaves=leaves, key_mode=int(leaves == 8),
                                       evals=[f] * n, checkpoints=(leaves, 2 * leaves, 33 * leaves, 34 * leaves))
    assert deepest >= 33, deepest


@pytest.mark.gpu
@pytest.mark.parametrize("leaves,sims", [(3, 99), (20, 100), (32, 128)])
def test_wide_virtual_loss_node_for_node(mods, oracle, leaves, sims):
    """K = 3 (not a power of two), 20 and 32 with the synthetic evaluator and root noise"""
    hb, _ = mods
    n = 64
    roots = _mixed_roots(hb, n, 430 + leaves)
    rng = np.random.default_rng(leaves)
    skeys = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    checks = [s for s in range(leaves, sims + 1, leaves) if s in (leaves, 2 * leaves) or s // 32 != (s - leaves) // 32]
    run_and_compare(mods, oracle, roots, skeys, sims, 2.0, leaves=leaves, key_mode=leaves % 2, noise=_noise(rng, n),
                    eps=0.25, checkpoints=checks)


@pytest.mark.gpu
@pytest.mark.parametrize("cpuct,eps,key_mode", [(0.0, 0.0, 1), (2.0, 1.0, 0), (3e38, 0.25, 1), (2.0, 0.0, 0)])
def test_degenerate_priors_and_values(mods, oracle, cpuct, eps, key_mode):
    """priors of exactly 0, subnormal priors (the build must not flush them), cpuct * P = inf (P = 2, cpuct 3e38),
    cpuct = 0, all-equal and all-zero rows (exact ties at every level); values +-1, -0.0, 0.1f; root noise with eps
    0 and 1 and a noise row with one non-zero legal entry"""
    hb, _ = mods
    kinds = ["stair", "zeros", "equal"]
    per = 6
    n = per * len(kinds)
    roots = _mixed_roots(hb, n, 440 + key_mode, depths=(0, 6, 31))
    skeys = np.arange(n, dtype=np.uint64) * 3 + int(cpuct % 97)
    rng = np.random.default_rng(int(eps * 8) + key_mode)
    noise = _noise(rng, n)
    legal = _legal_bits(oracle, roots)
    for i in range(0, n, 2):                                 # every other tree: one legal entry carries all the noise
        acts = np.nonzero(legal[i])[0]
        if len(acts):
            noise[i] = 0.0
            noise[i, acts[i % len(acts)]] = 0.75
    fs = {k: ev_row(oracle, k) for k in kinds}
    evals = [fs[kinds[i % len(kinds)]] for i in range(n)]
    run_and_compare(mods, oracle, roots, skeys, 66, cpuct, key_mode=key_mode, evals=evals, noise=noise, eps=eps,
                    checkpoints=(1, 2, 33, 65))


@pytest.mark.gpu
def test_exact_arena_fit(mods, oracle):
    """max_nodes = the smallest final tree of the batch: trees that fill the arena exactly are not flagged and equal the
    oracle node for node; every larger tree is flagged (status bit 0) and check_status raises"""
    hb, _ = mods
    n, sims = 48, 40
    roots = _mixed_roots(hb, n, 450, depths=(0, 6, 31))
    skeys = np.arange(n, dtype=np.uint64) + 99
    final = np.array([oracle.search(roots[i], skeys[i], sims, 2.0, key_mode=1)["n_nodes"] for i in range(n)])
    fit = int(final.min())
    exact = final == fit
    assert exact.any() and (~exact).any()
    t, g, _, _ = run_and_compare(mods, oracle, roots, skeys, sims, 2.0, checkpoints=(33,), max_nodes=fit, compare=exact)
    assert (g["n_nodes"][exact] == fit).all() and (g["status"][exact] == 0).all()
    assert (g["status"][~exact] & 1).all()
    with pytest.raises(RuntimeError):
        t.check_status()


@pytest.mark.gpu
def test_root_policy_and_choice_at_threshold_boundaries(mods, oracle):
    """hz_tree_root_policy: visits = N, pi = float32(N / sum N) bit for bit, zeros at a root without visits.
    hz_tree_choose == oracle.choose with exploratory flags mixed, at u = 0, every exact prefix fraction acc / sum N
    (65 simulations: sum N = 64, so the fractions are exact) and its float neighbours, nextafter(1, 0) and 1.0"""
    hb, _ = mods
    n, sims = 64, 65
    roots = _mixed_roots(hb, n - 2, 460, depths=(0, 6, 31, 52))
    over = hb.init_states(2, seed=461)
    hb.playout(over)                                          # two finished games: roots without visits
    roots = np.concatenate([roots, over.cpu().numpy().view(np.uint32)])
    skeys = np.arange(n, dtype=np.uint64) + 1
    t, g, _, res = run_and_compare(mods, oracle, roots, skeys, sims, 2.0, checkpoints=())
    visits, pi = (x.cpu().numpy() for x in t.root_policy())
    N = np.stack([res[i]["N"] for i in range(n)])
    assert np.array_equal(visits, N)
    tot = N.sum(axis=1, keepdims=True)
    want = np.where(tot > 0, N / np.maximum(tot, 1), 0.0).astype(np.float32)
    assert np.array_equal(pi.view(np.uint32), want.view(np.uint32))
    assert (tot[-2:] == 0).all() and (tot[:-2] == 64).all()
    one = np.float32(1.0)
    us = []
    for i in range(n):
        u = [np.float32(0.0), np.nextafter(one, np.float32(0.0)), one]
        for acc in np.cumsum(N[i][N[i] > 0]):
            x = np.float32(acc / max(int(tot[i, 0]), 1))
            u += [x, np.nextafter(x, np.float32(0.0)), np.nextafter(x, np.float32(2.0))]
        us.append(u)
    width = max(len(u) for u in us)
    expl = (np.arange(n) % 3 != 0).astype(np.uint8)
    expl_t = torch.from_numpy(expl).cuda()
    for j in range(width):
        u = np.array([us[i][min(j, len(us[i]) - 1)] for i in range(n)], np.float32)
        a = t.choose(torch.from_numpy(u).cuda(), expl_t).cpu().numpy()
        want = [oracle.choose(N[i], float(u[i]), bool(expl[i])) for i in range(n)]
        assert np.array_equal(a, want), (j, np.nonzero(a != want)[0])
    greedy = t.choose().cpu().numpy()
    assert np.array_equal(greedy, [oracle.choose(N[i]) for i in range(n)])
