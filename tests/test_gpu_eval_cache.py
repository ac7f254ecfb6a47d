"""The leaf evaluation cache (tree.EvalCache, hz_tree_select_cached / hz_evalcache_fill) on the GPU.

A hit must return the bits the evaluator would return, so every search, self-play game and arena match must be
bit-identical with the cache on or off.  That rests on the evaluator being row-invariant, which is checked first for the
tile path of the default network."""

import pytest
import torch

from tests.conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    from harmonies_alphazero_b200 import arena, batched, net, selfplay, tree

    return batched, net, selfplay, tree, arena


def _default_net(net, weights, seed=0):
    from oracle import synth_weights

    model = net.AlphaZeroNet.from_config(net.DEFAULT_MODEL_CONFIG)
    if weights == "golden":
        synth_weights.fill_(model, int(load_golden("net_default")["seed"]))
    else:
        torch.manual_seed(seed)
    return net.InferenceNet(model.eval(), device="cuda")


class ElementwiseNet:
    """Exact row-wise function of the encoded leaf: bitwise independent of the batch shape and the row."""

    dtype, device, row_invariant = torch.float32, torch.device("cuda"), True

    def __call__(self, board, glob, out=None):
        a = torch.arange(143, device=glob.device, dtype=torch.float32)
        x = glob[:, 36:42].repeat(1, 24)[:, :143] * 3.0 + glob[:, 30:36].repeat(1, 24)[:, :143]
        logits = torch.sin(a * 0.37 + x * 5.0) + board[:, 36, 2, 3].unsqueeze(1) * torch.cos(a) + board[:, 3].sum(dim=(1, 2)).unsqueeze(1)
        value = torch.tanh(glob[:, 36] * 3.0 - glob[:, 41] * 2.0 - glob[:, 33] + board[:, 5].sum(dim=(1, 2)) * 0.1)
        if out is None:
            return logits, value
        out[0].copy_(logits)
        out[1].copy_(value)
        return out


def _positions(hb, n, seed):
    st = hb.init_states(n, seed=seed)
    hb.playout(st[: n // 2], max_steps=40)
    hb.playout(st[n // 2:], max_steps=110)
    return st


@pytest.mark.parametrize("weights", ["random", "golden"])
def test_tile_path_is_row_invariant(mods, weights):
    """The precondition: a board's logits and value do not depend on its row, its neighbours or the active count."""
    hb, net, _, _, _ = mods
    inf = _default_net(net, weights)
    assert inf.row_invariant and inf.wants_tiles
    N = 4096
    st = _positions(hb, N, seed=5)
    b, g = hb.encode(st, dtype=torch.bfloat16, channels_last=True)
    b40 = torch.zeros((N, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    b40[:, :38] = b

    def run(order, n_active):
        x0 = inf.hand.x0_buffer(N)
        inf.hand.to_tiles(b40[order].contiguous(memory_format=torch.channels_last), 40, True, x0)
        out = (torch.full((N, 143), float("nan"), device="cuda"), torch.full((N,), float("nan"), device="cuda"))
        na = None if n_active is None else torch.tensor([n_active], dtype=torch.int32, device="cuda")
        inf.forward_tiles(x0, g[order].contiguous(), N, out=out, n_active=na)
        return out

    ref_l, ref_v = run(torch.arange(N, device="cuda"), None)
    gen = torch.Generator(device="cuda").manual_seed(3)
    for n_act in (1, 15, 16, 17, 4095, 4096):
        order = torch.randperm(N, device="cuda", generator=gen)
        l, v = run(order, n_act)
        sel = order[:n_act]
        assert torch.equal(l[:n_act].view(torch.int32), ref_l[sel].view(torch.int32)), n_act
        assert torch.equal(v[:n_act].view(torch.int32), ref_v[sel].view(torch.int32)), n_act


# ---- search chains along real games --------------------------------------------------------------------------------

def _layout_buffers(kind, rows, inf=None):
    if kind == "tiles":
        board, glob, _, _ = inf.leaf_buffers(rows)
        return board, glob, dict(dtype=torch.bfloat16, tiles=True)
    C = 40 if kind == "nhwc40" else 38
    mf = torch.contiguous_format if kind == "nchw" else torch.channels_last
    board = torch.zeros((rows, C, 5, 7), dtype=torch.float32, device="cuda").contiguous(memory_format=mf)
    glob = torch.zeros((rows, 42), dtype=torch.float32, device="cuda")
    return board, glob, dict(dtype=torch.float32, channels_last=kind != "nchw", pad40=kind == "nhwc40")


class _Searcher:
    """One tree (+ cache) that runs whole searches with the network evaluator of a layout kind."""

    def __init__(self, mods, net, kind, n, sims, key_mode, K, sym, entries):
        _, _, _, tr, _ = mods
        self.net, self.kind, self.sims, self.K = net, kind, sims, K
        self.t = tr.BatchedMCTS(n, sims, key_mode=key_mode, leaves=K)
        self.t.set_symmetry(sym)
        rows = n * K
        self.board, self.glob, self.kw = _layout_buffers(kind, rows, net if kind == "tiles" else None)
        z = lambda *s: torch.zeros(s, dtype=torch.float32, device="cuda")  # noqa: E731
        self.policy, self.value, self.nl, self.nv = z(rows, 143), z(rows), z(rows, 143), z(rows)
        self.eval_rows = torch.zeros(rows, dtype=torch.int32, device="cuda")
        self.n_eval = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.cache = tr.EvalCache(entries, rows) if entries else None

    def evaluate(self, out, n_active=None):
        if self.kind == "tiles":
            self.net.forward_tiles(self.board, self.glob, self.glob.shape[0], out=out, n_active=n_active)
        else:
            self.net(self.board, self.glob, out=out)

    def step(self, noise, on_select=None):
        t = self.t
        if self.cache is None:
            t.select(2.0, self.board, self.glob, **self.kw)
            self.evaluate((self.policy, self.value))
        else:
            t.select_cached(self.cache, 2.0, self.board, self.glob, self.policy, self.value, self.eval_rows, self.n_eval,
                            leaf_states=self.leaf_states if on_select else None, **self.kw)
            if on_select:
                on_select()
            self.evaluate((self.nl, self.nv), self.n_eval)
            self.cache.fill(self.nl, self.nv, self.eval_rows, self.n_eval, self.policy, self.value)
        t.expand_backup(self.policy, self.value, is_logits=True, noise=noise, eps=0.25 if noise is not None else 0.0)

    def search(self, roots, noise, on_select=None):
        self.t.reset(roots)
        for _ in range(self.sims // self.K):
            self.step(noise, on_select)


def _snapshot(t):
    N, W, P, child = t.root_edges()
    visits, pi = t.root_policy()
    return N, W.view(torch.int64), P.view(torch.int32), child, visits, pi.view(torch.int32), t.choose()


def _chain(mods, net, kind, key_mode, K, noise, sym, entries, n=48, sims=32, moves=60, seed=1):
    hb = mods[0]
    off = _Searcher(mods, net, kind, n, sims, key_mode, K, sym, 0)
    on = _Searcher(mods, net, kind, n, sims, key_mode, K, sym, entries)
    roots = hb.init_states(n, seed=seed)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for mv in range(moves):
        nz = torch.rand((n, 143), device="cuda", generator=gen).add_(1e-3) if noise else None
        off.search(roots, nz)
        on.search(roots, nz)
        a, b = _snapshot(off.t), _snapshot(on.t)
        for x, y in zip(a, b):
            assert torch.equal(x, y), f"move {mv}"
        over, _ = hb.outcome(roots)
        if bool(over.bool().all()):
            break
        acts = a[-1]
        acts = torch.where(acts < 0, hb.random_actions(roots), acts)
        hb.apply(roots, torch.where(over.bool(), torch.full_like(acts, -1), acts))
    on.t.check_status()
    return on.cache.stats()


CHAINS = [
    # evaluator/layout, key mode, K, root noise, symmetry
    ("nchw", "reference", 1, False, None),
    ("nhwc", "exact", 4, True, "board"),
    ("nhwc40", "reference", 1, True, "full"),
    ("nhwc40", "exact", 1, False, None),
    ("tiles", "reference", 1, True, None),
    ("tiles", "exact", 4, False, "board"),
    ("tiles", "reference", 4, True, "full"),
]


@pytest.mark.parametrize("kind,key,K,noise,sym", CHAINS)
def test_search_chains_identical_with_cache(mods, kind, key, K, noise, sym):
    hb, net = mods[0], mods[1]
    ev = _default_net(net, "random", seed=2) if kind == "tiles" else ElementwiseNet()
    key_mode = hb.KEY_REFERENCE if key == "reference" else hb.KEY_EXACT
    st = _chain(mods, ev, kind, key_mode, K, noise, sym, entries=1 << 18)
    assert st["looked_up"] == st["hits"] + st["terminal"] + st["misses"] and st["inserts"] <= st["misses"]
    if sym != "full":
        assert st["hits"] > 0 and st["terminal"] > 0


def test_tiny_cache_evicts_and_stays_identical(mods):
    hb = mods[0]
    st = _chain(mods, ElementwiseNet(), "nhwc40", hb.KEY_REFERENCE, 1, True, None, entries=64, moves=40)
    assert st["evictions"] > 0 and st["hits"] > 0


def test_counters_match_a_host_recount(mods):
    """hits = rows whose (exact key, frame) an earlier step inserted since the last clear; terminal = rows whose leaf is
    over; hits + misses + terminal = active rows; with room to spare nothing is evicted."""
    hb = mods[0]
    for sym in (None, "board"):
        n, sims = 32, 16
        s = _Searcher(mods, ElementwiseNet(), "nhwc", n, sims, hb.KEY_REFERENCE, 1, sym, 1 << 18)
        s.leaf_states = torch.zeros((n, 32), dtype=torch.int32, device="cuda")
        seen, tally = set(), dict(hits=0, terminal=0, misses=0)

        def on_select():
            keys = hb.canon_hash(s.leaf_states, hb.KEY_EXACT).cpu().numpy()
            frames = s.t.leaf_frames().cpu().numpy()
            over = hb.outcome(s.leaf_states)[0].cpu().numpy()
            fresh, misses = set(), 0
            for r in range(n):
                if over[r]:
                    tally["terminal"] += 1
                elif (int(keys[r]), int(frames[r])) in seen:
                    tally["hits"] += 1
                else:
                    tally["misses"] += 1
                    misses += 1
                    fresh.add((int(keys[r]), int(frames[r])))     # two trees at one leaf in a step: both miss
            assert int(s.n_eval.item()) == misses
            step_misses.append(misses)
            seen.update(fresh)

        step_misses = []
        roots = hb.init_states(n, seed=4)
        hb.playout(roots[: n // 2], max_steps=120)       # half the roots near the end: terminal leaves
        for mv in range(12):
            s.search(roots, None, on_select)
            acts = s.t.choose()
            over = hb.outcome(roots)[0].bool()
            acts = torch.where(acts < 0, hb.random_actions(roots), acts)
            hb.apply(roots, torch.where(over, torch.full_like(acts, -1), acts))
        st = s.cache.stats()
        assert st["looked_up"] == n * sims * 12
        assert st["hits"] == tally["hits"] and st["terminal"] == tally["terminal"] and st["misses"] == tally["misses"] == sum(step_misses)
        assert st["inserts"] == st["misses"] and st["evictions"] == 0 and st["hits"] > 0 and st["terminal"] > 0
        s.cache.clear()
        assert all(v == 0 for v in s.cache.stats().values())


# ---- whole games ----------------------------------------------------------------------------------------------------

def _same_traj(a, b):
    oa = torch.argsort(a.game_id * 1000 + a.move_no.to(torch.int64))
    ob = torch.argsort(b.game_id * 1000 + b.move_no.to(torch.int64))
    for x, y in ((a.states, b.states), (a.visits, b.visits), (a.z, b.z), (a.game_id, b.game_id), (a.move_no, b.move_no)):
        assert torch.equal(x[oa], y[ob])


def test_selfplay_identical_with_cache(mods):
    _, net, sp, _, _ = mods
    inf = _default_net(net, "random", seed=7)
    for streams in (1, 2):
        base = dict(n_slots=48, num_simulations=16, seed=9, n_streams=streams)
        off = sp.BatchedSelfPlay(inf, sp.SelfPlayConfig(**base))
        on = sp.BatchedSelfPlay(inf, sp.SelfPlayConfig(**base, eval_cache=1 << 16))
        torch.manual_seed(5)
        a = off.play(72)
        torch.manual_seed(5)
        b = on.play(72)
        _same_traj(a, b)
        st = b.stats["eval_cache"]
        assert st["hits"] > 0 and st["looked_up"] == st["hits"] + st["terminal"] + st["misses"] and 0 < st["hit_rate"] < 1
        if streams == 1:       # new weights between calls: no stale hits
            torch.manual_seed(11)
            other = net.AlphaZeroNet.from_config(net.DEFAULT_MODEL_CONFIG).eval()
            inf.load(other)
            torch.manual_seed(6)
            a2 = off.play(40)
            torch.manual_seed(6)
            b2 = on.play(40)
            _same_traj(a2, b2)


def test_arena_identical_with_cache(mods):
    _, net, _, _, arena = mods
    cand, best = _default_net(net, "random", seed=1), _default_net(net, "random", seed=2)
    cfg = {"num_simulations": 16, "cpuct": 2.0}
    a = arena.play_match(cand, best, 6, cfg, seed=3)
    b = arena.play_match(cand, best, 6, cfg, seed=3, eval_cache=1 << 14)
    assert a == b
    a = arena.play_match(cand, arena.GREEDY, 4, cfg, seed=4, symmetry="board")
    b = arena.play_match(cand, arena.GREEDY, 4, cfg, seed=4, symmetry="board", eval_cache=1 << 14)
    assert a == b


def test_cache_rejects_evaluators_it_cannot_serve(mods):
    _, net, sp, tr, arena = mods
    model = net.AlphaZeroNet.from_config(net.DEFAULT_MODEL_CONFIG).eval()
    cudnn = net.InferenceNet(model, device="cuda", tower="cudnn")
    assert not cudnn.row_invariant
    cfg = sp.SelfPlayConfig(n_slots=8, num_simulations=4, eval_cache=1024)
    for ev in (cudnn, sp.SyntheticEvaluator(), sp.RolloutEvaluator(4)):
        with pytest.raises(ValueError):
            sp.BatchedSelfPlay(ev, cfg)
    with pytest.raises(ValueError):
        arena.play_match(sp.RolloutEvaluator(4), arena.GREEDY, 2, {"num_simulations": 4, "cpuct": 2.0}, eval_cache=1024)
    with pytest.raises(ValueError):
        arena.play_match(cudnn, arena.GREEDY, 2, {"num_simulations": 4, "cpuct": 2.0}, eval_cache=1024)
    with pytest.raises(ValueError):
        tr.EvalCache(100, 16)
    # a tree with more leaf rows than the cache was sized for is refused
    t = tr.BatchedMCTS(8, 4, leaves=2)
    c = tr.EvalCache(64, 8)
    t.reset(mods[0].init_states(8))
    board, glob, kw = _layout_buffers("nchw", 16)
    z = torch.zeros((16, 143), device="cuda")
    with pytest.raises(Exception):
        t.select_cached(c, 2.0, board, glob, z, z[:, 0].contiguous(), torch.zeros(16, dtype=torch.int32, device="cuda"),
                        torch.zeros(1, dtype=torch.int32, device="cuda"), **kw)
