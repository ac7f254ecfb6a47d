"""GPU: the game's symmetries — hz_sym_states / hz_sym_actions against the numpy reference, the engine's equivariance
on a large batch, and random-frame leaf evaluation in the search (hz_tree_set_symmetry): frame-free evaluators give
the same search with the mode on or off, a frame-dependent evaluator gives what oracle.search gives when its evaluator
applies the same frame rule, and self-play, the arena and the replay ring's augmented batches work end to end."""

import numpy as np
import pytest
import torch

from harmonies_alphazero_b200 import symmetry as sy
from tests.conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    from harmonies_alphazero_b200 import _lib, batched, selfplay, tree

    _lib.load()
    return batched, tree, selfplay


def _host(t):
    return t.cpu().numpy().view(np.uint32)


def _reachable(hb, n, seed):
    """n records at game depths 0..~150 (a spread of playout caps), terminal ones included"""
    st = hb.init_states(n, seed=seed)
    caps = torch.arange(n, device="cuda") % 160
    for d in sorted(set(caps.tolist())):
        idx = torch.nonzero(caps == d).flatten()
        sl = st[idx].contiguous()
        hb.playout(sl, max_steps=d)
        st[idx] = sl
    return st


def _fewer_piles(words, rng):
    """gap-free records with m < 5: piles beyond a random m cleared and n_piles set to m"""
    w = np.array(words, dtype=np.uint32)
    m = rng.integers(0, 5, len(w))
    for i in range(len(w)):
        codes = [w[i, 18] & 0xFFFF, w[i, 18] >> 16, w[i, 19] & 0xFFFF, w[i, 19] >> 16, w[i, 20] & 0xFFFF]
        codes = [c if k < m[i] else 0 for k, c in enumerate(codes)]
        w[i, 18] = codes[0] | (codes[1] << 16)
        w[i, 19] = codes[2] | (codes[3] << 16)
        w[i, 20] = codes[4] | (w[i, 20] & 0xFFFF0000)
        w[i, 22] = (w[i, 22] & 0xFF00FFFF) | (int(m[i]) << 16)
    return w


def _mask_bits(mask):
    """int32 [n,5] mask words -> int16 [n,143] 0/1 rows"""
    a = torch.arange(143, device=mask.device)
    return ((mask[:, a >> 5] >> (a & 31)) & 1).to(torch.int16)


# ---- hz_sym_states / hz_sym_actions -------------------------------------------------------------
def test_sym_states_all_elements(mods):
    hb, _, _ = mods
    rng = np.random.default_rng(3)
    reach = _host(_reachable(hb, 320, 17))
    over = _host(_reachable(hb, 64, 18))
    st = hb.states_from_numpy(over)
    hb.playout(st)                                                         # terminal records
    base = np.concatenate([reach, _fewer_piles(reach[:160], rng), _host(st), np.unique(load_golden("weird")["states"], axis=0)[:64]])
    words = np.repeat(base, 480, axis=0)
    g = np.tile(np.arange(480), len(base))
    want = sy.transform_words(words, g)
    x = hb.states_from_numpy(words)
    sym = torch.from_numpy(g).cuda()
    got = sy.transform_states(x, sym)
    assert np.array_equal(_host(got), want)
    assert np.array_equal(_host(x), words)                                 # input untouched
    sy.transform_states(x, sym, out=x)                                     # in place
    assert np.array_equal(_host(x), want)
    # the inverse element undoes it
    m = sy.n_piles_of(words)
    inv = torch.tensor([sy.inverse(int(a), int(b)) for a, b in zip(g[::97], m[::97])], device="cuda")
    back = sy.transform_states(x[::97].contiguous(), inv)
    assert np.array_equal(_host(back), words[::97])
    # n = 0, null pointers
    from harmonies_alphazero_b200 import _lib

    lib = _lib.load()
    assert lib.hz_sym_states(None, 0, None, None, None) == 0
    assert lib.hz_sym_states(None, 4, sym.data_ptr(), x.data_ptr(), None) == -1
    assert lib.hz_sym_states(x.data_ptr(), 4, None, x.data_ptr(), None) == -1
    assert lib.hz_sym_states(x.data_ptr(), 4, sym.data_ptr(), None, None) == -1


@pytest.mark.parametrize("dtype", [torch.float32, torch.int16, torch.int32])
def test_sym_actions(mods, dtype):
    hb, _, _ = mods
    rng = np.random.default_rng(5)
    reach = _host(_reachable(hb, 512, 21))
    words = np.concatenate([reach, _fewer_piles(reach[:256], rng)])
    n = len(words)
    g = rng.integers(0, 480, n)
    g[:480] = np.arange(480)
    states = hb.states_from_numpy(words)
    if dtype == torch.float32:
        xh = rng.standard_normal((n, 143)).astype(np.float32)
    else:
        xh = rng.integers(-30000, 30000, (n, 143)).astype(np.int16 if dtype == torch.int16 else np.int32)
    x = torch.from_numpy(xh).cuda()
    sym = torch.from_numpy(g).cuda()
    y = sy.transform_actions(x, sym, states)
    want = sy.transform_action_rows(xh, g, sy.n_piles_of(words))
    assert np.array_equal(y.cpu().numpy(), want)
    assert torch.equal(sy.transform_actions(y, sym, states, inverse=True), x)
    assert np.array_equal(sy.transform_actions(x, sym, states, inverse=True).cpu().numpy(),
                          sy.transform_action_rows(xh, g, sy.n_piles_of(words), inverse_=True))
    # a legal mask maps to the legal mask of the transformed state
    ts = sy.transform_states(states, sym)
    bits = _mask_bits(hb.legal_mask(states)).to(dtype)
    assert torch.equal(sy.transform_actions(bits, sym, states), _mask_bits(hb.legal_mask(ts)).to(dtype))
    assert torch.equal(sy.transform_actions(bits, sym, ts), _mask_bits(hb.legal_mask(ts)).to(dtype))   # n_piles is frame-free
    if dtype == torch.float32:
        from harmonies_alphazero_b200 import _lib

        lib = _lib.load()
        out = torch.empty_like(x)
        assert lib.hz_sym_actions(x.data_ptr(), n, 1, sym.to(torch.int16).data_ptr(), states.data_ptr(), 0, out.data_ptr(), None) == -1
        assert lib.hz_sym_actions(x.data_ptr(), n, 7, sym.to(torch.int16).data_ptr(), states.data_ptr(), 0, out.data_ptr(), None) == -1
        assert lib.hz_sym_actions(x.data_ptr(), n, 0, None, states.data_ptr(), 0, out.data_ptr(), None) == -1
        assert lib.hz_sym_actions(x.data_ptr(), n, 0, sym.to(torch.int16).data_ptr(), None, 0, out.data_ptr(), None) == -1
        assert lib.hz_sym_actions(None, 0, 0, None, None, 0, None, None) == 0


# ---- engine equivariance on a large batch -------------------------------------------------------
def _cell_perm_table():
    from harmonies_alphazero_b200 import constants as K

    t = np.tile(np.arange(35), (4, 1))
    for b in range(4):
        for i, (y, x) in enumerate(K.HEX_CELL):
            yy, xx = K.HEX_CELL[sy.HEX_MAPS[b][i]]
            t[b, y * 7 + x] = yy * 7 + xx
    return torch.from_numpy(t).cuda()


def test_engine_equivariance_large_batch(mods):
    hb, _, _ = mods
    n = 65536
    s = _reachable(hb, n, 99)
    g = torch.randint(0, 480, (n,), device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    ts = sy.transform_states(s, g)
    # legal masks and scores
    assert torch.equal(sy.transform_actions(_mask_bits(hb.legal_mask(s)), g, s), _mask_bits(hb.legal_mask(ts)))
    assert torch.equal(hb.score(s), hb.score(ts))
    assert all(torch.equal(a, b) for a, b in zip(hb.outcome(s), hb.outcome(ts)))
    # encodes: cells follow the hexes, pile blocks follow the piles
    cp = _cell_perm_table()[(g & 3).long()]                                # [n, 35]
    ident = torch.arange(143, dtype=torch.int32, device="cuda").expand(n, 143).contiguous()
    src_pile = sy.transform_actions(ident, g, s)[:, :5].long()             # new pile position j holds old pile src[j]
    gidx = torch.arange(42, device="cuda").expand(n, 42).clone()
    for j in range(5):
        for t in range(6):
            gidx[:, 6 * j + t] = 6 * src_pile[:, j] + t
    for dtype in (torch.float32, torch.bfloat16):
        for cl in (False, True):
            b, gl = hb.encode(s, dtype=dtype, channels_last=cl)
            tb, tgl = hb.encode(ts, dtype=dtype, channels_last=cl)
            b, tb = b.reshape(n, 38, 35), tb.reshape(n, 38, 35)
            want = torch.empty_like(b).scatter_(2, cp[:, None, :].expand(n, 38, 35), b)
            assert torch.equal(tb, want), (dtype, cl)
            assert torch.equal(tgl, torch.gather(gl, 1, gidx)), (dtype, cl)
    # apply: apply(T s, sigma a) against T apply(s, a)
    a = hb.random_actions(s)
    live = a >= 0
    s, ts, g, a = s[live].contiguous(), ts[live].contiguous(), g[live].contiguous(), a[live].contiguous()
    onehot = torch.zeros((len(a), 143), dtype=torch.int32, device="cuda")
    onehot[torch.arange(len(a), device="cuda"), a.long()] = 1
    for board_only in (True, False):
        gg = (g & 3) if board_only else g
        tsg = sy.transform_states(s, gg)
        ta = sy.transform_actions(onehot, gg, s).argmax(dim=1).to(torch.int16)
        after = s.clone()
        assert int(hb.apply(after, a).max()) == 0
        got = tsg.clone()
        assert int(hb.apply(got, ta).max()) == 0
        want = sy.transform_states(after, gg)
        if board_only:
            assert torch.equal(got, want)
            continue
        keep = [w for w in range(32) if w not in (18, 19, 20)]
        assert torch.equal(got[:, keep], want[:, keep])
        assert torch.equal(got[:, 20] >> 16, want[:, 20] >> 16)             # the hand

        def piles(x):
            c = torch.stack([x[:, 18] & 0xFFFF, (x[:, 18] >> 16) & 0xFFFF, x[:, 19] & 0xFFFF, (x[:, 19] >> 16) & 0xFFFF,
                             x[:, 20] & 0xFFFF], dim=1)
            return torch.sort(c, dim=1).values

        assert torch.equal(piles(got), piles(want))
        assert not torch.equal(got, want)


# ---- the search -----------------------------------------------------------------------------------
def _roots(hb, n, seed):
    st = hb.init_states(n, seed=seed)
    caps = [0, 1, 5, 12, 31, 52]
    for k, d in enumerate(caps):
        lo, hi = n * k // len(caps), n * (k + 1) // len(caps)
        sl = st[lo:hi].clone()
        hb.playout(sl, max_steps=d)
        st[lo:hi] = sl
    return st


def _edges(t):
    return [x.cpu().numpy() for x in t.root_edges()]


def _same_edges(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))


@pytest.mark.parametrize("key_mode", [0, 1])
@pytest.mark.parametrize("leaves", [1, 4])
def test_frame_free_evaluators_give_the_same_search(mods, key_mode, leaves):
    hb, tr, _ = mods
    n, sims = 192, 24
    roots = _roots(hb, n, 40 + key_mode)
    keys = tr.search_keys_tensor(np.arange(n, dtype=np.uint64) * 7 + 3)
    nz = torch.from_numpy(np.random.default_rng(leaves).gamma(0.4, size=(n, 143)).astype(np.float32) + 1e-6).cuda()

    def run(mode, evaluator):
        t = tr.BatchedMCTS(n, sims, key_mode=key_mode, leaves=leaves)
        t.set_symmetry(mode)
        t.reset(roots, keys)
        policy = torch.empty((t.rows, 143), device="cuda")
        value = torch.empty(t.rows, device="cuda")
        for _ in range(sims // leaves):
            t.select(2.0)
            if evaluator == "fake":
                t.fake_eval(policy, value)
            else:
                t.rollout_eval(policy, value, 4)
            t.expand_backup(policy, value, noise=nz, eps=0.25)
        t.check_status()
        return _edges(t), [x.cpu().numpy() for x in t.stats()[:2]]

    for evaluator in ("fake", "rollout"):
        off = run(None, evaluator)
        for mode in ("board", "full"):
            on = run(mode, evaluator)
            _same_edges(off[0], on[0])
            _same_edges(off[1], on[1])


# A frame-dependent evaluator whose outputs are exact dyadic functions of (board, glob): integer features (the 37
# 0/1 planes of the tile bits and the player, and 3 x the 36 pile / hand features) times a fixed integer matrix.
_W = np.random.default_rng(2024).integers(0, 4, size=(37 * 35 + 36, 144)).astype(np.float64)


def _features_np(board, glob):
    n = board.shape[0]
    return np.concatenate([board[:, :37].reshape(n, -1).astype(np.float64), np.rint(glob[:, :36].astype(np.float64) * 3)], axis=1)


def _eval_np(board, glob):
    s = _features_np(board, glob) @ _W
    p = ((1 + np.fmod(s[:, :143], 64)) * 2.0 ** -7).astype(np.float32)
    v = ((np.fmod(s[:, 143], 255) - 127) / 128).astype(np.float32)
    return p, v


def _eval_torch(board, glob, W):
    n = board.shape[0]
    f = torch.cat([board[:, :37].reshape(n, -1).to(torch.float64), torch.round(glob[:, :36].to(torch.float64) * 3)], dim=1)
    s = f @ W
    p = ((1 + torch.fmod(s[:, :143], 64)) * 2.0 ** -7).to(torch.float32)
    v = ((torch.fmod(s[:, 143], 255) - 127) / 128).to(torch.float32)
    return p.contiguous(), v.contiguous()


def _framed_search(hb, tr, roots, skeys, sims, leaves, mode, noise, eps, key_mode=1):
    n = roots.shape[0]
    t = tr.BatchedMCTS(n, sims, key_mode=key_mode, leaves=leaves)
    t.set_symmetry(mode)
    t.reset(roots, tr.search_keys_tensor(skeys))
    W = torch.from_numpy(_W).cuda()
    board = torch.zeros((t.rows, 38, 5, 7), device="cuda")
    glob = torch.zeros((t.rows, 42), device="cuda")
    for _ in range(sims // leaves):
        t.select(2.0, board, glob)
        p, v = _eval_torch(board, glob, W)
        t.expand_backup(p, v, noise=noise, eps=eps)
    t.check_status()
    return t


@pytest.mark.parametrize("mode", ["board", "full"])
@pytest.mark.parametrize("leaves", [1, 4])
def test_framed_search_matches_oracle(mods, oracle, mode, leaves):
    hb, tr, _ = mods
    n, sims, eps = 48, 24, 0.25
    roots = _roots(hb, n, 7 + leaves)
    rng = np.random.default_rng(leaves)
    skeys = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    noise = rng.gamma(0.4, size=(n, 143)).astype(np.float32) + np.float32(1e-6)
    t = _framed_search(hb, tr, roots, skeys, sims, leaves, mode, torch.from_numpy(noise).cuda(), eps)
    N, W, P, _ = _edges(t)
    nn, ne, _ = (x.cpu().numpy() for x in t.stats())
    rh = _host(roots)
    for i in range(n):
        def eval_fn(w, sk=int(skeys[i])):
            w = np.array(w, dtype=np.uint32)
            g = sy.leaf_frame(w, sk, mode)
            b, gl = oracle.encode(sy.transform_words(w, g))
            p, v = _eval_np(b, gl)
            return sy.transform_action_rows(p[0], g, sy.n_piles_of(w)[0], inverse_=True), float(v[0])

        r = oracle.search(rh[i], skeys[i], sims, 2.0, noise[i], eps, eval_fn=eval_fn, key_mode=1, leaves=leaves)
        assert np.array_equal(N[i], r["N"]), i
        assert np.array_equal(W[i], r["W"]), i
        assert np.array_equal(P[i].view(np.uint32), r["P"].view(np.uint32)), i
        assert nn[i] == r["n_nodes"] and ne[i] == r["n_edges"], i
    # the frames of a select are the Python rule's
    leaf = torch.empty((t.rows, 32), dtype=torch.int32, device="cuda")
    t.select(2.0, leaf_states=leaf)
    fr = t.leaf_frames().cpu().numpy()
    lw = _host(leaf)
    sk = np.repeat(skeys, leaves)
    assert [sy.leaf_frame(lw[r], int(sk[r]), mode) for r in range(t.rows)] == fr.tolist()
    assert len(set(fr.tolist())) > 1


def test_mode_off_after_a_mode_change_is_todays_search(mods, oracle):
    hb, tr, _ = mods
    n, sims = 48, 16
    roots = _roots(hb, n, 3)
    skeys = np.arange(n, dtype=np.uint64) + 11
    fresh = _edges(_framed_search(hb, tr, roots, skeys, sims, 1, None, None, 0.0))
    t = _framed_search(hb, tr, roots, skeys, sims, 1, "full", None, 0.0)
    framed = _edges(t)
    assert not all(np.array_equal(x, y) for x, y in zip(fresh, framed))   # the frame matters to this evaluator
    t.set_symmetry(None)
    t.reset(roots, tr.search_keys_tensor(skeys))
    W = torch.from_numpy(_W).cuda()
    board = torch.zeros((t.rows, 38, 5, 7), device="cuda")
    glob = torch.zeros((t.rows, 42), device="cuda")
    for _ in range(sims):
        t.select(2.0, board, glob)
        p, v = _eval_torch(board, glob, W)
        t.expand_backup(p, v)
    _same_edges(fresh, _edges(t))
    assert (t.leaf_frames() == 0).all()
    # and today's search is the oracle's plain search
    rh = _host(roots)
    for i in range(0, n, 5):
        def eval_fn(w):
            b, gl = oracle.encode(np.array(w, dtype=np.uint32))
            p, v = _eval_np(b, gl)
            return p[0], float(v[0])

        r = oracle.search(rh[i], skeys[i], sims, 2.0, eval_fn=eval_fn, key_mode=1)
        assert np.array_equal(fresh[0][i], r["N"]) and np.array_equal(fresh[1][i], r["W"])


def test_equivariant_evaluator_gives_the_same_search(mods):
    """placement logits per cell, pile logits per pile block, value summed over cells: the same root statistics
    with the mode on or off (the fused softmax runs in the tree's order)"""
    from harmonies_alphazero_b200 import constants as K

    hb, tr, _ = mods
    n, sims = 256, 24
    roots = _roots(hb, n, 77)
    keys = tr.search_keys_tensor(np.arange(n, dtype=np.uint64) * 3 + 1)
    gen = torch.Generator().manual_seed(9)
    wt = torch.randint(-3, 4, (6, 37), generator=gen).to(torch.float64).cuda()      # placement of type t, per plane
    wp = torch.randint(-3, 4, (6,), generator=gen).to(torch.float64).cuda()         # pile: per type count
    wv = torch.randint(-3, 4, (37,), generator=gen).to(torch.float64).cuda()
    hex_cell = torch.tensor([y * 7 + x for (y, x) in K.HEX_CELL], device="cuda")

    def evaluate(board, glob):
        m = board.shape[0]
        cells = board.reshape(m, 38, 35)[:, :37, :].to(torch.float64)[:, :, hex_cell]   # [m, 37, 23]
        place = torch.einsum("tc,mch->mth", wt, cells).reshape(m, 138)
        piles = torch.round(glob[:, :30].to(torch.float64) * 3).reshape(m, 5, 6) @ wp
        logits = (torch.cat([piles, place], dim=1) * 0.125).to(torch.float32).contiguous()
        value = ((torch.einsum("c,mch->m", wv, cells) % 64) / 64).to(torch.float32).contiguous()
        return logits, value

    def run(mode):
        t = tr.BatchedMCTS(n, sims, leaves=2)
        t.set_symmetry(mode)
        t.reset(roots, keys)
        board = torch.zeros((t.rows, 38, 5, 7), device="cuda")
        glob = torch.zeros((t.rows, 42), device="cuda")
        for _ in range(sims // 2):
            t.select(2.0, board, glob)
            lg, v = evaluate(board, glob)
            t.expand_backup(lg, v, is_logits=True)
        return _edges(t)

    off = run(None)
    for mode in ("board", "full"):
        _same_edges(off, run(mode))


def test_select_writes_the_framed_leaf_in_every_fast_layout(mods):
    hb, tr, _ = mods
    from harmonies_alphazero_b200 import _lib

    lib = _lib.load()
    n, K = 93, 2
    t = tr.BatchedMCTS(n, 16, leaves=K)
    t.set_symmetry("full")
    t.reset(_roots(hb, n, 5))
    t.run_synthetic(8, 2.0)
    rows = n * K
    leaf = torch.empty((rows, 32), dtype=torch.int32, device="cuda")
    b40 = torch.zeros((rows, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    g40 = torch.zeros((rows, 42), dtype=torch.bfloat16, device="cuda")
    # a second tree in the same state takes the tile layout (a select leaves in-flight visits behind)
    t2 = tr.BatchedMCTS(n, 16, leaves=K)
    t2.set_symmetry("full")
    t2.reset(_roots(hb, n, 5))
    t2.run_synthetic(8, 2.0)
    t.select(2.0, b40, g40, leaf_states=leaf, dtype=torch.bfloat16, pad40=True)
    nbytes = (rows + 15) // 16 * 71680
    tiles = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    gt = torch.zeros((rows, 42), dtype=torch.bfloat16, device="cuda")
    leaf2 = torch.empty_like(leaf)
    t2.select(2.0, tiles, gt, leaf_states=leaf2, dtype=torch.bfloat16, tiles=True)
    assert torch.equal(leaf, leaf2)
    fr = t.leaf_frames()
    assert torch.equal(fr, t2.leaf_frames())
    ts = sy.transform_states(leaf, fr)
    rb, rg = hb.encode(ts, dtype=torch.bfloat16, channels_last=True)
    assert torch.equal(b40[:, :38], rb) and not b40[:, 38:].any()
    assert torch.equal(g40, rg) and torch.equal(gt, rg)
    ref40 = torch.zeros((rows, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    ref40[:, :38] = rb
    nhwc = ref40.permute(0, 2, 3, 1).contiguous()
    want = torch.zeros(lib.hz_tower_tile_bytes(rows, 1), dtype=torch.uint8, device="cuda")
    assert lib.hz_tower_to_tiles(nhwc.data_ptr(), want.data_ptr(), rows, 40, 1, torch.cuda.current_stream().cuda_stream) == 0
    assert torch.equal(tiles[: want.numel()], want)
    # the leaf states stay in the tree's frame
    assert not torch.equal(leaf, ts)


# ---- self-play, arena, replay ------------------------------------------------------------------
@pytest.mark.parametrize("graph,compact", [(False, False), (True, True), (True, False)])
def test_selfplay_trajectories_do_not_depend_on_the_mode_with_frame_free_evaluators(mods, graph, compact):
    _, _, sp = mods
    out = []
    for mode in (None, "board", "full"):
        cfg = sp.SelfPlayConfig(n_slots=24, num_simulations=12, seed=3, use_cuda_graph=graph, compact_live=compact,
                                eval_symmetry=mode, leaves_per_step=2)
        torch.manual_seed(0)
        out.append(sp.BatchedSelfPlay(sp.SyntheticEvaluator(), cfg).play(30))
    for tr_ in out[1:]:
        assert torch.equal(tr_.states, out[0].states) and torch.equal(tr_.visits, out[0].visits)
        assert torch.equal(tr_.z, out[0].z) and torch.equal(tr_.game_id, out[0].game_id)


def test_selfplay_and_arena_with_the_default_net_on_the_tower(mods):
    hb, _, sp = mods
    from harmonies_alphazero_b200 import arena
    from harmonies_alphazero_b200 import net as hnet

    torch.manual_seed(4)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    inf = hnet.InferenceNet(model, device="cuda", tower="hand")
    assert inf.wants_tiles
    cfg = sp.SelfPlayConfig(n_slots=32, num_simulations=8, seed=6, eval_symmetry="full")
    traj = sp.BatchedSelfPlay(inf, cfg).play(32)
    assert traj.stats["games"] == 32 and len(traj) > 32 * 20
    assert (traj.visits.sum(dim=1) == cfg.num_simulations - 1).all()
    legal = _mask_bits(hb.legal_mask(traj.states.contiguous()))
    assert not ((traj.visits > 0) & (legal == 0)).any()
    r = arena.play_match(inf, arena.GREEDY, 4, {"num_simulations": 8, "cpuct": 2.0}, seed=2, symmetry="full")
    assert r["games"] == 4 and r["candidate_wins"] + r["best_wins"] + r["draws"] == 4
    # Trajectories.transform
    g = torch.randint(0, 480, (len(traj),), device="cuda")
    tt = traj.transform(g)
    assert torch.equal(tt.states, sy.transform_states(traj.states.contiguous(), g))
    assert torch.equal(tt.visits, sy.transform_actions(traj.visits.contiguous(), g, traj.states.contiguous()))
    assert torch.equal(tt.z, traj.z)


def test_replay_ring_augmented_batches(mods):
    hb, _, sp = mods
    from harmonies_alphazero_b200.replay import ReplayRing

    cfg = sp.SelfPlayConfig(n_slots=16, num_simulations=8, seed=8)
    traj = sp.BatchedSelfPlay(sp.SyntheticEvaluator(), cfg).play(16)
    ring = ReplayRing(4096)
    ring.extend(traj)
    n = len(ring)
    # augment=None: exactly today's batch, and the generator advances as today
    g1, g2 = torch.Generator("cuda").manual_seed(5), torch.Generator("cuda").manual_seed(5)
    a = ring.sample(300, generator=g1)
    b = ring.sample(300, generator=g2, augment=None)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert torch.equal(torch.randint(0, 9, (20,), device="cuda", generator=g1), torch.randint(0, 9, (20,), device="cuda", generator=g2))
    # every augmented row is (encode(T_g s), T_g(visits) normalised, z) for some g of the group
    for mode, G in (("board", 4), ("full", 480)):
        gen = torch.Generator("cuda").manual_seed(11)
        board, glob, pi, z = ring.sample(20000, generator=gen, augment=mode)
        gen = torch.Generator("cuda").manual_seed(11)
        idx = torch.randint(0, ring.size, (20000,), device="cuda", generator=gen)
        g = torch.randint(0, G, (20000,), device="cuda", generator=gen)
        s = ring.states[idx].contiguous()
        eb, eg = hb.encode(sy.transform_states(s, g))
        v = sy.transform_actions(ring.visits[idx].contiguous(), g, s).to(torch.float64)
        assert torch.equal(board, eb) and torch.equal(glob, eg)
        assert torch.equal(pi, (v / v.sum(dim=1, keepdim=True).clamp_min(1)).to(torch.float32))
        assert torch.equal(z, ring.z[idx].view(-1, 1))
        assert torch.unique(g).numel() == G
        # consistency that needs no knowledge of g: visits sit on legal moves of the transformed state, and the
        # state's pile features are a reordering of the original's
        if mode == "board":
            lm = _mask_bits(hb.legal_mask(sy.transform_states(s, g)))
            assert not ((pi > 0) & (lm == 0)).any()
    parts = list(ring.epoch(1000, generator=torch.Generator("cuda").manual_seed(1), augment="full"))
    assert sum(p[0].shape[0] for p in parts) == n
