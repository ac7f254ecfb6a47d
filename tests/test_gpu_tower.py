"""GPU tests of the hand-written sm_100a residual tower (csrc/hz_tower.cu, SURVEY.md §8 row f4)
through the C ABI.

* exact: with small-integer activations / weights every fp32 partial sum is an integer below
  2^24, so tcgen05 accumulation order cannot matter and the bf16 outputs must equal
  RNE(conv2d) BIT FOR BIT — for the stem shape (one 64-channel half, K-major input image), the
  residual shape (two halves, MN-major image), with and without residual / ReLU, and with many
  tiles pushed through few CTAs (ring, tile-buffer and TMEM-unit phase wrap-around).
* model: the whole tower against the cuDNN path of InferenceNet (same folded bf16 weights) and the
  fp32 reference architecture (model.py:325-357), at bf16 tolerance (stated in the test).
"""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tw():
    from harmonies_alphazero_b200 import _lib, tower

    _lib.load()
    return tower


class _Raw:
    """HandTower plumbing without a model: buffers + ctypes calls."""

    def __init__(self, tower):
        self.t = tower.HandTower.__new__(tower.HandTower)
        self.t.device = torch.device("cuda")
        from harmonies_alphazero_b200 import _lib

        self.t.lib = _lib.load()
        self.t._bufs = {}
        self.t.fault = None
        self.tower = tower

    def tiles(self, x_nchw):
        """bf16 [B,C,5,7] -> tiles: C <= 64: T16K (one half, the stem's input), C == 128: T16"""
        B, C = x_nchw.shape[:2]
        halves = 1 if C <= 64 else 2
        n_pad = (B + 15) // 16 * 16
        nhwc = x_nchw.permute(0, 2, 3, 1).contiguous()
        dst = torch.zeros(n_pad // 16 * halves * self.tower.KH_BYTES, dtype=torch.uint8, device="cuda")
        self.t.to_tiles(nhwc, C, halves == 1, dst)
        return dst, halves, n_pad

    def conv(self, x_nchw, w, bias, res_nchw=None, relu=True):
        B = x_nchw.shape[0]
        xt, halves, n_pad = self.tiles(x_nchw)
        img, nkh = self.tower.pack_conv_weight(w)
        assert nkh == halves
        rt = None if res_nchw is None else self.tiles(res_nchw)[0]
        y = torch.zeros(n_pad // 16 * 2 * self.tower.KH_BYTES, dtype=torch.uint8, device="cuda")
        self.t.conv(xt, halves, (img.cuda(), bias.float().cuda(), nkh), rt, y, n_pad, relu=relu, kmajor=halves == 1)
        torch.cuda.synchronize()
        return self.t.from_tiles(y, n_pad)[:B].view(B, 5, 7, 128).permute(0, 3, 1, 2)


def _ref(x, w, bias, res, relu):
    y = F.conv2d(x.double().cpu(), w.double().cpu(), bias.double().cpu(), padding=1)
    if res is not None:
        y = y + res.double().cpu()
    if relu:
        y = torch.relu(y)
    return y.float().to(torch.bfloat16)


def _ints(shape, lo, hi, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(lo, hi + 1, shape, generator=g).float()


def test_tile_layout_roundtrip(tw):
    raw = _Raw(tw)
    x = _ints((37, 128, 5, 7), -3, 3, 1).to(torch.bfloat16).cuda()
    xt, halves, n_pad = raw.tiles(x)
    back = raw.t.from_tiles(xt, 37).view(37, 5, 7, 128).permute(0, 3, 1, 2)
    assert torch.equal(back, x)
    # the documented address of an element (include/harmonies_b200.h): p = cell*16 + board
    img = xt.cpu().numpy()
    xs = x.cpu()
    for (b, c, y, xx) in [(0, 0, 0, 0), (5, 77, 3, 4), (36, 127, 4, 6), (17, 64, 2, 1)]:
        tile, p = b // 16, (y * 7 + xx) * 16 + b % 16
        off = tile * 2 * tw.KH_BYTES + (c // 8) * 8960 + (p // 8) * 128 + (c % 8) * 16 + (p % 8) * 2
        got = torch.from_numpy(img[off:off + 2].copy()).view(torch.bfloat16)[0]
        assert got == xs[b, c, y, xx]
    # T16K, the stem's input image
    x40 = _ints((19, 40, 5, 7), -3, 3, 2).to(torch.bfloat16).cuda()
    kt = raw.tiles(x40)[0].cpu().numpy()
    for (b, c, y, xx) in [(0, 0, 0, 0), (5, 37, 3, 4), (18, 39, 4, 6), (17, 8, 2, 1)]:
        tile, p = b // 16, (y * 7 + xx) * 16 + b % 16
        off = tile * tw.KH_BYTES + p * 128 + (((c // 8) ^ (p & 7)) << 4) + (c % 8) * 2
        got = torch.from_numpy(kt[off:off + 2].copy()).view(torch.bfloat16)[0]
        assert got == x40.cpu()[b, c, y, xx]


@pytest.mark.parametrize("cin,boards,res,relu", [
    (128, 16, False, True),
    (128, 16, True, True),
    (128, 48, True, False),
    (40, 16, False, True),
    (40, 33, False, False),
    (128, 16 * 9 + 5, True, True),
])
def test_conv_bit_exact_on_integers(tw, cin, boards, res, relu):
    raw = _Raw(tw)
    x = _ints((boards, cin, 5, 7), -2, 2, 10 + boards).to(torch.bfloat16).cuda()
    w = _ints((128, cin, 3, 3), -1, 1, 20 + cin)
    bias = _ints((128,), -4, 4, 30)
    r = _ints((boards, 128, 5, 7), -8, 8, 40).to(torch.bfloat16).cuda() if res else None
    got = raw.conv(x, w, bias, r, relu=relu)
    want = _ref(x, w, bias, r, relu)
    assert torch.equal(got.cpu(), want), f"max abs diff {(got.cpu().float() - want.float()).abs().max()}"


def test_conv_many_tiles_through_few_ctas(tw):
    """23 tiles through 3 CTAs: every ring / buffer / TMEM-unit barrier wraps its phase several times."""
    raw = _Raw(tw)
    raw.t.lib.hz_tower_set_max_ctas(3)
    try:
        boards = 16 * 23
        x = _ints((boards, 128, 5, 7), -2, 2, 5).to(torch.bfloat16).cuda()
        w = _ints((128, 128, 3, 3), -1, 1, 6)
        bias = _ints((128,), -4, 4, 7)
        r = _ints((boards, 128, 5, 7), -8, 8, 8).to(torch.bfloat16).cuda()
        got = raw.conv(x, w, bias, r)
        assert torch.equal(got.cpu(), _ref(x, w, bias, r, True))
    finally:
        raw.t.lib.hz_tower_set_max_ctas(0)


def test_conv_random_values_bf16_tolerance(tw):
    """Real-valued data: fp32 accumulation order differs from the reference's, so the bound is one
    bf16 rounding of the output (2^-8 relative) plus fp32 accumulation noise."""
    raw = _Raw(tw)
    g = torch.Generator().manual_seed(3)
    x = torch.randn((64, 128, 5, 7), generator=g).to(torch.bfloat16).cuda()
    w = (torch.randn((128, 128, 3, 3), generator=g) * 0.03).to(torch.bfloat16).float()
    bias = torch.randn((128,), generator=g)
    r = torch.randn((64, 128, 5, 7), generator=g).to(torch.bfloat16).cuda()
    got = raw.conv(x, w, bias, r).float().cpu()
    y = F.conv2d(x.double().cpu(), w.double(), bias.double(), padding=1) + r.double().cpu()
    want = torch.relu(y).float()
    err = (got - want).abs()
    assert float((err - want.abs() * 2.0 ** -8).max()) <= 1e-3


def test_fused_launch_equals_layer_by_layer(tw):
    """The persistent all-layers launch (each CTA carries its tiles through the 17 layers) must
    reproduce the one-launch-per-layer result (hz_tower_conv3x3 chained here) bit for bit — with one tile
    per CTA, several tiles per CTA, and all ten tiles through a single CTA (the ready queue hands it every
    item of every layer)."""
    from harmonies_alphazero_b200 import net as hnet
    from harmonies_alphazero_b200 import tower as htower

    torch.manual_seed(2)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    hand = hnet.InferenceNet(model, device="cuda", tower="hand")
    ht = hand.hand
    B = 16 * 9 + 3
    g = torch.Generator().manual_seed(4)
    b40 = torch.zeros((B, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    b40[:, :38] = (torch.rand((B, 38, 5, 7), generator=g) < 0.2).to(torch.bfloat16).cuda()
    n_pad = (B + 15) // 16 * 16
    x0 = ht.x0_buffer(B)
    ht.to_tiles(b40, 40, True, x0)
    x, y, z = (torch.zeros(n_pad // 16 * 2 * htower.KH_BYTES, dtype=torch.uint8, device="cuda") for _ in range(3))
    ht.conv(x0, 1, ht.stem, None, x, n_pad, kmajor=True)
    for c1, c2 in ht.blocks:
        ht.conv(x, 2, c1, None, y, n_pad)
        ht.conv(y, 2, c2, x, z, n_pad)
        x, z = z, x
    want = ht.from_tiles(x, n_pad)[:B].view(B, 5, 7, 128).permute(0, 3, 1, 2)
    try:
        for ctas in (0, 4, 1):       # 10 tiles: one per CTA / up to 3 per CTA / all 10 in one CTA
            ht.lib.hz_tower_set_max_ctas(ctas)
            got = ht.forward(b40).clone()
            torch.cuda.synchronize()
            assert torch.equal(got, want), ctas
    finally:
        ht.lib.hz_tower_set_max_ctas(0)


def test_whole_tower_against_cudnn_and_fp32(tw):
    from harmonies_alphazero_b200 import net as hnet

    torch.manual_seed(0)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    # non-trivial BatchNorm statistics so that folding is exercised
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0, 0.1)
            m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.normal_(0, 0.1)
    B = 100
    g = torch.Generator().manual_seed(1)
    board = (torch.rand((B, 38, 5, 7), generator=g) < 0.15).float()
    glob = torch.rand((B, 42), generator=g)
    with torch.no_grad():
        ref_logits, ref_value = model(board, glob)
    hand = hnet.InferenceNet(model, device="cuda", tower="hand")
    lib = hnet.InferenceNet(model, device="cuda", tower="cudnn")
    b40 = torch.zeros((B, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    b40[:, :38] = board.cuda().to(torch.bfloat16)
    gl = glob.cuda().to(torch.bfloat16)
    lh, vh = hand(b40, gl)
    ll, vl = lib(b40, gl)
    torch.cuda.synchronize()
    # both bf16 paths differ from the fp32 reference by bf16 rounding of 17 layers of activations;
    # they must agree with each other at least as well as cuDNN agrees with fp32
    e_lib = float((ll.cpu() - ref_logits).abs().max())
    e_hand = float((lh.cpu() - ref_logits).abs().max())
    scale = float(ref_logits.abs().max())
    assert e_hand <= max(2.0 * e_lib, 0.02 * scale), (e_hand, e_lib, scale)
    assert float((vh.cpu() - ref_value.view(-1)).abs().max()) <= max(2.0 * float((vl.cpu() - ref_value.view(-1)).abs().max()), 0.02)
    # tower outputs themselves
    xh = hand.tower_out(b40).float().cpu()
    xl = lib.tower_out(b40).float().cpu()
    with torch.no_grad():
        x = F.relu(model.bn(model.conv(board)))
        for blk in model.residual_blocks:
            x = blk(x)
    tol = 0.03 * float(x.abs().max())
    assert float((xh - x).abs().max()) <= tol and float((xl - x).abs().max()) <= tol


def test_leaf_encoder_writes_the_stem_image(tw):
    """hz_tree_select with HZ_LAYOUT_T16K must produce byte for byte what hz_tower_to_tiles makes of
    the NHWC40 encoding of the same leaves (no layout-conversion kernel on the self-play path)."""
    from harmonies_alphazero_b200 import batched as hb
    from harmonies_alphazero_b200 import tree as tr

    n, K = 37, 2
    st = hb.init_states(n, seed=5)
    hb.playout(st, max_steps=11)
    raw = _Raw(tw)
    outs = []
    for tiles in (False, True):
        t = tr.BatchedMCTS(n, 8, leaves=K)
        t.reset(st, tr.search_keys_tensor(np.arange(n, dtype=np.uint64)))
        t.run_synthetic(4, 2.0)              # a few simulations so that the leaves are not all the root
        rows = n * K
        glob = torch.zeros((rows, 42), dtype=torch.bfloat16, device="cuda")
        if tiles:
            board = torch.zeros((rows + 15) // 16 * tw.KH_BYTES, dtype=torch.uint8, device="cuda")
        else:
            board = torch.zeros((rows, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
        t.select(2.0, board, glob, dtype=torch.bfloat16, channels_last=True, pad40=not tiles, tiles=tiles)
        torch.cuda.synchronize()
        outs.append((board, glob))
    want = torch.zeros_like(outs[1][0])
    raw.t.to_tiles(outs[0][0], 40, True, want)
    torch.cuda.synchronize()
    assert torch.equal(outs[1][0], want)
    assert torch.equal(outs[1][1], outs[0][1])


def test_tile_path_equals_tensor_path(tw):
    """InferenceNet.forward_tiles (encoder image -> tower -> head convs from T16 -> FC heads) against
    the tensor path of the same network (to_tiles / from_tiles / hz_net_heads).  The towers are the
    same kernel (identical bits); the 1x1 head convolutions differ in arithmetic only (fp32 FMA vs
    bf16 hi+lo tensor-core split, both fp32-weight accurate): tolerance 1e-4 absolute on O(1) logits."""
    from harmonies_alphazero_b200 import net as hnet

    torch.manual_seed(3)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    hand = hnet.InferenceNet(model, device="cuda", tower="hand")
    assert hand.wants_tiles
    B = 50
    g = torch.Generator().manual_seed(9)
    b40 = torch.zeros((B, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    b40[:, :38] = (torch.rand((B, 38, 5, 7), generator=g) < 0.2).to(torch.bfloat16).cuda()
    glob = torch.rand((B, 42), generator=g).to(torch.bfloat16).cuda()
    l1, v1 = hand(b40, glob)
    x0 = hand.hand.x0_buffer(B)
    hand.hand.to_tiles(b40, 40, True, x0)
    l2, v2 = hand.forward_tiles(x0, glob, B)
    torch.cuda.synchronize()
    assert float((l1 - l2).abs().max()) <= 1e-4 and float((v1 - v2).abs().max()) <= 1e-4


def test_self_play_runs_on_the_hand_written_tower(tw):
    from harmonies_alphazero_b200 import net as hnet
    from harmonies_alphazero_b200 import selfplay as sp

    torch.manual_seed(0)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    hand = hnet.InferenceNet(model, device="cuda", tower="hand")
    cfg = sp.SelfPlayConfig(n_slots=48, num_simulations=12, seed=3)
    drv = sp.BatchedSelfPlay(hand, cfg)
    assert drv.groups[0].tiles
    traj = drv.play(60)
    assert traj.stats["games"] == 60 and len(traj) > 60 * 40
    v = traj.visits.to(torch.int64).sum(dim=1)
    assert int(v.max()) == 11 and int(v.min()) >= 0          # sum N = sims - 1 (MCTS.py:355-381)
    assert set(traj.z.unique().tolist()) <= {-1.0, 0.0, 1.0}


def test_active_prefix_of_the_tile_path(tw):
    """hz_tower_forward_heads / hz_net_heads_fc_active: with a device-side row count the evaluated prefix is
    bit-identical to the full evaluation and the rows beyond the last active tile are left untouched."""
    from harmonies_alphazero_b200 import net as hnet

    torch.manual_seed(4)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    hand = hnet.InferenceNet(model, device="cuda", tower="hand")
    B = 200
    g = torch.Generator().manual_seed(11)
    b40 = torch.zeros((B, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    b40[:, :38] = (torch.rand((B, 38, 5, 7), generator=g) < 0.2).to(torch.bfloat16).cuda()
    glob = torch.rand((B, 42), generator=g).to(torch.bfloat16).cuda()
    x0 = hand.hand.x0_buffer(B)
    hand.hand.to_tiles(b40, 40, True, x0)
    l_full, v_full = hand.forward_tiles(x0, glob, B)
    l_full, v_full = l_full.clone(), v_full.clone()
    na = torch.zeros(1, dtype=torch.int32, device="cuda")
    for k in (200, 131, 16, 1, 0):
        na.fill_(k)
        out = (torch.full((B, 143), -7.0, device="cuda"), torch.full((B,), -7.0, device="cuda"))
        hand.forward_tiles(x0, glob, B, out=out, n_active=na)
        torch.cuda.synchronize()
        assert torch.equal(out[0][:k], l_full[:k]) and torch.equal(out[1][:k], v_full[:k])
        assert bool((out[0][k:] == -7.0).all()) and bool((out[1][k:] == -7.0).all())


def test_self_play_with_live_prefix_compaction_equals_plain(tw):
    """SelfPlayConfig.compact_live: whole games on the hand-written tower with the live games kept in a
    dense prefix (device-side active counts under the captured graph) give exactly the trajectories of
    the plain loop — every row's evaluation is independent of where it sits in the batch."""
    from harmonies_alphazero_b200 import net as hnet
    from harmonies_alphazero_b200 import selfplay as sp

    torch.manual_seed(0)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    hand = hnet.InferenceNet(model, device="cuda", tower="hand")
    out = []
    for compact in (False, True):
        cfg = sp.SelfPlayConfig(n_slots=40, num_simulations=8, seed=5, testing=True, compact_live=compact)
        t = sp.BatchedSelfPlay(hand, cfg).play(56)
        assert t.stats["games"] == 56
        order = torch.argsort(t.game_id * 1000 + t.move_no.to(torch.int64))
        out.append((t.states[order].cpu(), t.visits[order].cpu(), t.z[order].cpu(), t.stats["searched_slots"], t.stats["move_steps"]))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]) and torch.equal(out[0][2], out[1][2])
    assert out[1][3] < out[0][3] and out[1][3] == len(out[1][0])      # compacted: exactly one searched slot per example


def test_search_is_a_function_of_the_priors_whichever_tower_produced_them(tw):
    """VERDICT r1 item 1 (i): the priors and values the hand-written path produced during a search are captured
    per simulation and fed to a second set of trees that encodes its leaves for the cuDNN path: visit counts, W
    and P of the roots are bit-identical (the tree kernels see the evaluator only through (policy, value)), and
    a cuDNN-evaluated search from the same roots agrees with the hand-evaluated one on the bf16-level."""
    from harmonies_alphazero_b200 import batched as hb
    from harmonies_alphazero_b200 import net as hnet
    from harmonies_alphazero_b200 import tree as htree

    torch.manual_seed(1)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    hand = hnet.InferenceNet(model, device="cuda", tower="hand")
    lib = hnet.InferenceNet(model, device="cuda", tower="cudnn")
    n, sims = 96, 24
    st = hb.init_states(n, seed=31)
    hb.playout(st, max_steps=11)
    t1 = htree.BatchedMCTS(n, sims)
    t1.reset(st)
    board, glob, logits, value = hand.leaf_buffers(n)
    captured = []
    for _ in range(sims):
        t1.select(2.0, board, glob, dtype=torch.bfloat16, tiles=True)
        hand.forward_tiles(board, glob, n, out=(logits, value))
        captured.append((logits.clone(), value.clone()))
        t1.expand_backup(logits, value, is_logits=True)
    t2 = htree.BatchedMCTS(n, sims)
    t2.reset(st)
    b2, g2, l2, v2 = lib.leaf_buffers(n)
    worst = 0.0
    for lg, vl in captured:
        t2.select(2.0, b2, g2, dtype=torch.bfloat16, channels_last=True, pad40=b2.shape[1] == 40)
        lib(b2, g2, out=(l2, v2))                      # the cuDNN path on the same leaves
        worst = max(worst, float((torch.softmax(l2, 1) - torch.softmax(lg, 1)).abs().max()), float((v2 - vl).abs().max()))
        t2.expand_backup(lg, vl, is_logits=True)       # ... but the tree is fed the captured values
    t1.check_status(); t2.check_status()
    N1, W1, P1, _ = t1.root_edges(); N2, W2, P2, _ = t2.root_edges()
    assert torch.equal(N1, N2) and torch.equal(W1, W2) and torch.equal(P1, P2)
    assert worst < 0.03          # same leaves, two towers: bf16-level agreement of priors and values


def test_reloaded_weights_take_effect_under_the_captured_graph(tw):
    """InferenceNet.load() after a weight broadcast: a driver that already captured its simulation step as a CUDA graph
    must search with the NEW weights (it re-captures on the network's version), exactly like a fresh driver."""
    from harmonies_alphazero_b200 import batched as hb
    from harmonies_alphazero_b200 import net as hnet
    from harmonies_alphazero_b200 import selfplay as sp

    def model(seed):
        torch.manual_seed(seed)
        return hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()

    cfg = sp.SelfPlayConfig(n_slots=32, num_simulations=16, seed=9, testing=True)
    states = hb.init_states(32, seed=17)
    hb.playout(states, max_steps=13)
    inf = hnet.InferenceNet(model(1), device="cuda", tower="hand")
    drv = sp.BatchedSelfPlay(inf, cfg)
    drv.search(states)
    v_old = drv.root_policy()[0].clone()
    assert drv.graph is not None
    inf.load(model(2))
    drv.search(states)
    v_new = drv.root_policy()[0].clone()
    fresh = sp.BatchedSelfPlay(hnet.InferenceNet(model(2), device="cuda", tower="hand"), cfg)
    fresh.search(states)
    v_ref = fresh.root_policy()[0]
    assert torch.equal(v_new, v_ref)
    assert not torch.equal(v_old, v_new)
