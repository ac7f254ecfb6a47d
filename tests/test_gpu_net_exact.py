"""The network inference paths (hand-written tower + head kernels) against an exact fp64 reference, bit for bit.

An exactly computable network: sparse +-1 integer conv and FC weights, integer biases, identity BatchNorm (eps = 0,
mean 0, var 1 or 4 with weight 1 or 2), 0/1 boards and integer global features.  Every tower sum is then an integer
far below 2^24, so the accumulation order of the tensor cores cannot matter, and the only rounding is the epilogue's
fp32 -> bf16 conversion after every layer.  The recipe makes that rounding matter: about half of the final activations
are above 256, where bf16 keeps fewer bits than the integer has, and thousands of outputs are exact ties.  A kernel that
truncates, or rounds ties away from zero, gives different logits.  The heads stay exact too: the 1x1 convolutions and FC
layers see integers below 2^16 (so every bf16 hi + lo split is exact), value_fc2 has dyadic weights, and only tanh
rounds.  So the logits must equal the reference bit for bit, and the value must be within the 2 ulp of ``tanhf``.

The reference is the module's own layers in float64, with bf16 round-to-nearest-even after every tower layer, as the
kernel does.  It asserts its own preconditions (``reference``), so a change of recipe that stops exercising the rounding
or leaves the exact range fails loudly instead of passing quietly.

The same exact network runs through every inference path, batch size, active prefix, grid size and tower depth.
Exact data cannot see a kernel that drops the low part of a bf16 hi + lo split: with integer weights
every low part is zero.  The split-precision tests use real-valued weights with large low parts, and a scale-free bound
derived in ``split_bound``.  Host-side negative controls show that the bound catches one dropped low product.  The last
test bounds the fused softmax of ``hz_tree_expand_backup`` per edge against fp64.
"""

import ctypes as ct

import numpy as np
import pytest
import torch
import torch.nn.functional as F

SIZES = (1, 15, 16, 17, 33, 203, 4096, 4103, 16384)
N_MAX = max(SIZES)
HZ_ERR_ARG = -1
SENTINEL = -7.0
V2_EXP = 16                  # value_fc2 weights are k * 2^-V2_EXP


# ---- the exact network ------------------------------------------------------------------------------------------------
def _sparse_pm1(n_out, fan_in, nnz, g):
    """[n_out, fan_in] fp32 with exactly ``nnz`` entries of +-1 per row"""
    idx = torch.rand((n_out, fan_in), generator=g).argsort(dim=1)[:, :nnz]
    sign = torch.randint(0, 2, (n_out, nnz), generator=g).float() * 2 - 1
    return torch.zeros((n_out, fan_in)).scatter_(1, idx, sign)


def exact_model(cfg=None, blocks=8, seed=0):
    """AlphaZeroNet whose bf16 inference is exact in every kernel (module docstring).  Deterministic in (cfg, blocks, seed)."""
    from harmonies_alphazero_b200 import net as hnet

    cfg = dict(cfg or hnet.DEFAULT_MODEL_CONFIG, num_res_blocks=blocks)
    m = hnet.AlphaZeroNet.from_config(cfg).eval()
    g = torch.Generator().manual_seed(7000 + seed)

    def layer(mod, nnz, lo, hi):
        w = mod.weight
        w.data.copy_(_sparse_pm1(w.shape[0], w[0].numel(), nnz, g).view_as(w))
        mod.bias.data.copy_(torch.randint(lo, hi + 1, (w.shape[0],), generator=g).float())

    with torch.no_grad():
        layer(m.conv, 16, -1, 2)
        for b in m.residual_blocks:
            layer(b.conv1, 5, -3, 1)
            layer(b.conv2, 5, -3, 1)
        layer(m.policy_conv, 2, -2, 2)
        layer(m.value_conv, 2, -2, 2)
        layer(m.policy_fc, 6, -4, 4)
        layer(m.value_fc1, 4, -4, 4)
        k = torch.randint(-3, 4, (1, m.value_fc2.in_features), generator=g).float()
        m.value_fc2.weight.copy_(k * 2.0 ** -V2_EXP)
        m.value_fc2.bias.fill_(0.25)
        for i, bn in enumerate(mod for mod in m.modules() if isinstance(mod, torch.nn.BatchNorm2d)):
            bn.eps = 0.0
            bn.running_mean.zero_()
            bn.bias.data.zero_()
            # scale = weight / sqrt(var): 1 either way, but the odd layers fold a non-trivial pair
            bn.running_var.fill_(4.0 if i % 2 else 1.0)
            bn.weight.data.fill_(2.0 if i % 2 else 1.0)
    return m


def exact_inputs(n, seed=0):
    """0/1 boards [n, 38, 5, 7] at density 0.2 (like the encoder's planes) and integer global features 0..3 [n, 42];
    the first rows of a larger call are the rows of a smaller one."""
    g = torch.Generator().manual_seed(9100 + seed)
    board = (torch.rand((n, 38, 5, 7), generator=g) < 0.2).float()
    glob = torch.randint(0, 4, (n, 42), generator=g).float()
    return board, glob


def _round_bf16(y, mode):
    """fp64 -> fp32 (exact below 2^24) -> bf16 with round-to-nearest-even, toward zero, or ties away from zero"""
    f = y.float()
    if mode == "rne":
        return f.to(torch.bfloat16).double()
    bits = f.view(torch.int32)
    if mode == "rha":
        assert bool((bits >= 0).all())                       # ReLU outputs: ties away from zero = ties up
        bits = bits + 0x8000
    return (bits & ~0xFFFF).view(torch.float32).double()


def _bf16_split_exact(v):
    hi = v.float().to(torch.bfloat16).float()
    lo = (v.float() - hi).to(torch.bfloat16).float()
    return bool((hi.double() + lo.double() == v).all())


@torch.no_grad()
def reference(model, board, glob, mode="rne", device="cpu", stats=True):
    """fp64 forward of ``model`` with bf16 rounding (``mode``) after every tower layer, and the recipe's preconditions.

    Returns dict(tower [B,128,5,7] fp64 (bf16 values), logits fp64, pre_tanh fp64, value fp64, stats)."""
    m = {k: v.double().to(device) for k, v in model.state_dict().items()}
    bns = {name: mod for name, mod in model.named_modules() if isinstance(mod, torch.nn.BatchNorm2d)}
    x = board.double().to(device)
    glob = glob.double().to(device)
    lim = 2.0 ** 22
    st = dict(worst_sum=0.0, ties=0, outputs=0)

    def bn(y, name):
        b = bns[name]
        return (y - m[name + ".running_mean"].view(1, -1, 1, 1)) / torch.sqrt(m[name + ".running_var"].view(1, -1, 1, 1) + b.eps) \
            * m[name + ".weight"].view(1, -1, 1, 1) + m[name + ".bias"].view(1, -1, 1, 1)

    def conv_layer(x, conv, bnn, res=None):
        w, b = m[conv + ".weight"], m[conv + ".bias"]
        pad = w.shape[-1] // 2
        y = bn(F.conv2d(x, w, b, padding=pad), bnn)
        # every partial sum of the kernel's fp32 accumulation is bounded by sum |w||x| + |b| (+ |residual|)
        s = F.conv2d(x.abs(), w.abs(), b.abs(), padding=pad)
        if res is not None:
            y = y + res
            s = s + res.abs()
        st["worst_sum"] = max(st["worst_sum"], float(s.max()))
        return torch.relu(y)

    def tower_layer(*args):
        y = conv_layer(*args)
        assert bool((y == torch.round(y)).all()), "tower sums must be integers"
        f = y.float().view(torch.int32)
        st["ties"] += int(((f & 0xFFFF) == 0x8000).sum())
        st["outputs"] += y.numel()
        return _round_bf16(y, mode)

    x = tower_layer(x, "conv", "bn")
    for i in range(len(model.residual_blocks)):
        p = f"residual_blocks.{i}."
        y = tower_layer(x, p + "conv1", p + "bn1")
        x = tower_layer(y, p + "conv2", p + "bn2", x)
    tower = x
    B = x.shape[0]
    pin = torch.cat((conv_layer(x, "policy_conv", "policy_bn").flatten(1), glob), 1)
    vin = torch.cat((conv_layer(x, "value_conv", "value_bn").flatten(1), glob), 1)

    def fc(v, name):
        w, b = m[name + ".weight"], m[name + ".bias"]
        assert _bf16_split_exact(v), f"{name}: an input is not bf16 hi + lo exact"
        st["worst_sum"] = max(st["worst_sum"], float((v.abs() @ w.abs().t() + b.abs()).max()))
        return v @ w.t() + b

    logits = fc(pin, "policy_fc")
    hidden = torch.relu(fc(vin, "value_fc1"))
    w2, b2 = m["value_fc2.weight"], m["value_fc2.bias"]
    s = (hidden @ w2.t() + b2).view(B)
    # value_fc2: every partial sum is a multiple of 2^-V2_EXP below 2^(24 - V2_EXP), hence exact in fp32
    s_abs = (hidden @ w2.abs().t() + b2.abs()).view(B)
    assert float(s_abs.max()) < 2.0 ** (24 - V2_EXP)
    assert bool((s * 2.0 ** V2_EXP == torch.round(s * 2.0 ** V2_EXP)).all())
    assert st["worst_sum"] < lim, f"a partial sum reaches {st['worst_sum']} (limit 2^22)"
    assert bool((logits.float().double() == logits).all())
    st["nonzero"] = float((tower > 0).double().mean())
    st["above_256"] = float((tower > 256).double().mean())
    if stats:
        # the recipe must exercise the bf16 rounding of the epilogue (measured on 64 boards: 0.51 above 256)
        assert st["above_256"] >= 0.3 and st["nonzero"] >= 0.5, st
        assert st["ties"] >= 3000 * max(1, B // 64), st
    return dict(tower=tower, logits=logits, pre_tanh=s, value=torch.tanh(s), stats=st)


def _ulp32(r):
    """fp32 ulp at the exact value r (fp64 tensor): 2^(e - 24) for r = m 2^e, 0.5 <= |m| < 1, floored at the denormals"""
    _, e = torch.frexp(r)
    return torch.pow(2.0, torch.clamp(e.double() - 24, min=-149))


def assert_exact(got, ref, n, what, lo=0):
    """logits bit for bit and the value within the 2 ulp tanhf guarantees, rows lo..n-1"""
    logits, value = got
    want = ref["logits"][lo:n].float()
    bad = (logits[lo:n] != want).any(dim=1)
    if bool(bad.any()):
        r = int(bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {n - lo} logit rows differ, first row {lo + r}: "
                             f"max |diff| {float((logits[lo + r] - want[r]).abs().max())}")
    r = ref["value"][lo:n]
    err = (value[lo:n].double() - r).abs()
    assert bool((err <= 2 * _ulp32(r)).all()), f"{what}: value off by {float((err / _ulp32(r)).max())} ulp"


def assert_bn_folds_exactly(model):
    """net._fold (what InferenceNet and HandTower use) must give the module's integer weights and biases bit for bit"""
    from harmonies_alphazero_b200 import net as hnet

    pairs = [(model.conv, model.bn), (model.policy_conv, model.policy_bn), (model.value_conv, model.value_bn)]
    pairs += [(c, b) for blk in model.residual_blocks for c, b in ((blk.conv1, blk.bn1), (blk.conv2, blk.bn2))]
    for conv, bn in pairs:
        w, b = hnet._fold(conv, bn)
        assert torch.equal(w, conv.weight.detach().float()) and torch.equal(b, conv.bias.detach().float())


# ---- host-side checks of the recipe (no GPU) ---------------------------------------------------------------------------
def test_recipe_folds_exactly_and_meets_its_preconditions():
    from harmonies_alphazero_b200 import net as hnet

    for cfg, blocks in ((None, 8), (None, 0), (None, 9), (hnet.TEST_MODEL_CONFIG, 1)):
        model = exact_model(cfg, blocks)
        assert_bn_folds_exactly(model)
        for t in model.state_dict().values():
            if t.dtype == torch.float32:
                assert torch.equal(t.to(torch.bfloat16).float(), t)      # bf16-exact: every hi + lo split has lo = 0
    board, glob = exact_inputs(64)
    model = exact_model()
    ref = {mode: reference(model, board, glob, mode, stats=mode == "rne") for mode in ("rne", "rz", "rha")}
    # an epilogue that truncates, or rounds ties away from zero, gives other logits on this data
    for mode in ("rz", "rha"):
        assert not torch.equal(ref[mode]["tower"], ref["rne"]["tower"])
        assert not torch.equal(ref[mode]["logits"], ref["rne"]["logits"]), mode
    assert not torch.equal(ref["rz"]["logits"], ref["rha"]["logits"])
    # the value is not saturated: tanh still has bits to get wrong
    assert 0.3 < float(ref["rne"]["pre_tanh"].abs().min()) and float(ref["rne"]["pre_tanh"].abs().max()) < 3.0


# ---- the exact network through every path ------------------------------------------------------------------------------
PATHS = ("forward", "tiles")


class Runner:
    """One exact network behind InferenceNet(tower="hand"), with a host-mapped fault word: a barrier that times out
    writes its id there before it traps."""

    def __init__(self, model):
        from harmonies_alphazero_b200 import net as hnet

        self.inf = hnet.InferenceNet(model, device="cuda", tower="hand")
        assert self.inf.wants_tiles
        self.fault = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.inf.hand.fault = self.fault.data_ptr()

    def inputs(self, board, glob):
        B = board.shape[0]
        b40 = torch.zeros((B, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
        b40[:, :38] = board
        x0 = self.inf.hand.x0_buffer(B)
        self.inf.hand.to_tiles(b40, 40, True, x0)
        return b40, x0, glob.to(torch.bfloat16).contiguous()

    def run(self, path, b40, x0, gl, n_active=None, out=None):
        inf, B = self.inf, gl.shape[0]
        if path == "forward":                    # hand tower + hz_net_heads (k_heads_p)
            res = inf(b40, gl, out=out)
        else:                                    # the tile path: head item in the tower, then k_heads_fc_mma
            res = inf.forward_tiles(x0, gl, B, out=out, n_active=n_active)
        torch.cuda.synchronize()
        assert int(self.fault[0]) == 0, f"{path}: barrier time-out {int(self.fault[0]):#x}"
        return tuple(t.clone() for t in res)


@pytest.fixture(scope="module")
def exact8():
    """the default network (8 blocks), N_MAX boards and their fp64 reference"""
    model = exact_model()
    board, glob = exact_inputs(N_MAX)
    ref = reference(model, board, glob, device="cuda")
    torch.cuda.synchronize()
    return dict(model=model, run=Runner(model), board=board.cuda(), glob=glob.cuda(), ref=ref)


def _check_paths(run, board, glob, ref, sizes, paths=PATHS, ctas=0):
    run.inf.hand.lib.hz_tower_set_max_ctas(ctas)
    try:
        for B in sizes:
            b40, x0, gl = run.inputs(board[:B], glob[:B])
            for path in paths:
                assert_exact(run.run(path, b40, x0, gl), ref, B, f"{path}, {B} boards, max_ctas {ctas}")
    finally:
        run.inf.hand.lib.hz_tower_set_max_ctas(0)


@pytest.mark.gpu
@pytest.mark.parametrize("B", SIZES)
def test_every_path_is_exact(exact8, B):
    """4,096 rows are a self-play step, 16,384 a virtual-loss step with K = 4 (DESIGN §5); at 16,384 boards a cluster
    hands about 125 items through its 64-slot mailbox, so the slot index wraps"""
    _check_paths(exact8["run"], exact8["board"], exact8["glob"], exact8["ref"], [B])


@pytest.mark.gpu
@pytest.mark.parametrize("B", [33, 203, 4103, 16384])
def test_active_prefix_is_exact_and_leaves_the_rest(exact8, B):
    run, ref = exact8["run"], exact8["ref"]
    b40, x0, gl = run.inputs(exact8["board"][:B], exact8["glob"][:B])
    na = torch.zeros(1, dtype=torch.int32, device="cuda")
    for k in (0, 1, 16, 17, 31, 32, 33, B - 1, B):
        na.fill_(k)
        out = (torch.full((B, 143), SENTINEL, device="cuda"), torch.full((B,), SENTINEL, device="cuda"))
        logits, value = run.run("tiles", b40, x0, gl, n_active=na, out=out)
        assert_exact((logits, value), ref, k, f"tiles, {B} boards, n_active {k}")
        assert bool((logits[k:] == SENTINEL).all()) and bool((value[k:] == SENTINEL).all()), k


@pytest.mark.gpu
@pytest.mark.parametrize("ctas", [1, 2, 3, 5])
def test_small_grids_are_exact(exact8, ctas):
    """many tiles through few CTAs: odd grids, a grid of one (no clusters), odd tile counts (4,103 boards = 257 tiles)"""
    _check_paths(exact8["run"], exact8["board"], exact8["glob"], exact8["ref"], [203, 4103], ctas=ctas)


@pytest.mark.gpu
def test_mailbox_slot_and_tag_wrap(exact8):
    """One cluster (max_ctas = 2) at 8,192 boards: 256 pairs of tiles x 18 items = 4,608 items through one mailbox, so
    both the slot index (k & 63) and the tag (k % 4095 + 1) wrap; 4,352 without the head item."""
    _check_paths(exact8["run"], exact8["board"], exact8["glob"], exact8["ref"], [8192], paths=("tiles", "forward"), ctas=2)


@pytest.mark.gpu
@pytest.mark.parametrize("blocks", [0, 1, 9])
def test_other_depths_are_exact(blocks):
    """MAX_LAYERS = 20 admits 0..9 residual blocks with the head item (8 is the default, above)"""
    model = exact_model(blocks=blocks)
    board, glob = exact_inputs(4103, seed=blocks)
    ref = reference(model, board, glob, device="cuda", stats=False)
    _check_paths(Runner(model), board.cuda(), glob.cuda(), ref, [17, 4103])


@pytest.mark.gpu
def test_ten_blocks_are_refused():
    run = Runner(exact_model(blocks=10))
    ht = run.inf.hand
    b40, x0, gl = run.inputs(*[t.cuda() for t in exact_inputs(16)])
    buf = ht._buffers(16)
    st = torch.cuda.current_stream().cuda_stream
    for heads in (True, False):
        res = ct.c_void_p()
        hw, hb, hc = (ht._head_w.data_ptr(), ht._head_b.data_ptr(), ht.head_conv(16).data_ptr()) if heads else (None, None, None)
        code = ht.lib.hz_tower_forward_heads(x0.data_ptr(), ht._w_ptrs, ht._b_ptrs, 10, buf["a"].data_ptr(), buf["b"].data_ptr(),
                                             buf["c"].data_ptr(), buf["sched"].data_ptr(), ct.byref(res), 16, None, hw, hb, hc,
                                             run.fault.data_ptr(), st)
        assert code == HZ_ERR_ARG, (heads, code)
    from harmonies_alphazero_b200 import _lib

    with pytest.raises(_lib.HarmoniesLibraryError):
        run.run("tiles", b40, x0, gl)


@pytest.mark.gpu
@pytest.mark.parametrize("B", SIZES)
def test_generic_heads_kernel_on_the_test_size_net(B):
    """hz_net_heads with C = 32, H = 64 (k_heads, the generic kernel), fed the exact tower output directly"""
    from harmonies_alphazero_b200 import net as hnet

    model = exact_model(hnet.TEST_MODEL_CONFIG, blocks=1)
    board, glob = exact_inputs(B, seed=3)
    ref = reference(model, board, glob, device="cuda", stats=False)
    inf = hnet.InferenceNet(model, device="cuda", tower="cudnn")
    assert inf.heads is not None and inf.heads["C"] == 32
    x = ref["tower"].to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    got = inf._fused_heads(x, glob.cuda().to(torch.bfloat16), None)
    torch.cuda.synchronize()
    assert_exact(got, ref, B, f"k_heads, {B} boards")


# ---- split precision: real-valued weights with large low parts -------------------------------------------------------
def split_bound(wx, wx_b, n_terms, c):
    """Bound on |kernel - exact| for one output sum_j w_j x_j + b computed from bf16 hi + lo splits in fp32.

    Splitting: for v = hi + lo + e with hi = bf16(v), lo = bf16(v - hi): |v - hi| <= 2^-8 |v| (half an ulp of an 8-bit
    significand), |lo| <= 2^-8 (1 + 2^-8) |v| and |e| <= 2^-8 |v - hi| <= 2^-16 |v|.
    * weights split, inputs bf16 (the head item, k_heads_p's head convolution): the products x hi and x lo are exact
      in fp32, the dropped part is x e: c = 1.
    * both split, three products kept (k_heads_fc_mma: wh xh + wh xl + wl xh): w x minus the kept products is
      wl xl + (wh + wl) ex + ew x, at most (2^-16 (1 + 2^-8)^2 + (1 + 2^-16) 2^-16 + 2^-16) |w||x|: c = 3.02 < 3.1.
    Accumulation: ``n_terms`` fp32 additions, each off by at most one ulp of the running sum even when the tensor core
    truncates, so at most n_terms 2^-23 (sum |terms|) with sum |terms| <= (1 + 2^-7) wx + |b| = ``wx_b``."""
    return c * 2.0 ** -16 * wx + n_terms * 2.0 ** -23 * wx_b


def big_lo_weights(shape, scale, g):
    """fp32 weights whose bf16 low part is 0.3-0.45 ulp of the high part, always positive: a dropped low product then
    shifts every output the same way"""
    hi = (torch.randn(shape, generator=g) * scale).to(torch.bfloat16).float()
    _, e = torch.frexp(hi)
    return hi + torch.pow(2.0, e.float() - 8) * (0.3 + 0.15 * torch.rand(shape, generator=g))


def _split(v):
    hi = v.float().to(torch.bfloat16).double()
    return hi, (v.float().double() - hi).float().to(torch.bfloat16).double()


def _head_conv_ref(x, w, b):
    """x [B,128,5,7] fp64 tower output, w [3,128], b [3] -> relu(conv + b) [B,3,35] fp64, sum |w||x| [B,3,35]"""
    xf = x.flatten(2)
    return torch.relu(torch.einsum("oc,bcp->bop", w, xf) + b.view(1, 3, 1)), torch.einsum("oc,bcp->bop", w.abs(), xf)


def _fc_ref(v, w, b):
    return v @ w.t() + b, v.abs() @ w.abs().t()


HEAD_ITEM_TERMS = 130      # 128 channels per accumulator (hi rows and lo rows apart), then hi + lo + bias
HEADS_P_TERMS = 257        # 2 x 128 products chained through the mma.sync accumulator, then the bias
FC_TERMS = 3 * 112 + 1     # three products per policy_fc input, after the bias


def real_heads(seed=0):
    """conv weights/biases of the three 1x1 head filters and policy_fc weights, real-valued with large low parts"""
    g = torch.Generator().manual_seed(500 + seed)
    w_conv = big_lo_weights((3, 128), 0.02, g)
    b_conv = torch.randn(3, generator=g) * 10
    w_fc = big_lo_weights((143, 112), 0.1, g)
    return w_conv, b_conv, w_fc, torch.randn(143, generator=g)


def test_split_bounds_catch_one_dropped_low_product():
    """Host-side negative control on the tower's own activations (the exact network, 64 boards): the fp64 model of each
    split path meets its bound, and the same model with any one low product dropped violates it."""
    board, glob = exact_inputs(64)
    x = reference(exact_model(), board, glob, stats=False)["tower"]
    w, b, wf, bf = (t.double() for t in real_heads())
    hc, wx = _head_conv_ref(x, w, b)
    for terms in (HEAD_ITEM_TERMS, HEADS_P_TERMS):
        bound = split_bound(wx, wx * (1 + 2 ** -7) + b.abs().view(1, 3, 1), terms, 1.0)
        hi, lo = _split(w)
        kept = torch.relu(torch.einsum("oc,bcp->bop", hi, x.flatten(2)) + torch.einsum("oc,bcp->bop", lo, x.flatten(2)) + b.view(1, 3, 1))
        assert bool(((kept - hc).abs() <= bound).all())
        dropped = torch.relu(torch.einsum("oc,bcp->bop", hi, x.flatten(2)) + b.view(1, 3, 1))
        assert float(((dropped - hc).abs() / bound).max()) > 4
    # policy_fc on the head convolution's (fp32) output and the global features
    v = torch.cat((hc[:, :2].flatten(1).float().double(), glob.double()), 1)
    want, vw = _fc_ref(v, wf, bf)
    bound = split_bound(vw, vw * (1 + 2 ** -7) + bf.abs(), FC_TERMS, 3.1)
    (wh, wl), (vh, vl) = _split(wf), _split(v)
    products = {"hi*hi": vh @ wh.t(), "hi*lo": vl @ wh.t(), "lo*hi": vh @ wl.t()}
    assert bool(((sum(products.values()) + bf - want).abs() <= bound).all())
    for drop in ("hi*lo", "lo*hi"):
        got = sum(p for k, p in products.items() if k != drop) + bf
        assert float(((got - want).abs() / bound).max()) > 4, drop


def _with_real_heads(model, w_conv, b_conv):
    with torch.no_grad():
        model.policy_conv.weight.copy_(w_conv[:2].view(2, 128, 1, 1))
        model.policy_conv.bias.copy_(b_conv[:2])
        model.value_conv.weight.copy_(w_conv[2:].view(1, 128, 1, 1))
        model.value_conv.bias.copy_(b_conv[2:])
    assert_bn_folds_exactly(model)         # BatchNorm scale 1.0: the folded filters are these fp32 values
    return model


@pytest.mark.gpu
def test_head_item_and_tensor_core_fc_meet_the_split_bound(exact8):
    """The tower's head item (pack_head_weight: bf16 hi rows 0..2, lo rows 3..5), then k_heads_fc_mma (three products)
    on the head item's own output, each against fp64 within ``split_bound``; the tower itself is the exact one."""
    w, b, wf, bf = real_heads()
    model = _with_real_heads(exact_model(), w, b)
    with torch.no_grad():
        model.policy_fc.weight.copy_(wf)
        model.policy_fc.bias.copy_(bf)
    run = Runner(model)
    B = 203
    b40, x0, gl = run.inputs(exact8["board"][:B], exact8["glob"][:B])
    logits, _ = run.run("tiles", b40, x0, gl)
    hc = run.inf.hand.head_conv(B).view(-1, 3, 35, 16).permute(0, 3, 1, 2).reshape(-1, 3, 35)[:B].double()
    x = exact8["ref"]["tower"][:B]
    wd, bd = w.double().cuda(), b.double().cuda()
    want, wx = _head_conv_ref(x, wd, bd)
    assert float(wx.max()) > 1e3                                    # inputs at the integer tower's scale
    bound = split_bound(wx, wx * (1 + 2 ** -7) + bd.abs().view(1, 3, 1), HEAD_ITEM_TERMS, 1.0)
    err = (hc - want).abs()
    assert bool((err <= bound).all()), f"head item: {float((err / bound).max())} x the bound"
    v = torch.cat((hc[:, :2].flatten(1), exact8["glob"][:B].double()), 1)
    want, vw = _fc_ref(v, wf.double().cuda(), bf.double().cuda())
    bound = split_bound(vw, vw * (1 + 2 ** -7) + bf.double().cuda().abs(), FC_TERMS, 3.1)
    err = (logits.double() - want).abs()
    assert bool((err <= bound).all()), f"k_heads_fc_mma: {float((err / bound).max())} x the bound"


@pytest.mark.gpu
def test_heads_p_head_convolution_meets_the_split_bound(exact8):
    """k_heads_p's head convolution (mma.sync, filters split into bf16 hi + lo) is read through FC layers that copy it:
    policy_fc passes the 70 policy cells through (weights 0 and 1 are exact in the fp32 FMAs), value_fc1 the 35 value
    cells, and value_fc2 sums them at 2^-12 before tanh."""
    w, b, _, _ = real_heads(1)
    model = _with_real_heads(exact_model(), w, b)
    with torch.no_grad():
        model.policy_fc.weight.zero_()
        model.policy_fc.weight[:70, :70] = torch.eye(70)
        model.policy_fc.bias.zero_()
        model.value_fc1.weight.zero_()
        model.value_fc1.weight[:35, :35] = torch.eye(35)
        model.value_fc1.bias.zero_()
        model.value_fc2.weight.zero_()
        model.value_fc2.weight[0, :35] = 2.0 ** -12
        model.value_fc2.bias.zero_()
    run = Runner(model)
    B = 4103
    b40, x0, gl = run.inputs(exact8["board"][:B], exact8["glob"][:B])
    logits, value = run.run("forward", b40, x0, gl)
    x = exact8["ref"]["tower"][:B]
    bd = b.double().cuda()
    want, wx = _head_conv_ref(x, w.double().cuda(), bd)
    bound = split_bound(wx, wx * (1 + 2 ** -7) + bd.abs().view(1, 3, 1), HEADS_P_TERMS, 1.0)
    err = (logits[:, :70].double() - want[:, :2].flatten(1)).abs()
    assert bool((err <= bound[:, :2].flatten(1)).all()), f"k_heads_p policy filters: {float((err / bound[:, :2].flatten(1)).max())} x the bound"
    assert bool((logits[:, 70:] == 0).all())
    # value: s = 2^-12 sum_cells relu(conv); the reduction over 256 units is at most 11 fp32 additions deep (bound: 40)
    s = want[:, 2].sum(1) * 2.0 ** -12
    ds = bound[:, 2].sum(1) * 2.0 ** -12 + 40 * 2.0 ** -24 * s
    assert 0.2 < float(s.median()) < 2                              # tanh is not saturated, the value filter is live
    err = (value.double() - torch.tanh(s)).abs()
    assert bool((err <= ds + 2 * _ulp32(torch.tanh(s))).all()), "k_heads_p value filter"


# ---- the fused softmax of hz_tree_expand_backup (is_logits = 1) -------------------------------------------------------
SOFTMAX_ROWS = ("equal", "dominant", "spread", "offset", "max_illegal", "neg_inf")


def softmax_rows(legal, g):
    """[n,143] fp32 logits, row type i % 6 (SOFTMAX_ROWS); every row has a logit >= 89, so exp without the max shift
    overflows fp32 on every row"""
    n = legal.shape[0]
    kind = torch.arange(n) % len(SOFTMAX_ROWS)
    u = torch.rand((n, 143), generator=g)
    pick = lambda mask: (torch.rand((n, 143), generator=g) + mask.float() * 2).argmax(1)   # noqa: E731  a random entry of mask
    rows = torch.arange(n)
    l = torch.full((n, 143), 100.0)                                                   # equal
    dom = u * 40
    dom[rows, pick(legal)] = 100.0                                                    # +60 over everything else
    spread = u * 200 - 100
    a1 = pick(legal)
    spread[rows, a1] = 100.0
    spread[rows, pick(legal & (torch.arange(143).view(1, -1) != a1.view(-1, 1)))] = -100.0   # exp(-200) is 0 in fp32
    offset = 1e4 + torch.randn((n, 143), generator=g)
    max_ill = 90 + 3 * torch.randn((n, 143), generator=g)
    max_ill[rows, pick(~legal)] = 130.0
    ninf = torch.where(legal, 95 + 3 * torch.randn((n, 143), generator=g), torch.tensor(float("-inf")))
    for i, t in enumerate((l, dom, spread, offset, max_ill, ninf)):
        l = torch.where((kind == i).view(-1, 1), t, l)
    return l.float().contiguous(), kind


def test_softmax_rows_need_the_max_shift():
    g = torch.Generator().manual_seed(2)
    legal = torch.rand((600, 143), generator=g) < 0.3
    logits, _ = softmax_rows(legal, g)
    assert bool(torch.isinf(torch.exp(logits)).any(dim=1).all())


@pytest.mark.gpu
def test_fused_softmax_per_edge_bound():
    """P of every root edge after one simulation over 4,096 trees against fp64 softmax over all 143 logits.

    The kernel computes m = max l (exact), e_a = expf(l_a - m), S = sum of the 143 e_i in fp32 (five per lane, then five
    shuffle rounds: at most 9 additions deep) and P_a = e_a * (1 / S).  Relative errors, in units of 2^-24:
    l_a - m rounds by at most |l_a - m| (exp turns an absolute argument error into a relative one); expf is within
    2 ulp = 4; S: each e_i carries |l_i - m| + 4 and sum_i e_i |l_i - m| / S <= 142 max_x x e^-x < 53 (S >= 1, the
    maximum contributes exp(0) = 1), + 4, + 9 for the additions = 66; the division and the product 1 each.  Together
    |l_a - m| + 72 (second order terms are far below 1): the test allows |l_a - m| + 150.  Below the normal range the
    fp32 results are denormal, and expf and the product are exact there only to 2 x 2^-149 + 2^-150 absolute: the
    floor is 2^-147."""
    from harmonies_alphazero_b200 import batched as hb
    from harmonies_alphazero_b200 import tree as tr

    n = 4096
    st = hb.init_states(n, seed=21)
    hb.playout(st, max_steps=11)
    keys = tr.search_keys_tensor(np.arange(n, dtype=np.uint64) + 5)
    t = tr.BatchedMCTS(n, 2)
    value = torch.zeros(n, device="cuda")
    t.reset(st, keys)
    t.select(2.0)
    t.expand_backup(torch.zeros((n, 143), device="cuda"), value)
    legal = (t.root_edges()[3] >= 0).cpu()
    assert bool(legal.any(dim=1).all())
    logits, kind = softmax_rows(legal, torch.Generator().manual_seed(3))
    t.reset(st, keys)
    t.select(2.0)
    t.expand_backup(logits.cuda(), value, is_logits=True)
    _, _, P, child = t.root_edges()
    t.check_status()
    assert torch.equal((child >= 0).cpu(), legal)
    l = logits.double()
    m = l.max(dim=1, keepdim=True).values
    e = torch.exp(l - m)
    want = e / e.sum(dim=1, keepdim=True)
    dist = torch.where(legal, (l - m).abs(), torch.zeros(()))
    bound = (dist + 150) * 2.0 ** -24 * want + 2.0 ** -147
    err = torch.where(legal, (P.cpu().double() - want).abs(), torch.zeros(()))
    for i, name in enumerate(SOFTMAX_ROWS):
        rows = kind == i
        r = err[rows] / bound[rows]
        assert float(r.max()) <= 1.0, f"{name}: {float(r.max())} x the bound"
    assert bool((want[legal] < 2.0 ** -126).any())          # the denormal range is exercised (spread rows)
