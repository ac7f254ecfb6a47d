"""Policy/value network for batched leaf evaluation.

north_star keeps the network a PyTorch forward on tensor cores ("the only dense
contraction").  Two classes:

* ``AlphaZeroNet`` — the reference architecture (model.py:277-357: 3x3 conv stem, N residual
  blocks, 1x1-conv policy/value heads whose FC layers also take the 42 global features) with
  the SAME parameter names, so ``load_state_dict`` accepts the reference's checkpoints
  (``model_state_dict`` of ModelManager.save_checkpoint, model.py:161-182) and vice versa.
* ``InferenceNet`` — what self-play actually runs: eval-mode BatchNorm folded into the
  convolutions, bf16 (or fp32) weights in channels-last layout, bias+ReLU(+residual) fused into
  the cuDNN convolution call, meant to be captured in a CUDA graph together with the tree
  kernels.  ``predict`` mirrors ModelManager.predict (model.py:81-110) for a batch.
"""

import torch
from torch import nn
import torch.nn.functional as F

from .constants import ACTION_SIZE, BOARD_SIZE, GLOBAL_FEATURE_SIZE, INPUT_CHANNELS

DEFAULT_MODEL_CONFIG = {  # config.py:18-29
    "input_channels": INPUT_CHANNELS,
    "cnn_filters": 128,
    "board_size": BOARD_SIZE,
    "action_size": ACTION_SIZE,
    "global_feature_size": GLOBAL_FEATURE_SIZE,
    "value_head_hidden_dim": 256,
    "num_res_blocks": 8,
    "policy_head_conv_filters": 2,
    "value_head_conv_filters": 1,
}
TEST_MODEL_CONFIG = dict(DEFAULT_MODEL_CONFIG, cnn_filters=32, value_head_hidden_dim=64, num_res_blocks=1)  # config.py:103-113


class _Block(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv1 = nn.Conv2d(c, c, 3, padding=1)
        self.bn1 = nn.BatchNorm2d(c)
        self.conv2 = nn.Conv2d(c, c, 3, padding=1)
        self.bn2 = nn.BatchNorm2d(c)

    def forward(self, x):
        y = F.relu(self.bn1(self.conv1(x)))
        return F.relu(self.bn2(self.conv2(y)) + x)


class AlphaZeroNet(nn.Module):
    def __init__(self, input_channels=INPUT_CHANNELS, cnn_filters=128, board_size=BOARD_SIZE, action_size=ACTION_SIZE,
                 global_feature_size=GLOBAL_FEATURE_SIZE, value_head_hidden_dim=256, num_res_blocks=8,
                 policy_head_conv_filters=2, value_head_conv_filters=1):
        super().__init__()
        h, w = board_size
        self.conv = nn.Conv2d(input_channels, cnn_filters, 3, padding=1)
        self.bn = nn.BatchNorm2d(cnn_filters)
        self.residual_blocks = nn.ModuleList(_Block(cnn_filters) for _ in range(num_res_blocks))
        self.policy_conv = nn.Conv2d(cnn_filters, policy_head_conv_filters, 1)
        self.policy_bn = nn.BatchNorm2d(policy_head_conv_filters)
        self.policy_fc = nn.Linear(policy_head_conv_filters * h * w + global_feature_size, action_size)
        self.value_conv = nn.Conv2d(cnn_filters, value_head_conv_filters, 1)
        self.value_bn = nn.BatchNorm2d(value_head_conv_filters)
        self.value_fc1 = nn.Linear(value_head_conv_filters * h * w + global_feature_size, value_head_hidden_dim)
        self.value_fc2 = nn.Linear(value_head_hidden_dim, 1)

    @classmethod
    def from_config(cls, cfg):
        return cls(**{k: cfg[k] for k in DEFAULT_MODEL_CONFIG if k in cfg})

    def forward(self, x_board, x_global):
        x = F.relu(self.bn(self.conv(x_board)))
        for blk in self.residual_blocks:
            x = blk(x)
        p = F.relu(self.policy_bn(self.policy_conv(x))).flatten(1)
        logits = self.policy_fc(torch.cat((p, x_global), dim=1))
        v = F.relu(self.value_bn(self.value_conv(x))).flatten(1)
        v = F.relu(self.value_fc1(torch.cat((v, x_global), dim=1)))
        return logits, torch.tanh(self.value_fc2(v))


def _fold(conv, bn):
    """eval-mode BatchNorm folded into the preceding convolution (fp32 math)."""
    scale = bn.weight.detach().float() * torch.rsqrt(bn.running_var.detach().float() + bn.eps)
    w = conv.weight.detach().float() * scale.view(-1, 1, 1, 1)
    b = (conv.bias.detach().float() - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()
    return w, b


class InferenceNet:
    """Folded, channels-last inference copy of an AlphaZeroNet on one device."""

    heads_in_tower = True   # the tile path runs the 1x1 head convolutions inside the tower launch; bench.py reads it

    def __init__(self, model, device="cuda", dtype=torch.bfloat16, fused=True, fused_heads=True, tower="auto"):
        """tower: "hand" = csrc/hz_tower.cu, the hand-written sm_100a tcgen05 tower (bf16 on CUDA
        with 128 filters and <= 64 input planes; it raises for anything else, there is no silent
        fallback); "cudnn" = library convolutions (other shapes / dtypes, and the A/B switch);
        "auto" (default) = "hand" exactly when the network has the shape it supports."""
        self.device, self.dtype = torch.device(device), dtype
        self.fused = fused and self.device.type == "cuda"
        self.use_fused_heads = fused_heads
        if tower == "auto":
            ok = (self.device.type == "cuda" and dtype == torch.bfloat16 and model.conv.out_channels == 128
                  and model.conv.in_channels <= 64)
            tower = "hand" if ok else "cudnn"
        if tower not in ("cudnn", "hand"):
            raise ValueError("tower must be 'auto', 'cudnn' or 'hand'")
        if tower == "hand" and not (self.device.type == "cuda" and dtype == torch.bfloat16):
            raise ValueError("the hand-written tower is bf16 on CUDA only")
        self.tower = tower
        self.hand = None
        self.load(model)

    def load(self, model):
        """(Re)build the folded weights from ``model`` (after a weight broadcast / checkpoint).  Every load gets a new
        ``version``: drivers that captured CUDA graphs over the previous weight tensors re-capture (selfplay._Group)."""
        dev, dt = self.device, self.dtype
        self.version = getattr(self, "version", 0) + 1

        def conv_params(conv, bn):
            w, b = _fold(conv, bn)
            return (w.to(dev, dt).contiguous(memory_format=torch.channels_last), b.to(dev, dt))

        self.stem = conv_params(model.conv, model.bn)
        # same stem for a 40-channel input (channels 38, 39 are zero): C % 8 == 0 lets cuDNN run
        # the bf16 tensor-op kernel without its input-padding pre-pass (HZ_LAYOUT_NHWC40)
        w38, b38 = _fold(model.conv, model.bn)
        w40 = torch.zeros((w38.shape[0], 40, 3, 3), dtype=w38.dtype)
        w40[:, : w38.shape[1]] = w38
        self.stem40 = (w40.to(dev, dt).contiguous(memory_format=torch.channels_last), b38.to(dev, dt))
        self.blocks = [(conv_params(b.conv1, b.bn1), conv_params(b.conv2, b.bn2)) for b in model.residual_blocks]
        self.phead = conv_params(model.policy_conv, model.policy_bn)
        self.vhead = conv_params(model.value_conv, model.value_bn)
        lin = lambda l: (l.weight.detach().to(dev, dt).contiguous(), l.bias.detach().to(dev, dt))  # noqa: E731
        self.policy_fc, self.value_fc1, self.value_fc2 = lin(model.policy_fc), lin(model.value_fc1), lin(model.value_fc2)
        self._build_fused_heads(model)
        if self.tower == "hand":
            from .tower import HandTower

            self.hand = HandTower(model, dev)
            if self.heads is not None and self.heads["C"] == 128:
                self.hand.set_heads(self.heads["w_conv"], self.heads["b_conv"])
        if self.fused:
            # the fused cuDNN entry points do not cover every dtype/arch combination: probe once
            # and use conv2d + relu (still cuDNN) if they refuse
            try:
                x = torch.zeros((2, self.stem[0].shape[1], 5, 7), device=dev, dtype=dt).contiguous(memory_format=torch.channels_last)
                y = self._conv_relu(x, self.stem, 1)
                self._conv_relu(y, self.blocks[0][0] if self.blocks else self.phead, 1 if self.blocks else 0, residual=y if self.blocks else None)
                torch.cuda.synchronize(dev)
            except Exception as e:  # noqa: BLE001
                self.fused, self.fused_error = False, repr(e)

    def _conv_relu(self, x, wb, pad, residual=None):
        w, b = wb
        if self.fused:
            # one cuDNN kernel: relu(conv(x) + bias [+ residual])
            if residual is None:
                return torch.cudnn_convolution_relu(x, w, b, (1, 1), (pad, pad), (1, 1), 1)
            return torch.cudnn_convolution_add_relu(x, w, residual, 1.0, b, (1, 1), (pad, pad), (1, 1), 1)
        y = F.conv2d(x, w, b, padding=pad)
        if residual is not None:
            y = y + residual
        return F.relu(y)

    def _build_fused_heads(self, model):
        """fp32 weights for hz_net_heads (csrc/hz_heads.cu): both 1x1 head convolutions with
        BatchNorm folded, FC weights transposed so that threads read them coalesced."""
        self.heads = None
        if not (self.device.type == "cuda" and self.dtype == torch.bfloat16):
            return
        if model.policy_conv.out_channels != 2 or model.value_conv.out_channels != 1 or model.policy_fc.out_features != 143:
            return
        C = model.policy_conv.in_channels
        if C % 8 or model.policy_fc.in_features != 112 or model.value_fc1.in_features != 77:
            return
        dev = self.device
        wp, bp = _fold(model.policy_conv, model.policy_bn)
        wv, bv = _fold(model.value_conv, model.value_bn)
        f32 = lambda t: t.detach().float().contiguous().to(dev)  # noqa: E731
        self.heads = dict(
            C=C, H=model.value_fc1.out_features,
            w_conv=f32(torch.cat((wp.view(2, C), wv.view(1, C)))), b_conv=f32(torch.cat((bp, bv))),
            w_pol_t=f32(model.policy_fc.weight.t()), b_pol=f32(model.policy_fc.bias),
            w_v1_t=f32(model.value_fc1.weight.t()), b_v1=f32(model.value_fc1.bias),
            w_v2=f32(model.value_fc2.weight.view(-1)), b_v2=float(model.value_fc2.bias.item()),
        )

    def _fused_heads(self, x, glob, out):
        from . import _lib

        h = self.heads
        B = x.shape[0]
        if not x.is_contiguous(memory_format=torch.channels_last):
            x = x.contiguous(memory_format=torch.channels_last)
        glob = glob.contiguous()
        if out is None:
            out = (torch.empty((B, 143), dtype=torch.float32, device=x.device), torch.empty(B, dtype=torch.float32, device=x.device))
        logits, value = out
        lib = _lib.load()
        with torch.cuda.device(x.device):
            _lib.check(lib.hz_net_heads(
                x.data_ptr(), glob.data_ptr(), B, h["C"], h["H"], h["w_conv"].data_ptr(), h["b_conv"].data_ptr(),
                h["w_pol_t"].data_ptr(), h["b_pol"].data_ptr(), h["w_v1_t"].data_ptr(), h["b_v1"].data_ptr(),
                h["w_v2"].data_ptr(), h["b_v2"], logits.data_ptr(), value.data_ptr(),
                torch.cuda.current_stream(x.device).cuda_stream), "hz_net_heads")
        return logits, value

    # ---- leaf-evaluation plumbing shared by selfplay / arena -----------------------------------
    @property
    def wants_tiles(self):
        """True when leaves should be encoded straight into the hand-written tower's input image
        (hz_tree_select layout HZ_LAYOUT_T16K) and evaluated with ``forward_tiles``."""
        return self.hand is not None and self.heads is not None and self.use_fused_heads and self.heads["C"] == 128 and self.heads["H"] == 256

    @property
    def row_invariant(self):
        """True when a board's outputs do not depend on its row, its neighbours in the batch or the active count (the
        precondition of the leaf evaluation cache, tree.EvalCache): the tile path, whose tower and heads compute every
        board on its own with a fixed schedule.  The cuDNN path picks kernels by batch shape and promises no such thing."""
        return self.wants_tiles

    def leaf_buffers(self, rows):
        """(board, glob, logits, value) static buffers for ``rows`` leaves per step."""
        dev = self.device
        if self.wants_tiles:
            board = self.hand.x0_buffer(rows)
        else:
            cl = dev.type == "cuda"
            board = torch.empty((rows, 40 if (cl and hasattr(self, "stem40")) else 38, 5, 7), dtype=self.dtype, device=dev,
                                memory_format=torch.channels_last if cl else torch.contiguous_format).zero_()
        return (board, torch.zeros((rows, 42), dtype=self.dtype, device=dev),
                torch.zeros((rows, 143), dtype=torch.float32, device=dev), torch.zeros(rows, dtype=torch.float32, device=dev))

    @torch.no_grad()
    def forward_tiles(self, x0, glob, n, out=None, n_active=None, tag=0):
        """Leaves already in the T16K image (hz_tree_select, HZ_LAYOUT_T16K): hand-written tower, the
        1x1 head convolutions straight from its T16 output, then the FC heads.  No layout-conversion
        kernels on this path.  n_active: int32 device tensor (one element): only rows 0..n_active-1
        are evaluated (read on the device, so a captured graph follows it)."""
        from . import _lib

        if not self.wants_tiles:
            raise ValueError("forward_tiles needs tower='hand' and the default head shape")
        h = self.heads
        if out is None:
            out = (torch.empty((n, 143), dtype=torch.float32, device=self.device), torch.empty(n, dtype=torch.float32, device=self.device))
        logits, value = out
        lib = _lib.load()
        glob = glob.contiguous()
        na = None if n_active is None else n_active.data_ptr()
        # the 1x1 head convolutions run inside the tower launch, as one more work item per tile
        self.hand.forward_tiles(x0, n, n_active=n_active, tag=tag, heads=True)
        hc = self.hand.head_conv(n, tag)
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(lib.hz_net_heads_fc_active(hc.data_ptr(), glob.data_ptr(), n, na, h["H"], h["w_pol_t"].data_ptr(), h["b_pol"].data_ptr(),
                                                  h["w_v1_t"].data_ptr(), h["b_v1"].data_ptr(), h["w_v2"].data_ptr(), h["b_v2"],
                                                  logits.data_ptr(), value.data_ptr(), st), "hz_net_heads_fc")
        return logits, value

    @torch.no_grad()
    def evaluate(self, board, glob, out):
        """``board`` as produced for this net by ``leaf_buffers`` (tiles or a tensor)."""
        if self.wants_tiles:
            return self.forward_tiles(board, glob, glob.shape[0], out=out)
        return self.forward(board, glob, out=out)

    @torch.no_grad()
    def forward(self, board, glob, out=None):
        """board [B,38,5,7] (channels-last preferred), glob [B,42], both ``dtype``.
        Returns (logits fp32 [B,143], value fp32 [B]); ``out`` = preallocated pair to fill."""
        x = self.tower_out(board)
        B = x.shape[0]
        if self.heads is not None and self.use_fused_heads:
            return self._fused_heads(x, glob, out)
        if out is not None:
            logits, value = self._torch_heads(x, glob, B)
            out[0].copy_(logits)
            out[1].copy_(value)
            return out
        return self._torch_heads(x, glob, B)

    @torch.no_grad()
    def tower_out(self, board):
        """Output of the stem + residual blocks, [B,C,5,7] (channels-last on CUDA)."""
        if self.hand is not None:
            if board.shape[1] % 8:      # 38 planes: pad to the 40-plane leaf layout
                b40 = torch.zeros((board.shape[0], 40, 5, 7), dtype=self.dtype, device=self.device).contiguous(memory_format=torch.channels_last)
                b40[:, : board.shape[1]] = board
                board = b40
            elif not board.is_contiguous(memory_format=torch.channels_last):
                board = board.contiguous(memory_format=torch.channels_last)
            return self.hand.forward(board)
        x = self._conv_relu(board, self.stem40 if board.shape[1] == 40 else self.stem, 1)
        for c1, c2 in self.blocks:
            y = self._conv_relu(x, c1, 1)
            x = self._conv_relu(y, c2, 1, residual=x)
        return x

    def _torch_heads(self, x, glob, B):
        p = self._conv_relu(x, self.phead, 0).contiguous(memory_format=torch.contiguous_format).view(B, -1)
        logits = F.linear(torch.cat((p, glob), dim=1), *self.policy_fc)
        v = self._conv_relu(x, self.vhead, 0).contiguous(memory_format=torch.contiguous_format).view(B, -1)
        v = F.relu(F.linear(torch.cat((v, glob), dim=1), *self.value_fc1))
        v = torch.tanh(F.linear(v, *self.value_fc2))
        return logits.float(), v.float().view(B)

    __call__ = forward

    @torch.no_grad()
    def predict(self, board, glob):
        """Batched ModelManager.predict (model.py:81-110): softmax over ALL 143 logits (no
        legal masking), value as a scalar per position."""
        logits, v = self.forward(board.to(self.device, self.dtype), glob.to(self.device, self.dtype))
        return torch.softmax(logits, dim=1), v


def flops_per_position(cfg=DEFAULT_MODEL_CONFIG):
    """Forward FLOPs (2*MAC) of the network for one position: 168.31 MFLOP for the default
    configuration (SURVEY.md §6)."""
    h, w = cfg["board_size"]
    c, hw = cfg["cnn_filters"], h * w
    f = 2 * hw * 9 * cfg["input_channels"] * c
    f += cfg["num_res_blocks"] * 2 * (2 * hw * 9 * c * c)
    f += 2 * hw * c * (cfg["policy_head_conv_filters"] + cfg["value_head_conv_filters"])
    f += 2 * (cfg["policy_head_conv_filters"] * hw + cfg["global_feature_size"]) * cfg["action_size"]
    f += 2 * (cfg["value_head_conv_filters"] * hw + cfg["global_feature_size"]) * cfg["value_head_hidden_dim"]
    f += 2 * cfg["value_head_hidden_dim"]
    return f
