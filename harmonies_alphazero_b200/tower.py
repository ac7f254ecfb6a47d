"""Hand-written sm_100a residual tower (csrc/hz_tower.cu) behind a small Python handle.

Replaces the 17 cuDNN convolutions of the reference network's body (model.py:325-339: stem
conv+bn+relu, then ``num_res_blocks`` x ResidualBlock.forward, model.py:380-392) for the
default width (128 filters).  BatchNorm is folded in fp32 exactly as ``net._fold`` does for the
cuDNN path, weights are rounded to bf16 once, accumulation is fp32 in tensor memory.

There is no fallback: without the CUDA library every call raises.  ``InferenceNet(tower="cudnn")``
is the A/B switch for measurements.
"""

import ctypes as ct

import torch

from . import _lib

G = 16            # boards per tile
KH_BYTES = 71680  # 560 rows x 128 bytes: one 64-channel half of a tile


def pack_conv_weight(w):
    """[128, Cin, 3, 3] fp32 (BatchNorm folded) -> uint8 [9, nkh, 128, 128]: per tap (ky*3+kx) and
    64-channel half a K-major SWIZZLE_128B tile of bf16 (16-byte group g stored at g ^ (out & 7)):
    the A operand of the tower's tcgen05.mma."""
    O, I = w.shape[0], w.shape[1]
    if O != 128 or w.shape[2:] != (3, 3):
        raise ValueError("hand-written tower needs 128 output channels and 3x3 kernels")
    nkh = (I + 63) // 64
    wp = torch.zeros((O, nkh * 64, 3, 3), dtype=torch.float32)
    wp[:, :I] = w.detach().float().cpu()
    t = wp.permute(2, 3, 0, 1).reshape(9, O, nkh, 8, 8).to(torch.bfloat16)       # [tap][o][kh][g][8]
    t = t.permute(0, 2, 1, 3, 4).contiguous()                                     # [tap][kh][o][g][8]
    o = torch.arange(O).view(O, 1)
    j = torch.arange(8).view(1, 8)
    src_group = (j ^ (o & 7)).view(1, 1, O, 8, 1).expand(9, nkh, O, 8, 8)        # position j holds group j ^ (o & 7)
    img = torch.gather(t, 3, src_group).contiguous()
    return img.view(torch.uint8).reshape(9, nkh, O, 128), nkh


def pack_head_weight(w_conv):
    """[3, 128] fp32 (the two policy and the value 1x1 filters, BatchNorm folded) -> uint8 [2, 128, 128]: the head item's
    A operand (hz_tower_forward_heads): rows 0..2 = bf16 high parts, rows 3..5 = bf16 low parts (filter = hi + lo), rows
    6..127 zero; per 64-channel half a K-major SWIZZLE_128B tile like pack_conv_weight's."""
    w = w_conv.detach().float().cpu()
    hi = w.to(torch.bfloat16)
    lo = (w - hi.float()).to(torch.bfloat16)
    full = torch.zeros((128, 128, 3, 3), dtype=torch.float32)
    full[0:3, :, 1, 1] = hi.float()
    full[3:6, :, 1, 1] = lo.float()
    img, nkh = pack_conv_weight(full)          # exact: the values are bf16 already
    return img[4].contiguous(), nkh            # the centre tap: [nkh][128][128 B]


class HandTower:
    """Folded stem + residual blocks of an AlphaZeroNet on one CUDA device."""

    def __init__(self, model, device="cuda"):
        from .net import _fold

        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.HarmoniesLibraryError("the hand-written tower runs on a CUDA device only (no CPU fallback)")
        self.lib = _lib.load()
        if model.conv.out_channels != 128 or model.conv.in_channels > 64:
            raise ValueError("hand-written tower supports cnn_filters == 128 and <= 64 input planes")
        self.in_channels = model.conv.in_channels
        dev = self.device

        def conv(c, bn):
            w, b = _fold(c, bn)
            img, nkh = pack_conv_weight(w)
            return img.to(dev), b.detach().float().contiguous().to(dev), nkh

        self.stem = conv(model.conv, model.bn)
        self.blocks = [(conv(b.conv1, b.bn1), conv(b.conv2, b.bn2)) for b in model.residual_blocks]
        self._bufs = {}
        self.fault = None     # optional host-mapped fault word (tests)
        layers = [self.stem] + [cv for blk in self.blocks for cv in blk]
        self._w_ptrs = (ct.c_void_p * len(layers))(*[l[0].data_ptr() for l in layers])
        self._b_ptrs = (ct.c_void_p * len(layers))(*[l[1].data_ptr() for l in layers])

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _buffers(self, n_pad, tag=0):
        """scratch of one caller: callers that run concurrently on different streams pass different tags"""
        b = self._bufs.get((n_pad, tag))
        if b is None:
            tiles = n_pad // G
            mk = lambda halves: torch.zeros(tiles * halves * KH_BYTES, dtype=torch.uint8, device=self.device)  # noqa: E731
            b = self._bufs[(n_pad, tag)] = dict(x0=mk(1), a=mk(2), b=mk(2), c=mk(2),
                                         sched=torch.zeros(self.lib.hz_tower_sched_bytes(n_pad, len(self.blocks)), dtype=torch.uint8, device=self.device),
                                         out=torch.zeros((n_pad, 35, 128), dtype=torch.bfloat16, device=self.device))
        return b

    def to_tiles(self, src_nhwc, channels, kmajor, dst):
        """NHWC bf16 -> T16K (kmajor, <= 64 channels: the stem input) or T16 (128 channels) tiles"""
        n = src_nhwc.shape[0]
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tower_to_tiles(src_nhwc.data_ptr(), dst.data_ptr(), n, channels, 1 if kmajor else 0, self._stream()), "hz_tower_to_tiles")

    def from_tiles(self, src, n):
        out = torch.empty((n, 35, 128), dtype=torch.bfloat16, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tower_from_tiles(src.data_ptr(), out.data_ptr(), n, self._stream()), "hz_tower_from_tiles")
        return out

    def conv(self, x, halves, wb, res, y, n_pad, relu=True, kmajor=False):
        img, bias, nkh = wb
        assert nkh == halves
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tower_conv3x3(
                x.data_ptr(), halves, 1 if kmajor else 0, img.data_ptr(), bias.data_ptr(), None if res is None else res.data_ptr(),
                y.data_ptr(), n_pad, 1 if relu else 0, self.fault, self._stream()), "hz_tower_conv3x3")

    def x0_buffer(self, n):
        """Zeroed T16K input buffer for n boards (what hz_tree_select writes with HZ_LAYOUT_T16K)."""
        n_pad = (n + G - 1) // G * G
        return torch.zeros(n_pad // G * KH_BYTES, dtype=torch.uint8, device=self.device)

    @torch.no_grad()
    def set_heads(self, w_conv, b_conv):
        """1x1 head filters [3,128] + bias [3] (fp32, BatchNorm folded): forward_tiles(..., heads=True) then also runs them
        inside the tower launch and leaves relu(conv + bias) in the buffer ``head_conv(n, tag)``."""
        img, nkh = pack_head_weight(w_conv)
        assert nkh == 2
        self._head_w = img.to(self.device)
        self._head_b = b_conv.detach().float().contiguous().to(self.device)

    def head_conv(self, n, tag=0):
        n_pad = (n + G - 1) // G * G
        buf = self._buffers(n_pad, tag)
        if "hc" not in buf:
            buf["hc"] = torch.zeros(n_pad // G * 3 * 35 * G, dtype=torch.float32, device=self.device)
        return buf["hc"]

    def forward_tiles(self, x0, n, n_active=None, tag=0, heads=False):
        """x0: T16K tiles of n boards.  Returns the address of the T16 tiles holding the tower output
        (one of this object's scratch buffers: valid until the next call with the same n).
        n_active: int32 device tensor (one element) = boards to compute, read on the device."""
        n_pad = (n + G - 1) // G * G
        buf = self._buffers(n_pad, tag)
        res = ct.c_void_p()
        with torch.cuda.device(self.device):
            hw = hb = hc = None
            if heads:
                hw, hb, hc = self._head_w.data_ptr(), self._head_b.data_ptr(), self.head_conv(n, tag).data_ptr()
            _lib.check(self.lib.hz_tower_forward_heads(
                x0.data_ptr(), self._w_ptrs, self._b_ptrs, len(self.blocks), buf["a"].data_ptr(), buf["b"].data_ptr(), buf["c"].data_ptr(),
                buf["sched"].data_ptr(), ct.byref(res), n_pad, None if n_active is None else n_active.data_ptr(),
                hw, hb, hc, self.fault, self._stream()), "hz_tower_forward_heads")
        return res.value

    @torch.no_grad()
    def forward(self, board, out=None):
        """board: bf16 [B, C, 5, 7] in channels-last memory (NHWC, C = 38 or 40 with zero planes
        behind the 38), B arbitrary.  Returns the tower output as a channels-last [B,128,5,7]
        view of an NHWC buffer (what hz_net_heads reads)."""
        if board.dtype != torch.bfloat16 or not board.is_contiguous(memory_format=torch.channels_last):
            raise ValueError("HandTower.forward wants a channels-last bf16 board tensor")
        B, C = board.shape[0], board.shape[1]
        if C % 8:
            raise ValueError("channel count of the board tensor must be a multiple of 8 (use the 40-plane leaf layout)")
        n_pad = (B + G - 1) // G * G
        buf = self._buffers(n_pad)
        self.to_tiles(board, C, True, buf["x0"])
        if out is None:
            out = buf["out"]       # static: the same addresses every call (CUDA graphs)
        x_ptr = self.forward_tiles(buf["x0"], n_pad)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tower_from_tiles(x_ptr, out.data_ptr(), n_pad, self._stream()), "hz_tower_from_tiles")
        return out[:B].view(B, 5, 7, 128).permute(0, 3, 1, 2)
