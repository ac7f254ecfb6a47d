"""CPU: the C-ABI library loads and exports every symbol include/harmonies_b200.h declares
(no compute calls), device-side constant tables match the reference geometry, and the host
packer round-trips."""

import ctypes
import os
import re

import numpy as np
import pytest

from tests.conftest import ROOT, load_golden
from harmonies_alphazero_b200 import constants as K
from harmonies_alphazero_b200 import packed as pk

HEADER = os.path.join(ROOT, "include", "harmonies_b200.h")
CORE = os.path.join(ROOT, "harmonies_alphazero_b200", "csrc", "hz_core.cuh")


def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hz_[a-z_0-9]+)\s*\(", src)))


@pytest.fixture(scope="module")
def built_lib():
    from harmonies_alphazero_b200 import build

    return build.build()


def test_library_exports_every_declared_symbol(built_lib):
    from harmonies_alphazero_b200 import _lib

    syms = _declared_symbols()
    assert len(syms) >= 24
    lib = ctypes.CDLL(built_lib)
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in harmonies_b200.h but not exported"
    # the Python binding declares a signature for each of them, and nothing else
    assert sorted(_lib.SIGNATURES) == syms
    loaded = _lib.load()
    assert loaded.hz_abi_version() == 6
    assert loaded.hz_status_string(-4).decode().startswith("workspace")
    assert loaded.hz_launch_count() == 0
    assert loaded.hz_tree_workspace_bytes(4096, 100, 0, 1) > 4096 * 6901 * 128
    assert loaded.hz_tree_workspace_bytes(4096, 100, 0, 8) > loaded.hz_tree_workspace_bytes(4096, 100, 0, 1)
    assert loaded.hz_tree_workspace_bytes(4096, 100, 0, 0) == 0


def test_missing_library_fails_loudly(tmp_path):
    from harmonies_alphazero_b200 import _lib

    with pytest.raises(_lib.HarmoniesLibraryError):
        _lib.load(str(tmp_path / "nope.so"))


def test_device_tables_match_reference_geometry():
    """NBR / HEX_CELL / CELL_HEX / INIT_BAG literals in hz_core.cuh vs constants.py"""
    src = open(CORE).read()

    def table(name):
        m = re.search(name + r"\[\d+\]\s*=\s*\{(.*?)\}", src, flags=re.S)
        return [int(x.rstrip("u"), 0) for x in re.findall(r"0x[0-9A-Fa-f]+u?|\d+", m.group(1))]

    assert table("NBR") == K.NEIGHBOR_MASKS
    assert table("HEX_CELL") == [y * 7 + x for (y, x) in K.HEX_CELL]
    cell_hex = [31] * 35
    for i, (y, x) in enumerate(K.HEX_CELL):
        cell_hex[y * 7 + x] = i
    assert table("CELL_HEX") == cell_hex
    assert table("INIT_BAG") == K.INITIAL_BAG_BY_TYPE
    # the generated neighbour-expansion LUT is in sync with the geometry
    from harmonies_alphazero_b200 import gen_tables

    assert open(gen_tables.PATH).read() == gen_tables.render()
    lut = gen_tables.table()
    for m in (0x1, 0x7FFFFF, 0x155555, 0x0A0A0A):
        want = 0
        for i in range(23):
            if (m >> i) & 1:
                want |= K.NEIGHBOR_MASKS[i]
        assert lut[m & 255] | lut[256 + ((m >> 8) & 255)] | lut[512 + (m >> 16)] == want
    # neighbourhood is symmetric, degree histogram of the 5-4-5-4-5 grid (SURVEY App. B)
    deg = [bin(m).count("1") for m in K.NEIGHBOR_MASKS]
    assert sorted(deg) == sorted([2] * 4 + [3] * 2 + [4] * 6 + [5] * 4 + [6] * 7)
    for i, m in enumerate(K.NEIGHBOR_MASKS):
        for j in range(23):
            assert ((m >> j) & 1) == ((K.NEIGHBOR_MASKS[j] >> i) & 1)


def test_pack_unpack_roundtrip():
    g = load_golden("engine")
    for w in np.concatenate([g["before"][::97], g["after"][-3:]]):
        f = pk.unpack_fields(w)
        keys = {k: f.pop(k) for k in ("rng_key", "rng_event", "moves")}
        w2 = pk.pack_fields(**f, rng_key=keys["rng_key"], rng_event=keys["rng_event"], moves=keys["moves"])
        assert np.array_equal(w2, w)
    with pytest.raises(ValueError):
        pk.pack_fields([{(9, 9): ["water"]}, {}], {}, [], 0, [], "choose_pile")
    with pytest.raises(ValueError):
        pk.pack_fields([{(0, 0): ["lava"]}, {}], {}, [], 0, [], "choose_pile")
    with pytest.raises(ValueError):
        pk.pack_fields([{}, {}], {}, [], 0, [], "thinking")
    assert pk.action_to_move(3) == 3
    assert pk.action_to_move(5 + 23 * 2 + 11) == ("wood", (0, 0))
    assert pk.mask_to_actions(pk.actions_to_mask([0, 4, 31, 32, 142])) == [0, 4, 31, 32, 142]


def test_draw_source_is_uniform_without_replacement():
    """the counter-based draw is a permutation-uniform sample from the multiset bag"""
    counts = np.zeros(6)
    n = 4000
    for i in range(n):
        bag = list(pk.INITIAL_BAG_COUNTS)
        tiles = pk.draw_pile(bag, pk.rand(12345, i))
        assert len(tiles) == 3 and sum(bag) == 117
        for t in tiles:
            counts[t] += 1
    expect = np.array(pk.INITIAL_BAG_COUNTS) / 120 * 3 * n
    assert np.abs(counts - expect).max() < 5 * np.sqrt(expect.max())
    bag = [0, 0, 1, 0, 1, 0]
    assert sorted(pk.draw_pile(bag, pk.rand(1, 1))) == [2, 4] and bag == [0] * 6
    assert pk.draw_pile([0] * 6, 99) == []


def _golden_net():
    import torch

    from harmonies_alphazero_b200 import net

    g = load_golden("net")
    cfg = dict(net.DEFAULT_MODEL_CONFIG, **{k[4:]: int(g[k]) for k in g.files if k.startswith("cfg_")})
    m = net.AlphaZeroNet.from_config(cfg)
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")}
    m.load_state_dict(sd, strict=True)          # same parameter AND buffer names as model.py:277-323
    return g, m.eval()


def test_network_is_the_reference_model():
    """a17: tests/golden/net.npz holds the state_dict, inputs and outputs of the reference's own
    AlphaZeroModel (model.py:277-357, eval mode).  Our module loads that state_dict strictly
    and reproduces logits / value; the BatchNorm-folded inference copy agrees to fp32 noise.
    Tolerance: 1e-5 absolute (fp32 conv summation order)."""
    import torch

    from harmonies_alphazero_b200 import net

    g, m = _golden_net()
    b, gl = torch.from_numpy(g["board"]), torch.from_numpy(g["glob"])
    with torch.no_grad():
        logits, value = m(b, gl)
    assert np.abs(logits.numpy() - g["logits"]).max() < 1e-5 and np.abs(value.numpy().reshape(-1) - g["value"]).max() < 1e-5
    inf = net.InferenceNet(m, device="cpu", dtype=torch.float32)
    l2, v2 = inf(b, gl)
    assert np.abs(l2.numpy() - g["logits"]).max() < 1e-4 and np.abs(v2.numpy() - g["value"]).max() < 1e-5
    assert np.abs(torch.softmax(l2, 1).numpy() - g["probs"]).max() < 1e-5      # ModelManager.predict: unmasked softmax


def test_tower_weight_images_follow_the_documented_layout():
    """tower.pack_conv_weight / pack_head_weight (host side of hz_tower_forward_heads): element (tap, out o, in i) of the folded
    weights sits where include/harmonies_b200.h says the K-major SWIZZLE_128B tile keeps it — half i // 64, row o of 128
    bytes, 16-byte group ((i % 64) // 8) ^ (o & 7), element i % 8 — and the head filters are split into bf16 high + low rows
    whose sum reproduces the fp32 filter to 2^-16 relative."""
    import torch

    from harmonies_alphazero_b200 import tower

    g = torch.Generator().manual_seed(3)
    w = torch.randn((128, 128, 3, 3), generator=g)
    img, nkh = tower.pack_conv_weight(w)
    assert nkh == 2 and tuple(img.shape) == (9, 2, 128, 128) and img.dtype == torch.uint8
    as_bf16 = img.view(torch.bfloat16).reshape(9, 2, 128, 64)          # [tap][half][row o][64 elements of the row]
    wb = w.to(torch.bfloat16)
    rng = np.random.default_rng(0)
    for _ in range(300):
        tap, o, i = int(rng.integers(9)), int(rng.integers(128)), int(rng.integers(128))
        half, grp, e = i // 64, (i % 64) // 8, i % 8
        pos = ((grp ^ (o & 7)) * 8) + e
        assert as_bf16[tap, half, o, pos] == wb[o, i, tap // 3, tap % 3]
    # 38 input planes (the stem): one half, planes 38..63 zero
    ws = torch.randn((128, 38, 3, 3), generator=g)
    simg, snkh = tower.pack_conv_weight(ws)
    assert snkh == 1
    sb = simg.view(torch.bfloat16).reshape(9, 1, 128, 64)
    assert float(sb.float().abs().sum()) == pytest.approx(float(ws.to(torch.bfloat16).float().abs().sum()), rel=1e-6)
    # head filters: rows 0..2 high parts, rows 3..5 low parts, the rest zero
    wh = torch.randn((3, 128), generator=g) * 0.3
    himg, hnkh = tower.pack_head_weight(wh)
    assert hnkh == 2 and tuple(himg.shape) == (2, 128, 128)
    hb = himg.view(torch.bfloat16).reshape(2, 128, 64).float()
    assert float(hb[:, 6:, :].abs().max()) == 0.0
    for j in range(3):
        for i in (0, 7, 8, 63, 64, 100, 127):
            half, grp, e = i // 64, (i % 64) // 8, i % 8
            hi = hb[half, j, ((grp ^ (j & 7)) * 8) + e]
            lo = hb[half, j + 3, ((grp ^ ((j + 3) & 7)) * 8) + e]
            assert abs(float(hi + lo) - float(wh[j, i])) <= abs(float(wh[j, i])) * 2.0 ** -15 + 1e-12
