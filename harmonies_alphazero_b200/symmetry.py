"""The game's symmetries (include/harmonies_b200.h "Game symmetries"): group tables, a numpy reference of the state and
action transforms, the search's leaf-frame rule, and tensor wrappers over hz_sym_states / hz_sym_actions.

An element g (0..479) is a board symmetry b = g & 3 (the four automorphisms of the 23-hex board, a Klein four-group)
and a pile permutation c = g >> 2: with m = n_piles, the pile at position i < m moves to position
``itertools.permutations(range(m))[c % m!][i]``.  T_g moves the content of hex i to hex tau_b(i) and reorders the piles;
everything else in the record stays.  Actions follow: sigma_g(a) = pi[a] (a < m), a (m <= a < 5), 5 + 23t + tau_b(h)
(a = 5 + 23t + h); a policy, visit or mask row x maps to x' with x'[sigma_g(a)] = x[a].
"""

import itertools

import numpy as np
import torch

from . import _lib, gen_tables, packed
from .batched import _check_states, _ptr, _stream
from .constants import ACTION_SIZE, NUM_HEXES, NUM_PILES

# ---- the group --------------------------------------------------------------------------------
HEX_MAPS = np.array(gen_tables.hex_maps(), dtype=np.int64)              # [4, 23]: tau_b(i)
HEX_INV = np.array(gen_tables.hex_inverse_maps(), dtype=np.int64)       # [4, 23]: tau_b^-1(i)
PILE_PERMS = [list(itertools.permutations(range(m))) for m in range(NUM_PILES + 1)]
ORDER = 480
SYMMETRY_SALT = 0x53594D4D45545259       # HZ_SYMMETRY_SALT

OFF, BOARD, FULL = 0, 1, 2               # HZ_SYM_OFF / HZ_SYM_BOARD / HZ_SYM_FULL
GROUP_SIZE = {OFF: 1, BOARD: 4, FULL: ORDER}


def mode_code(mode):
    """None / "board" / "full" (or the HZ_SYM_* integer) -> HZ_SYM_* integer."""
    if mode is None:
        return OFF
    if isinstance(mode, str):
        try:
            return {"off": OFF, "board": BOARD, "full": FULL}[mode]
        except KeyError:
            raise ValueError(f"symmetry mode must be None, 'board' or 'full', not {mode!r}") from None
    if int(mode) not in GROUP_SIZE:
        raise ValueError(f"bad symmetry mode {mode!r}")
    return int(mode)


def _perm5(g, m):
    """pile permutation of g on all five positions (identity on positions >= m)"""
    m = min(int(m), NUM_PILES)
    p = PILE_PERMS[m][(int(g) >> 2) % len(PILE_PERMS[m])]
    return list(p) + list(range(m, NUM_PILES))


def pile_perm(g, n_piles):
    """pi of element g for n_piles piles: the pile at position i moves to pi[i]."""
    return tuple(_perm5(g, n_piles)[: min(int(n_piles), NUM_PILES)])


def _perm_index(p):
    return PILE_PERMS[len(p)].index(tuple(p))


def compose(g, h, n_piles):
    """The element k with T_k = T_g o T_h (h first) on states with n_piles piles."""
    m = min(int(n_piles), NUM_PILES)
    pg, ph = _perm5(g, m), _perm5(h, m)
    return (_perm_index([pg[ph[i]] for i in range(m)]) << 2) | ((int(g) ^ int(h)) & 3)


def inverse(g, n_piles):
    """The element whose transform undoes T_g on states with n_piles piles (board part: every b is an involution)."""
    m = min(int(n_piles), NUM_PILES)
    p = _perm5(g, m)
    q = [0] * m
    for i in range(m):
        q[p[i]] = i
    return (_perm_index(q) << 2) | (int(g) & 3)


def action_perm(g, n_piles):
    """sigma_g as np.int64[143]: sigma[a] = where action a goes."""
    p = _perm5(g, n_piles)
    b = int(g) & 3
    s = np.arange(ACTION_SIZE, dtype=np.int64)
    m = min(int(n_piles), NUM_PILES)
    s[:m] = p[:m]
    t, h = np.divmod(np.arange(ACTION_SIZE - 5), NUM_HEXES)
    s[5:] = 5 + NUM_HEXES * t + HEX_MAPS[b][h]
    return s


# ---- numpy reference --------------------------------------------------------------------------
def _rows(words, g):
    w = np.array(np.asarray(words, dtype=np.uint32).reshape(-1, 32), dtype=np.uint32)
    g = np.broadcast_to(np.asarray(g, dtype=np.int64).reshape(-1), (w.shape[0],))
    return w, g


def transform_words(words, g):
    """T_g of packed records: words uint32[32] or [n, 32], g an int or int[n].  Same shape out."""
    shape = np.asarray(words).shape
    w, g = _rows(words, g)
    out = w.copy()
    src = HEX_INV[g & 3].astype(np.uint32)                                  # [n, 23]: new hex i reads old hex tau^-1(i)
    planes = np.zeros((w.shape[0], 18), dtype=np.uint32)
    for i in range(NUM_HEXES):
        planes |= ((w[:, :18] >> src[:, i:i + 1]) & np.uint32(1)) << np.uint32(i)
    out[:, :18] = planes
    piles = np.stack([w[:, 18] & 0xFFFF, w[:, 18] >> 16, w[:, 19] & 0xFFFF, w[:, 19] >> 16, w[:, 20] & 0xFFFF], axis=1)
    m = (w[:, 22] >> 16) & 0xFF
    dest = np.array([_perm5(gi, mi) for gi, mi in zip(g, m)], dtype=np.int64).reshape(-1, NUM_PILES)
    new = np.zeros_like(piles)
    np.put_along_axis(new, dest, piles, axis=1)
    out[:, 18] = new[:, 0] | (new[:, 1] << 16)
    out[:, 19] = new[:, 2] | (new[:, 3] << 16)
    out[:, 20] = new[:, 4] | (w[:, 20] & 0xFFFF0000)
    return out.reshape(shape)


def transform_action_rows(x, g, n_piles, inverse_=False):
    """x [n, 143] (or [143]) -> x' with x'[sigma_g(a)] = x[a] (inverse_: x'[a] = x[sigma_g(a)])."""
    shape = np.asarray(x).shape
    x = np.asarray(x).reshape(-1, ACTION_SIZE)
    g = np.broadcast_to(np.asarray(g, dtype=np.int64).reshape(-1), (x.shape[0],))
    m = np.broadcast_to(np.asarray(n_piles, dtype=np.int64).reshape(-1), (x.shape[0],))
    sig = np.stack([action_perm(gi, mi) for gi, mi in zip(g, m)]) if x.shape[0] else np.zeros((0, ACTION_SIZE), np.int64)
    if inverse_:
        out = np.take_along_axis(x, sig, axis=1)
    else:
        out = np.empty_like(x)
        np.put_along_axis(out, sig, x, axis=1)
    return out.reshape(shape)


def transform_mask_words(mask, g, n_piles):
    """legal-mask words uint32[5] of a state -> those of T_g(state)."""
    bits = np.array([(int(mask[a >> 5]) >> (a & 31)) & 1 for a in range(ACTION_SIZE)], dtype=np.int64)
    return packed.actions_to_mask(np.nonzero(transform_action_rows(bits, g, n_piles))[0])


def n_piles_of(words):
    return (np.asarray(words, dtype=np.uint32).reshape(-1, 32)[:, 22] >> 16) & 0xFF


def leaf_frame(words, search_key, mode):
    """The frame of a leaf row in a search with symmetry mode ``mode`` (hz_tree_set_symmetry)."""
    G = GROUP_SIZE[mode_code(mode)]
    if G == 1:
        return 0
    z = packed.rand((int(search_key) & packed.M64) ^ SYMMETRY_SALT, packed.canon_hash(words, packed.KEY_EXACT))
    return ((z >> 32) * G) >> 32


# ---- tensors (hz_sym_states / hz_sym_actions) ---------------------------------------------------
def _sym_tensor(sym, n, device):
    sym = torch.as_tensor(sym, device=device)
    if sym.dim() == 0:
        sym = sym.expand(n)
    if sym.shape != (n,):
        raise ValueError(f"sym must have one element per row ({n}), got {tuple(sym.shape)}")
    if sym.dtype != torch.int16 or not sym.is_contiguous():
        if bool(((sym < 0) | (sym >= ORDER)).any()):
            raise ValueError("group elements are 0..479")
        sym = sym.to(torch.int16).contiguous()
    return sym


def transform_states(states, sym, out=None):
    """T_{sym[i]}(states[i]) on the device: states int32[n, 32] CUDA, sym int[n] (or one int).  out may be states."""
    n = _check_states(states)
    sym = _sym_tensor(sym, n, states.device)
    out = torch.empty_like(states) if out is None else out
    if out.shape != states.shape or out.dtype != torch.int32 or not out.is_contiguous():
        raise TypeError("out must be a contiguous int32[n, 32] tensor")
    with torch.cuda.device(states.device):
        _lib.check(_lib.load().hz_sym_states(_ptr(states), n, _ptr(sym), _ptr(out), _stream(states)), "hz_sym_states")
    return out


_DTYPES = {torch.float32: 0, torch.int16: 2, torch.int32: 3}     # HZ_DTYPE_F32 / I16 / I32


def transform_actions(x, sym, states, inverse=False):
    """Rows x [n, 143] (float32, int16 or int32, CUDA) -> x' with x'[i][sigma(a)] = x[i][a], sigma = sigma_{sym[i]}
    (inverse=True: sigma^-1).  states: the rows' records (either frame; only n_piles is read)."""
    n = _check_states(states)
    if x.dtype not in _DTYPES or x.shape != (n, ACTION_SIZE) or not x.is_contiguous() or x.device != states.device:
        raise TypeError("x must be a contiguous [n, 143] float32 / int16 / int32 tensor on the states' device")
    sym = _sym_tensor(sym, n, states.device)
    out = torch.empty_like(x)
    with torch.cuda.device(states.device):
        _lib.check(
            _lib.load().hz_sym_actions(_ptr(x), n, _DTYPES[x.dtype], _ptr(sym), _ptr(states), 1 if inverse else 0, _ptr(out),
                                       _stream(states)),
            "hz_sym_actions",
        )
    return out


def random_elements(n, mode, device="cuda", generator=None):
    """n uniform elements of the group of ``mode`` ("board": 0..3, "full": 0..479) as int16, from ``generator``."""
    G = GROUP_SIZE[mode_code(mode)]
    return torch.randint(0, G, (n,), device=device, generator=generator, dtype=torch.int64).to(torch.int16)
