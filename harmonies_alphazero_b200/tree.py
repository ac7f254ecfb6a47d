"""Batched search trees: Python handle over the hz_tree_* entry points of the C ABI.

One tree per game, all trees advance one simulation per ``select`` / ``expand_backup``
pair; the evaluator (the policy/value network, or the synthetic one for tests) runs in
between on the whole batch of leaves.  Mirrors MCTS.py (Node/Edge/MCTS, move_to_leaf,
expand_leaf, back_fill and the tail of get_best_action_and_pi).
"""

import ctypes as C

import numpy as np
import torch

from . import _lib
from .batched import F32, BF16, NCHW, NHWC, KEY_EXACT, KEY_REFERENCE, _ptr  # noqa: F401


class BatchedMCTS:
    def __init__(self, n_trees, max_sims, device="cuda", key_mode=KEY_REFERENCE, max_nodes=0, leaves=1):
        """leaves = simulations in flight per tree and step: 1 = the reference's sequential search
        (parity mode); K > 1 = virtual-loss mode, the evaluator then sees n_trees*K rows."""
        self.lib = _lib.load()
        self.n, self.max_sims, self.key_mode, self.leaves = int(n_trees), int(max_sims), key_mode, int(leaves)
        self.rows = self.n * self.leaves
        self.device = torch.device(device)
        nbytes = self.lib.hz_tree_workspace_bytes(self.n, self.max_sims, max_nodes, self.leaves)
        if nbytes == 0:
            raise ValueError("bad tree dimensions")
        # caller-owned workspace (a torch allocation is >=512 B aligned)
        self.workspace = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)   # zeroed: counters/status are defined before the first reset
        h = C.c_void_p()
        _lib.check(
            self.lib.hz_tree_create(C.byref(h), self.workspace.data_ptr(), nbytes, self.n, self.max_sims, max_nodes, key_mode, self.leaves),
            "hz_tree_create",
        )
        self.handle = h
        self.workspace_bytes = nbytes

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            self.lib.hz_tree_destroy(h)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def set_active(self, n_active):
        """n_active: int32 device tensor with one element (kept alive by this object) or None.  Only trees
        0..n_active-1 take part in the following reset / select / expand_backup calls; the value may be
        changed between calls (``n_active.fill_(k)``), also between replays of a captured graph."""
        if n_active is not None:
            assert n_active.dtype == torch.int32 and n_active.numel() >= 1 and n_active.device == self.workspace.device
        self._n_active = n_active
        _lib.check(self.lib.hz_tree_set_active(self.handle, _ptr(n_active)), "hz_tree_set_active")

    def set_symmetry(self, mode):
        """Random-frame leaf evaluation (hz_tree_set_symmetry): None / "board" / "full".  With a mode on, the evaluator sees
        every leaf in a frame T_g drawn from the leaf and the search key, and its policy row is read back through sigma_g;
        the tree does not change.  Acts on the calls that follow; a captured CUDA graph keeps the mode of its capture."""
        from .symmetry import mode_code

        _lib.check(self.lib.hz_tree_set_symmetry(self.handle, mode_code(mode)), "hz_tree_set_symmetry")

    def leaf_frames(self):
        """int64[rows]: the frame g of every leaf row of the last ``select`` (0 when it ran with the mode off)."""
        out = torch.empty(self.rows, dtype=torch.int16, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tree_leaf_frames(self.handle, _ptr(out), self._stream()), "hz_tree_leaf_frames")
        return out.to(torch.int64)

    def reset(self, root_states, search_keys=None):
        """New search per tree (no tree reuse, MCTS.py:288-289).  search_keys int64[n] or None
        (derived per (game, move) from the root's own rng key and move counter)."""
        assert root_states.shape == (self.n, 32) and root_states.dtype == torch.int32 and root_states.is_contiguous()
        assert search_keys is None or (search_keys.shape == (self.n,) and search_keys.dtype == torch.int64)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tree_reset(self.handle, _ptr(root_states), _ptr(search_keys), self._stream()), "hz_tree_reset")

    def select(self, cpuct, board=None, glob=None, leaf_states=None, dtype=torch.float32, channels_last=False, pad40=False, tiles=False):
        """move_to_leaf for every tree + encoding of the leaves into (board, glob).
        pad40: board is [n,40,5,7] channels-last (HZ_LAYOUT_NHWC40, two zero channels).
        tiles: board is the uint8 T16K image of the hand-written tower (HZ_LAYOUT_T16K, bf16)."""
        code = {torch.float32: F32, torch.bfloat16: BF16}[dtype]
        layout = 3 if tiles else 2 if pad40 else (NHWC if channels_last else NCHW)
        if tiles:
            assert board.dtype == torch.uint8 and board.numel() >= (self.rows + 15) // 16 * 71680 and glob.shape[0] == self.rows
        elif board is not None:
            assert board.shape[1] == (40 if pad40 else 38) and board.shape[0] == self.rows and glob.shape[0] == self.rows
        with torch.cuda.device(self.device):
            _lib.check(
                self.lib.hz_tree_select(
                    self.handle, float(cpuct), _ptr(leaf_states), _ptr(board), _ptr(glob), code,
                    layout, self._stream(),
                ),
                "hz_tree_select",
            )

    def expand_backup(self, policy, value, is_logits=False, noise=None, eps=0.0):
        assert policy.dtype == torch.float32 and policy.shape == (self.rows, 143) and policy.is_contiguous()
        assert value.dtype == torch.float32 and value.numel() == self.rows and value.is_contiguous()
        if noise is not None:
            assert noise.dtype == torch.float32 and noise.shape == (self.n, 143) and noise.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(
                self.lib.hz_tree_expand_backup(
                    self.handle, _ptr(policy), _ptr(value), 1 if is_logits else 0, _ptr(noise), float(eps), self._stream()
                ),
                "hz_tree_expand_backup",
            )

    def fake_eval(self, policy, value):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tree_fake_eval(self.handle, _ptr(policy), _ptr(value), self._stream()), "hz_tree_fake_eval")

    def rollout_eval(self, policy, value, rollouts, total_steps=None):
        """Network-free leaf evaluation (hz_tree_rollout_eval): ``rollouts`` (a power of two <= 64) random
        playouts per leaf row of the last ``select``; value = mean outcome for the leaf's mover, priors uniform
        over the legal moves (probabilities: pass ``is_logits=False`` to ``expand_backup``).  total_steps: an
        int64 device tensor with one element to which the rollout actions played are added, or None."""
        assert policy.dtype == torch.float32 and policy.shape == (self.rows, 143) and policy.is_contiguous()
        assert value.dtype == torch.float32 and value.numel() == self.rows and value.is_contiguous()
        if total_steps is not None:
            assert total_steps.dtype == torch.int64 and total_steps.numel() >= 1 and total_steps.device == self.workspace.device
        with torch.cuda.device(self.device):
            _lib.check(
                self.lib.hz_tree_rollout_eval(self.handle, int(rollouts), _ptr(policy), _ptr(value), _ptr(total_steps), self._stream()),
                "hz_tree_rollout_eval",
            )

    def root_policy(self):
        visits = torch.empty((self.n, 143), dtype=torch.int32, device=self.device)
        pi = torch.empty((self.n, 143), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tree_root_policy(self.handle, _ptr(visits), _ptr(pi), self._stream()), "hz_tree_root_policy")
        return visits, pi

    def choose(self, u01=None, exploratory=None):
        actions = torch.empty(self.n, dtype=torch.int16, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tree_choose(self.handle, _ptr(u01), _ptr(exploratory), _ptr(actions), self._stream()), "hz_tree_choose")
        return actions

    def stats(self):
        nn = torch.empty(self.n, dtype=torch.int32, device=self.device)
        ne = torch.empty(self.n, dtype=torch.int32, device=self.device)
        st = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tree_stats(self.handle, _ptr(nn), _ptr(ne), _ptr(st), self._stream()), "hz_tree_stats")
        return nn, ne, st

    def root_edges(self):
        N = torch.empty((self.n, 143), dtype=torch.int32, device=self.device)
        W = torch.empty((self.n, 143), dtype=torch.float64, device=self.device)
        P = torch.empty((self.n, 143), dtype=torch.float32, device=self.device)
        child = torch.empty((self.n, 143), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hz_tree_root_edges(self.handle, _ptr(N), _ptr(W), _ptr(P), _ptr(child), self._stream()), "hz_tree_root_edges")
        return N, W, P, child

    def check_status(self):
        """Raise if any tree overflowed an arena (never silently drop a search)."""
        _, _, st = self.stats()
        bad = torch.nonzero(st).flatten()
        if bad.numel():
            raise RuntimeError(f"{bad.numel()} search trees overflowed (first: tree {int(bad[0])}, status {int(st[bad[0]])})")

    def run_synthetic(self, sims, cpuct, noise=None, eps=0.0):
        """``sims`` simulations with the synthetic evaluator (tests, tree-only benchmarks)."""
        policy = torch.empty((self.rows, 143), dtype=torch.float32, device=self.device)
        value = torch.empty(self.rows, dtype=torch.float32, device=self.device)
        assert sims % self.leaves == 0
        for _ in range(sims // self.leaves):
            self.select(cpuct)
            self.fake_eval(policy, value)
            self.expand_backup(policy, value, noise=noise, eps=eps)


def search_keys_tensor(keys, device="cuda"):
    return torch.as_tensor(np.asarray(keys, dtype=np.uint64).view(np.int64)).to(device)
