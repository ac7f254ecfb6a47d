"""Host-side checks of the Gumbel search's C entry points (no GPU needed: the rejections happen before any device call)."""

import ctypes as C

from harmonies_alphazero_b200 import _lib

HZ_OK, HZ_ERR_ARG, HZ_ERR_WORKSPACE = 0, -1, -4
FAKE = 1 << 20          # a 256-byte-aligned address: the calls below refuse before they touch it


def _tree(lib, n_trees=8, max_sims=32, leaves=1):
    h = C.c_void_p()
    need = lib.hz_tree_workspace_bytes(n_trees, max_sims, 0, leaves)
    assert lib.hz_tree_create(C.byref(h), FAKE, need, n_trees, max_sims, 0, 1, leaves) == HZ_OK
    return h


def test_gumbel_bytes_validates_sizes():
    lib = _lib.load()
    t = _tree(lib)
    assert lib.hz_tree_gumbel_bytes(None, 16, 32) == 0
    for m, n in ((0, 32), (65, 32), (-1, 32), (16, 0), (16, 33), (16, -5)):
        assert lib.hz_tree_gumbel_bytes(t, m, n) == 0, (m, n)
    small, big = lib.hz_tree_gumbel_bytes(t, 1, 1), lib.hz_tree_gumbel_bytes(t, 64, 32)
    assert small > 0 and big > small and small % 256 == 0 and big % 256 == 0
    assert small >= 8 * (1 + 69 * 32) * 4              # one fp32 node value per node slot of every tree
    assert lib.hz_tree_destroy(t) == HZ_OK


def test_set_gumbel_rejects_bad_arguments():
    lib = _lib.load()
    t = _tree(lib)
    need = lib.hz_tree_gumbel_bytes(t, 16, 32)
    assert lib.hz_tree_set_gumbel(None, FAKE, need, 16, 32, 50.0, 0.1, 1.0, None) == HZ_ERR_ARG
    assert lib.hz_tree_set_gumbel(t, FAKE, need, 0, 32, 50.0, 0.1, 1.0, None) == HZ_ERR_ARG
    assert lib.hz_tree_set_gumbel(t, FAKE, need, 65, 32, 50.0, 0.1, 1.0, None) == HZ_ERR_ARG
    assert lib.hz_tree_set_gumbel(t, FAKE, need, 16, 0, 50.0, 0.1, 1.0, None) == HZ_ERR_ARG
    assert lib.hz_tree_set_gumbel(t, FAKE, need, 16, 33, 50.0, 0.1, 1.0, None) == HZ_ERR_ARG      # num_sims > max_sims
    assert lib.hz_tree_set_gumbel(t, FAKE, need, 16, 32, float("nan"), 0.1, 1.0, None) == HZ_ERR_ARG
    assert lib.hz_tree_set_gumbel(t, FAKE, need, 16, 32, 50.0, 0.1, float("inf"), None) == HZ_ERR_ARG
    assert lib.hz_tree_set_gumbel(t, FAKE, need - 1, 16, 32, 50.0, 0.1, 1.0, None) == HZ_ERR_WORKSPACE
    assert lib.hz_tree_set_gumbel(t, FAKE + 16, need, 16, 32, 50.0, 0.1, 1.0, None) == HZ_ERR_WORKSPACE
    # off (NULL buffer) is always accepted, and with the mode off the root call refuses
    assert lib.hz_tree_set_gumbel(t, None, 0, 0, 0, 0.0, 0.0, 0.0, None) == HZ_OK
    assert lib.hz_tree_gumbel_root(t, FAKE, FAKE, None, None) == HZ_ERR_ARG
    assert lib.hz_tree_gumbel_root(None, FAKE, FAKE, None, None) == HZ_ERR_ARG
    assert lib.hz_tree_destroy(t) == HZ_OK


def test_set_gumbel_rejects_virtual_loss_trees():
    lib = _lib.load()
    t = _tree(lib, leaves=4)
    need = lib.hz_tree_gumbel_bytes(t, 16, 32)
    assert need > 0
    assert lib.hz_tree_set_gumbel(t, FAKE, need, 16, 32, 50.0, 0.1, 1.0, None) == HZ_ERR_ARG
    assert lib.hz_tree_destroy(t) == HZ_OK
