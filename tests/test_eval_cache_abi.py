"""Host-side checks of the leaf evaluation cache's C entry points (no GPU needed: nothing here touches the device)."""

import ctypes as C

from harmonies_alphazero_b200 import _lib

HZ_OK, HZ_ERR_ARG, HZ_ERR_WORKSPACE = 0, -1, -4


def test_evalcache_bytes_rejects_bad_sizes():
    lib = _lib.load()
    for entries, rows in ((0, 16), (-8, 16), (7, 16), (12, 16), (8, 0), (8, -1), (1 << 32, 16)):
        assert lib.hz_evalcache_bytes(entries, rows) == 0, (entries, rows)
    small, big = lib.hz_evalcache_bytes(8, 16), lib.hz_evalcache_bytes(64, 16)
    assert small > 0 and big > small and small % 256 == 0
    assert big - small >= 56 * 576      # at least the 144-float row of every extra entry


def test_evalcache_create_checks_workspace_and_arguments():
    lib = _lib.load()
    need = lib.hz_evalcache_bytes(64, 32)
    h = C.c_void_p()
    fake = 1 << 20                       # a 256-byte-aligned address: create stores pointers, it never dereferences them
    assert lib.hz_evalcache_create(C.byref(h), fake, need - 1, 64, 32) == HZ_ERR_WORKSPACE
    assert lib.hz_evalcache_create(C.byref(h), fake + 16, need, 64, 32) == HZ_ERR_WORKSPACE
    assert lib.hz_evalcache_create(None, fake, need, 64, 32) == HZ_ERR_ARG
    assert lib.hz_evalcache_create(C.byref(h), None, need, 64, 32) == HZ_ERR_ARG
    assert lib.hz_evalcache_create(C.byref(h), fake, need, 60, 32) == HZ_ERR_ARG
    assert lib.hz_evalcache_create(C.byref(h), fake, need, 64, 32) == HZ_OK and h.value
    assert lib.hz_evalcache_destroy(h) == HZ_OK
    assert lib.hz_evalcache_clear(None, None) == HZ_ERR_ARG
    assert lib.hz_evalcache_stats(None, None, None) == HZ_ERR_ARG
    assert lib.hz_evalcache_fill(None, None, None, None, None, None, None, None) == HZ_ERR_ARG
    assert lib.hz_tree_select_cached(None, None, 2.0, None, None, None, 1, 3, None, None, None, None, None) == HZ_ERR_ARG
