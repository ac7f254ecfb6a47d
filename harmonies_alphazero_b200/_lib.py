"""ctypes binding of libharmonies_b200.so (C ABI: include/harmonies_b200.h).

There is no CPU fallback: if the library is missing or a call fails, this raises.
"""

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# HZ_LIB_PATH selects another build of the same sources (profiles/run_bounds.sh: the -DHZ_DEBUG_BOUNDS library)
LIB_PATH = os.environ.get("HZ_LIB_PATH") or os.path.join(HERE, "libharmonies_b200.so")

# every symbol include/harmonies_b200.h declares: name -> (restype, argtypes)
_vp, _i64, _u64, _i, _f, _d = C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.c_float, C.c_double
SIGNATURES = {
    "hz_abi_version": (_i, []),
    "hz_status_string": (C.c_char_p, [_i]),
    "hz_last_cuda_error": (C.c_char_p, []),
    "hz_launch_count": (_u64, []),
    "hz_init_states": (_i, [_vp, _i64, _vp, _u64, _u64, _vp]),
    "hz_legal_mask": (_i, [_vp, _i64, _vp, _vp]),
    "hz_apply": (_i, [_vp, _i64, _vp, _vp, _vp, _vp]),
    "hz_end_turn": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "hz_replenish_piles": (_i, [_vp, _i64, _vp]),
    "hz_draw_tiles": (_i, [_vp, _i64, _i, _vp, _vp]),
    "hz_score": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "hz_encode": (_i, [_vp, _i64, _vp, _vp, _i, _i, _vp]),
    "hz_canon_hash": (_i, [_vp, _i64, _i, _vp, _vp]),
    "hz_outcome": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "hz_random_actions": (_i, [_vp, _i64, _vp, _vp]),
    "hz_greedy_actions": (_i, [_vp, _i64, _vp, _vp]),
    "hz_playout": (_i, [_vp, _i64, _i, _vp, _vp, _vp]),
    "hz_playout_keys": (_i, [_vp, _i64, _u64, _u64, _i, _vp, _vp, _vp]),
    "hz_sym_states": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "hz_sym_actions": (_i, [_vp, _i64, _i, _vp, _vp, _i, _vp, _vp]),
    "hz_tree_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i]),
    "hz_tree_create": (_i, [C.POINTER(_vp), _vp, C.c_size_t, _i, _i, _i, _i, _i]),
    "hz_tree_destroy": (_i, [_vp]),
    "hz_tree_reset": (_i, [_vp, _vp, _vp, _vp]),
    "hz_tree_set_active": (_i, [_vp, _vp]),
    "hz_tree_set_symmetry": (_i, [_vp, _i]),
    "hz_tree_leaf_frames": (_i, [_vp, _vp, _vp]),
    "hz_tree_select": (_i, [_vp, _f, _vp, _vp, _vp, _i, _i, _vp]),
    "hz_tree_expand_backup": (_i, [_vp, _vp, _vp, _i, _vp, _d, _vp]),
    "hz_tree_gumbel_bytes": (C.c_size_t, [_vp, _i, _i]),
    "hz_tree_set_gumbel": (_i, [_vp, _vp, C.c_size_t, _i, _i, _f, _f, _f, _vp]),
    "hz_tree_gumbel_root": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "hz_tree_fake_eval": (_i, [_vp, _vp, _vp, _vp]),
    "hz_tree_rollout_eval": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "hz_tree_root_policy": (_i, [_vp, _vp, _vp, _vp]),
    "hz_tree_choose": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "hz_tree_stats": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "hz_tree_root_edges": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "hz_evalcache_bytes": (C.c_size_t, [_i64, _i]),
    "hz_evalcache_create": (_i, [C.POINTER(_vp), _vp, C.c_size_t, _i64, _i]),
    "hz_evalcache_destroy": (_i, [_vp]),
    "hz_evalcache_clear": (_i, [_vp, _vp]),
    "hz_evalcache_stats": (_i, [_vp, _vp, _vp]),
    "hz_tree_select_cached": (_i, [_vp, _vp, _f, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "hz_evalcache_fill": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hz_net_heads": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp]),
    "hz_net_heads_fc_active": (_i, [_vp, _vp, _i64, _vp, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp]),
    "hz_tower_tile_bytes": (C.c_size_t, [_i64, _i]),
    "hz_tower_set_max_ctas": (_i, [_i]),
    "hz_tower_set_debug": (_i, [_i]),
    "hz_tower_set_trace": (_i, [_vp]),
    "hz_tower_to_tiles": (_i, [_vp, _vp, _i64, _i, _i, _vp]),
    "hz_tower_from_tiles": (_i, [_vp, _vp, _i64, _vp]),
    "hz_tower_sched_bytes": (C.c_size_t, [_i64, _i]),
    "hz_tower_forward_heads": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hz_tower_conv3x3": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _i64, _i, _vp, _vp]),
}


class HarmoniesLibraryError(RuntimeError):
    pass


_lib = None


def load(path=None):
    """Load the CUDA library (once).  Raises HarmoniesLibraryError if it is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise HarmoniesLibraryError(
            f"{p} not found: build it with `python -m harmonies_alphazero_b200.build` "
            "(there is no CPU fallback)"
        )
    lib = C.CDLL(p)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    if lib.hz_abi_version() != 6:
        raise HarmoniesLibraryError("ABI version mismatch")
    if path is None:
        _lib = lib
    return lib


def check(status, what=""):
    if status != 0:
        lib = load()
        msg = lib.hz_status_string(status).decode()
        if status == -2:
            msg += ": " + lib.hz_last_cuda_error().decode()
        raise HarmoniesLibraryError(f"{what} failed: {msg}")
