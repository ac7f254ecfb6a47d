"""TEST INFRASTRUCTURE — ctypes binding of oracle/_build/libhz_oracle.so (hz_oracle.c).

Importable only by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs.
All arrays are numpy, states are uint32[n, 32] in the packed format.
"""

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "libhz_oracle.so")

EVAL_FN = C.CFUNCTYPE(None, C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(C.c_double), C.c_void_p)


def build(force=False):
    src = os.path.join(HERE, "hz_oracle.c")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-C", HERE, "-B" if force else "-s"], check=True, capture_output=True)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        _lib = C.CDLL(LIB_PATH)
        _lib.hzo_playout.restype = C.c_uint64
        _lib.hzo_search.restype = C.c_int
        _lib.hzo_search_vl.restype = C.c_int
        _lib.hzo_choose.restype = C.c_int
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _states(s):
    s = np.ascontiguousarray(s, dtype=np.uint32).reshape(-1, 32)
    return s


def init_states(n, keys=None, seed=0, first_id=0):
    out = np.zeros((n, 32), dtype=np.uint32)
    k = None if keys is None else np.ascontiguousarray(keys, dtype=np.uint64)
    lib().hzo_init_states(_p(out), C.c_int64(n), _p(k), C.c_uint64(seed), C.c_uint64(first_id))
    return out


def legal_mask(states):
    s = _states(states)
    out = np.zeros((len(s), 5), dtype=np.uint32)
    lib().hzo_legal_mask(_p(s), C.c_int64(len(s)), _p(out))
    return out


def apply(states, actions, draws=None):
    """Returns (new_states, status); input is not modified."""
    s = _states(states).copy()
    a = np.ascontiguousarray(actions, dtype=np.int16)
    d = None if draws is None else np.ascontiguousarray(draws, dtype=np.uint16)
    st = np.zeros(len(s), dtype=np.uint8)
    lib().hzo_apply(_p(s), C.c_int64(len(s)), _p(a), _p(d), _p(st))
    return s, st


def score(states):
    s = _states(states)
    sc = np.zeros((len(s), 2), dtype=np.int16)
    tm = np.zeros((len(s), 2, 5), dtype=np.int16)
    lib().hzo_score(_p(s), C.c_int64(len(s)), _p(sc), _p(tm))
    return sc, tm


def encode(states):
    s = _states(states)
    b = np.zeros((len(s), 38, 5, 7), dtype=np.float32)
    g = np.zeros((len(s), 42), dtype=np.float32)
    lib().hzo_encode(_p(s), C.c_int64(len(s)), _p(b), _p(g))
    return b, g


def canon_hash(states, mode=0):
    s = _states(states)
    out = np.zeros(len(s), dtype=np.uint64)
    lib().hzo_canon_hash(_p(s), C.c_int64(len(s)), C.c_int(mode), _p(out))
    return out


def outcome(states):
    s = _states(states)
    over = np.zeros(len(s), dtype=np.uint8)
    oc = np.zeros(len(s), dtype=np.int8)
    lib().hzo_outcome(_p(s), C.c_int64(len(s)), _p(over), _p(oc))
    return over, oc


def random_actions(states):
    s = _states(states)
    out = np.zeros(len(s), dtype=np.int16)
    lib().hzo_random_actions(_p(s), C.c_int64(len(s)), _p(out))
    return out


def greedy_actions(states):
    s = _states(states)
    out = np.zeros(len(s), dtype=np.int16)
    lib().hzo_greedy_actions(_p(s), C.c_int64(len(s)), _p(out))
    return out


def playout(states, max_steps=1000, n_threads=1):
    """Returns (final_states, steps_per_game, total_steps)."""
    s = _states(states).copy()
    steps = np.zeros(len(s), dtype=np.uint32)
    total = lib().hzo_playout(_p(s), C.c_int64(len(s)), C.c_int(max_steps), _p(steps), C.c_int(n_threads))
    return s, steps, int(total)


class _TreeDump(C.Structure):
    _fields_ = [("cap_nodes", C.c_int), ("cap_edges", C.c_int)] + [
        (f, C.c_void_p) for f in ("words", "hash", "first_edge", "n_edges", "player", "child", "N", "action", "mover", "V", "W", "P")
    ]


_DUMP_TYPES = {"words": (np.uint32, 32), "hash": (np.uint64, 0), "first_edge": (np.int32, 0), "n_edges": (np.int32, 0),
               "player": (np.int32, 0), "child": (np.int32, 0), "N": (np.int32, 0), "action": (np.int32, 0),
               "mover": (np.int32, 0), "V": (np.int32, 0), "W": (np.float64, 0), "P": (np.float32, 0)}
_NODE_FIELDS = ("words", "hash", "first_edge", "n_edges", "player")


def search(root, search_key, sims, cpuct, noise=None, eps=0.0, eval_fn=None, key_mode=1, leaves=1, tree=False, vl=None):
    """One reference-semantics search.  eval_fn(words[32]) -> (p[143] float32, v float) or
    None for the synthetic evaluator.  Returns dict(N, W, P, child, n_nodes, n_edges, rc).
    leaves > 1 (or vl=True) runs the virtual-loss schedule (hzo_search_vl, sims // leaves rounds).
    tree=True adds "tree": the whole arena as numpy arrays, nodes in creation order (words [n, 32],
    hash, first_edge, n_edges, player) and edges in append order (child, N, W, P, action, mover, V)."""
    r = np.ascontiguousarray(root, dtype=np.uint32).reshape(32)
    N = np.zeros(143, dtype=np.int32)
    W = np.zeros(143, dtype=np.float64)
    P = np.zeros(143, dtype=np.float32)
    child = np.zeros(143, dtype=np.int32)
    nn, ne = C.c_int32(0), C.c_int32(0)
    nz = None if noise is None else np.ascontiguousarray(noise, dtype=np.float32)
    cb = C.cast(None, EVAL_FN)
    if eval_fn is not None:

        def _cb(wp, pp, vp, user):
            w = np.ctypeslib.as_array(wp, shape=(32,))
            p, v = eval_fn(w)
            np.ctypeslib.as_array(pp, shape=(143,))[:] = np.asarray(p, dtype=np.float32)
            vp[0] = float(v)

        cb = EVAL_FN(_cb)
    dump, arrays = None, {}
    if tree:   # the oracle's arena capacities (hzo_search)
        caps = (1 + 69 * sims, 69 * sims + 1)
        for f, (dt, w) in _DUMP_TYPES.items():
            cap = caps[0] if f in _NODE_FIELDS else caps[1]
            arrays[f] = np.zeros((cap, w) if w else cap, dtype=dt)
        dump = _TreeDump(caps[0], caps[1], *(arrays[f].ctypes.data for f, _ in _TreeDump._fields_[2:]))
    pd = None if dump is None else C.byref(dump)
    if not (leaves > 1 if vl is None else vl):
        assert leaves == 1
        rc = lib().hzo_search(
            _p(r), C.c_uint64(int(search_key)), C.c_int(sims), C.c_double(cpuct), C.c_int(key_mode), _p(nz), C.c_double(eps),
            cb, None, _p(N), _p(W), _p(P), _p(child), C.byref(nn), C.byref(ne), pd,
        )
    else:   # virtual-loss mode: sims must be a multiple of leaves (sims // leaves rounds)
        assert sims % leaves == 0
        rc = lib().hzo_search_vl(
            _p(r), C.c_uint64(int(search_key)), C.c_int(sims // leaves), C.c_int(leaves), C.c_double(cpuct), C.c_int(key_mode),
            _p(nz), C.c_double(eps), cb, None, _p(N), _p(W), _p(P), _p(child), C.byref(nn), C.byref(ne), pd,
        )
    out = {"N": N, "W": W, "P": P, "child": child, "n_nodes": nn.value, "n_edges": ne.value, "rc": rc}
    if tree:
        out["tree"] = {f: a[: nn.value if f in _NODE_FIELDS else ne.value] for f, a in arrays.items()}
    return out


def choose(N, u=0.0, exploratory=False):
    n = np.ascontiguousarray(N, dtype=np.int32)
    return lib().hzo_choose(_p(n), C.c_float(u), C.c_int(1 if exploratory else 0))


def search_batch(roots, keys, sims, cpuct=2.0, n_threads=1):
    r = _states(roots)
    k = np.ascontiguousarray(keys, dtype=np.uint64)
    N = np.zeros((len(r), 143), dtype=np.int32)
    lib().hzo_search_batch(_p(r), _p(k), C.c_int64(len(r)), C.c_int(sims), C.c_double(cpuct), _p(N), C.c_int(n_threads))
    return N
