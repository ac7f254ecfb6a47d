"""TEST INFRASTRUCTURE — ctypes binding of tests/gumbel_oracle.c (the Gumbel search restated on the C oracle).

The library is compiled on first use into a temporary directory keyed by the sources' contents, so the tree stays
untouched.  The synthetic and callback evaluators are those of oracle/oracle.py.
"""

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "gumbel_oracle.c"), os.path.join(ROOT, "oracle", "hz_oracle.c"),
           os.path.join(ROOT, "include", "harmonies_b200.h")]
DEFAULTS = dict(m=16, c_visit=50.0, c_scale=0.1, scale=1.0)

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for s in SOURCES:
            with open(s, "rb") as f:
                h.update(f.read())
        out = os.path.join(tempfile.gettempdir(), f"hz_gumbel_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.run(["gcc", "-O2", "-fPIC", "-std=c11", "-pthread", "-fno-fast-math", "-ffp-contract=off", "-shared",
                            "-o", tmp, SOURCES[0], "-lm", "-lpthread"], check=True, capture_output=True)
            os.replace(tmp, out)
        _lib = C.CDLL(out)
        _lib.hzo_search_gumbel.restype = C.c_int
    return _lib


def considered_visits(m, n):
    out = np.zeros(n, dtype=np.int32)
    lib().hzo_considered_visits(C.c_int(m), C.c_int(n), orc._p(out))
    return out


def search(root, search_key, sims, gumbel, num_sims=None, eval_fn=None, key_mode=1, tree=False):
    """One Gumbel search (gumbel: dict with m, c_visit, c_scale, scale; num_sims: n of the considered-visit table,
    default sims).  Returns orc.search's dict plus policy [143] fp32, action, root_value and gap (the smallest non-zero
    distance between a decision's winning score and another candidate's, over every decision of the search)."""
    g = dict(DEFAULTS, **gumbel)
    r = np.ascontiguousarray(root, dtype=np.uint32).reshape(32)
    N = np.zeros(143, dtype=np.int32)
    W = np.zeros(143, dtype=np.float64)
    P = np.zeros(143, dtype=np.float32)
    child = np.zeros(143, dtype=np.int32)
    policy = np.zeros(143, dtype=np.float32)
    nn, ne, act, rv, gap = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_float(0), C.c_double(0)
    cb = C.cast(None, orc.EVAL_FN)
    if eval_fn is not None:
        def _cb(wp, pp, vp, user):
            w = np.ctypeslib.as_array(wp, shape=(32,))
            p, v = eval_fn(w)
            np.ctypeslib.as_array(pp, shape=(143,))[:] = np.asarray(p, dtype=np.float32)
            vp[0] = float(v)

        cb = orc.EVAL_FN(_cb)
    dump, arrays = None, {}
    if tree:
        caps = (1 + 69 * sims, 69 * sims + 1)
        for f, (dt, w) in orc._DUMP_TYPES.items():
            cap = caps[0] if f in orc._NODE_FIELDS else caps[1]
            arrays[f] = np.zeros((cap, w) if w else cap, dtype=dt)
        dump = orc._TreeDump(caps[0], caps[1], *(arrays[f].ctypes.data for f, _ in orc._TreeDump._fields_[2:]))
    rc = lib().hzo_search_gumbel(
        orc._p(r), C.c_uint64(int(search_key)), C.c_int(sims), C.c_int(key_mode), C.c_int(int(g["m"])),
        C.c_int(int(num_sims or sims)), C.c_float(g["c_visit"]), C.c_float(g["c_scale"]), C.c_float(g["scale"]), cb, None,
        orc._p(N), orc._p(W), orc._p(P), orc._p(child), C.byref(nn), C.byref(ne), None if dump is None else C.byref(dump),
        orc._p(policy), C.byref(act), C.byref(rv), C.byref(gap),
    )
    out = {"N": N, "W": W, "P": P, "child": child, "n_nodes": nn.value, "n_edges": ne.value, "rc": rc, "policy": policy,
           "action": act.value, "root_value": rv.value, "gap": gap.value}
    if tree:
        out["tree"] = {f: a[: nn.value if f in orc._NODE_FIELDS else ne.value] for f, a in arrays.items()}
    return out
