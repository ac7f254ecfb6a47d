"""The oracle's whole-tree export (oracle.search(..., tree=True)), which the GPU search tests
compare node for node with the device arenas.  CPU only."""

import numpy as np

from tests.conftest import load_golden
from harmonies_alphazero_b200 import packed as pk


def _roots(oracle, n, seed):
    st = oracle.init_states(n, seed=seed)
    for i in range(n):
        st[i], _, _ = oracle.playout(st[i : i + 1], max_steps=(13 * i) % 61)
    return st


def test_dump_root_edges_are_the_search_outputs(oracle):
    g = load_golden("mcts")
    for i in range(0, len(g["sims"]), 7):
        noise = None if g["testing"][i] else g["noise"][i]
        r = oracle.search(g["root"][i], g["skey"][i], int(g["sims"][i]), float(g["cpuct"][i]), noise, float(g["eps"][i]), tree=True)
        t = r["tree"]
        assert len(t["hash"]) == r["n_nodes"] and len(t["child"]) == r["n_edges"]
        assert np.array_equal(t["words"][0], g["root"][i])
        assert t["hash"][0] == oracle.canon_hash(g["root"][i], 1)[0]
        e0, ne = t["first_edge"][0], t["n_edges"][0]
        acts = t["action"][e0 : e0 + ne]
        assert (np.diff(acts) > 0).all()                               # ascending action order
        N, W, P, child = (np.zeros(143, dt) for dt in (np.int32, np.float64, np.float32, np.int32))
        child[:] = -1
        N[acts], W[acts], P[acts], child[acts] = (t[f][e0 : e0 + ne] for f in ("N", "W", "P", "child"))
        assert np.array_equal(N, r["N"]) and np.array_equal(W, r["W"]) and np.array_equal(child, r["child"])
        assert np.array_equal(P.view(np.uint32), r["P"].view(np.uint32))
        assert (t["V"] == 0).all() and (t["mover"][e0 : e0 + ne] == t["player"][0]).all()
        # every node's key is the key of its words
        assert np.array_equal(t["hash"], oracle.canon_hash(t["words"], 1))


def test_sequential_and_one_leaf_virtual_loss_searches_build_the_same_tree(oracle):
    roots = _roots(oracle, 12, 31)
    stair = np.ldexp(np.ones(143, np.float32), -8 * (142 - np.arange(143)))    # normals, subnormals, zeros

    def stair_eval(w):
        h = int(oracle.canon_hash(w, 0)[0])
        return stair, float(np.float32([1.0, -1.0, -0.0, 0.1, 0.0][h % 5]))

    for i, root in enumerate(roots):
        for ev, cpuct in ((None, 2.0), (stair_eval, 3.0), (stair_eval, 0.0)):
            a = oracle.search(root, 1000 + i, 40, cpuct, eval_fn=ev, tree=True)
            b = oracle.search(root, 1000 + i, 40, cpuct, eval_fn=ev, tree=True, vl=True)
            assert (a["n_nodes"], a["n_edges"]) == (b["n_nodes"], b["n_edges"])
            for f in a["tree"]:
                x, y = a["tree"][f], b["tree"][f]
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), (i, f)


def test_dump_matches_the_python_key_of_each_node(oracle):
    """node keys of the dump in the reference key mode are packed.canon_hash of the node's words"""
    r = oracle.search(_roots(oracle, 1, 5)[0], 77, 30, 2.0, tree=True, key_mode=pk.KEY_REFERENCE)
    t = r["tree"]
    for i in range(0, len(t["hash"]), 9):
        assert int(t["hash"][i]) == pk.canon_hash(t["words"][i], pk.KEY_REFERENCE)
