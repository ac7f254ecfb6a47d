"""CPU: the game's symmetry group (symmetry.py, include/harmonies_b200.h "Game symmetries").  The four hex maps are
automorphisms of the neighbour graph and match the generated device tables; the pile permutations form the
documented group; and the C oracle's rules are invariant / equivariant under every element: scores, outcomes, legal
masks, state tensors and move application."""

import re

import numpy as np
import pytest

from tests.conftest import load_golden
from harmonies_alphazero_b200 import constants as K
from harmonies_alphazero_b200 import gen_tables
from harmonies_alphazero_b200 import packed as pk
from harmonies_alphazero_b200 import symmetry as sy


def test_hex_maps_are_automorphisms_and_form_a_klein_group():
    nb = [[(K.NEIGHBOR_MASKS[i] >> j) & 1 for j in range(23)] for i in range(23)]
    maps = sy.HEX_MAPS
    for b in range(4):
        t = maps[b]
        assert sorted(t) == list(range(23))
        for i in range(23):
            for j in range(23):
                assert nb[i][j] == nb[t[i]][t[j]], (b, i, j)
        assert (sy.HEX_INV[b][t] == np.arange(23)).all()
        for c in range(4):
            assert (maps[b][maps[c]] == maps[b ^ c]).all()                 # closed, composition = xor of the indices
    assert (maps[0] == np.arange(23)).all() and (maps[3] == 22 - np.arange(23)).all()
    assert len({tuple(m) for m in maps}) == 4
    # no other automorphism of the neighbour graph exists (the degree sequence pins hexes down enough to search)
    deg = [bin(m).count("1") for m in K.NEIGHBOR_MASKS]

    def extend(p):
        i = len(p)
        if i == 23:
            yield list(p)
            return
        for j in range(23):
            if j in p or deg[j] != deg[i]:
                continue
            if all(nb[i][k] == nb[j][p[k]] for k in range(i)):
                yield from extend(p + [j])

    assert sorted(tuple(m) for m in extend([])) == sorted(tuple(int(x) for x in m) for m in maps)


def test_tables_match_the_generated_device_file():
    src = open(gen_tables.PATH).read()

    def arr(name):
        m = re.search(name + r"(\[\d+\])+\s*=\s*\{(.*?)\};", src, flags=re.S)
        return [int(x, 0) for x in re.findall(r"0x[0-9A-Fa-f]+|\d+", m.group(2))]

    assert arr("SYM_HEX_G") == [int(x) for x in sy.HEX_MAPS.reshape(-1)]
    assert arr("SYM_HEX_INV_G") == [int(x) for x in sy.HEX_INV.reshape(-1)]
    fwd, inv = arr("SYM_PILE_PERM_G"), arr("SYM_PILE_INV_G")
    for m in range(6):
        for c, p in enumerate(sy.PILE_PERMS[m]):
            e = gen_tables.PILE_PERM_OFFSETS[m] + c
            assert [(fwd[e] >> (3 * i)) & 7 for i in range(m)] == list(p)
            assert [p[(inv[e] >> (3 * i)) & 7] for i in range(m)] == list(range(m))
    assert open(gen_tables.PATH).read() == gen_tables.render()


def test_pile_group_laws():
    assert len({tuple(sy.action_perm(g, 5)) for g in range(480)}) == 480
    rng = np.random.default_rng(1)
    for m in range(6):
        fact = len(sy.PILE_PERMS[m])
        assert 120 % fact == 0
        counts = np.bincount([c % fact for c in range(120)], minlength=fact)
        assert (counts == 120 // fact).all()                               # a uniform g gives a uniform permutation
        ident = sy.action_perm(0, m)
        assert (ident == np.arange(143)).all()
        for _ in range(60):
            g, h = (int(x) for x in rng.integers(0, 480, 2))
            sg, sh = sy.action_perm(g, m), sy.action_perm(h, m)
            k = sy.compose(g, h, m)
            assert (sy.action_perm(k, m) == sg[sh]).all()                  # sigma_{g o h} = sigma_g o sigma_h
            gi = sy.inverse(g, m)
            assert (sy.action_perm(gi, m)[sg] == np.arange(143)).all()
            assert sorted(sg) == list(range(143))


def _playout_states(oracle, n_games=24, seed=5):
    """every state of oracle random playouts, from the first move to the end"""
    st = oracle.init_states(n_games, seed=seed)
    out = [st.copy()]
    for _ in range(170):
        a = oracle.random_actions(st)
        live = a >= 0
        if not live.any():
            break
        st2, status = oracle.apply(st[live], a[live])
        assert (status == 0).all()
        st = st2
        out.append(st.copy())
    return np.concatenate(out)


@pytest.fixture(scope="module")
def corpus(oracle):
    weird = np.unique(load_golden("weird")["states"], axis=0)
    scoring = load_golden("scoring")["states"][::5]
    return np.concatenate([_playout_states(oracle), weird, scoring]).astype(np.uint32)


def _cell_perm(b):
    """cell index (y*7+x) of the 5x7 plane -> cell of its image; cells outside the board stay"""
    cells = np.arange(35)
    for i, (y, x) in enumerate(K.HEX_CELL):
        yy, xx = K.HEX_CELL[sy.HEX_MAPS[b][i]]
        cells[y * 7 + x] = yy * 7 + xx
    return cells


def test_rules_are_invariant(oracle, corpus):
    rng = np.random.default_rng(7)
    g = rng.integers(0, 480, len(corpus))
    g[: 480] = np.arange(480)
    ts = sy.transform_words(corpus, g)
    m = sy.n_piles_of(corpus)
    assert (sy.n_piles_of(ts) == m).all()
    sc, terms = oracle.score(corpus)
    tsc, tterms = oracle.score(ts)
    assert np.array_equal(sc, tsc) and np.array_equal(terms, tterms)
    assert all(np.array_equal(x, y) for x, y in zip(oracle.outcome(corpus), oracle.outcome(ts)))
    lm, tlm = oracle.legal_mask(corpus), oracle.legal_mask(ts)
    for i in range(len(corpus)):
        assert np.array_equal(tlm[i], sy.transform_mask_words(lm[i], g[i], m[i])), i
    b, gl = oracle.encode(corpus)
    tb, tgl = oracle.encode(ts)
    for i in range(len(corpus)):
        cp = _cell_perm(g[i] & 3)
        want = np.empty_like(b[i].reshape(38, 35))
        want[:, cp] = b[i].reshape(38, 35)
        assert np.array_equal(tb[i].reshape(38, 35), want), i
        wg = gl[i].copy()
        for j, d in enumerate(sy.pile_perm(g[i], m[i])):
            wg[6 * d: 6 * d + 6] = gl[i][6 * j: 6 * j + 6]
        assert np.array_equal(tgl[i], wg), i
    # transforms are undone by the inverse element and compose like the group
    back = np.stack([sy.transform_words(ts[i], sy.inverse(g[i], m[i])) for i in range(0, len(ts), 7)])
    assert np.array_equal(back, corpus[::7])


def test_apply_is_equivariant(oracle, corpus):
    rng = np.random.default_rng(11)
    lm = oracle.legal_mask(corpus)
    src, act, gs = [], [], []
    for i in range(len(corpus)):
        acts = pk.mask_to_actions(lm[i])
        if not acts:
            continue
        for a in rng.choice(acts, size=min(2, len(acts)), replace=False):
            src.append(i); act.append(int(a)); gs.append(int(rng.integers(0, 480)))
    src, act, gs = np.array(src), np.array(act), np.array(gs)
    s = corpus[src]
    m = sy.n_piles_of(s)
    after, st = oracle.apply(s, act)
    assert (st == 0).all()
    for board_only in (True, False):
        g = gs & 3 if board_only else gs
        ta = np.array([sy.action_perm(g[k], m[k])[act[k]] for k in range(len(act))])
        got, st2 = oracle.apply(sy.transform_words(s, g), ta)
        assert (st2 == 0).all()
        want = sy.transform_words(after, g)
        if board_only:
            assert np.array_equal(got, want)
            continue
        rest = [w for w in range(32) if w not in (18, 19)]
        assert np.array_equal(got[:, rest] & np.where(np.arange(32)[rest] == 20, 0xFFFF0000, 0xFFFFFFFF).astype(np.uint32),
                              want[:, rest] & np.where(np.arange(32)[rest] == 20, 0xFFFF0000, 0xFFFFFFFF).astype(np.uint32))
        assert (sy.n_piles_of(got) == sy.n_piles_of(want)).all()
        for k in range(len(act)):
            piles = lambda w: sorted(pk.unpack_fields(w)["available_piles"])   # noqa: E731
            assert piles(got[k]) == piles(want[k]), k
        assert (got != want).any()                                         # the pile list really does depend on the state


def test_leaf_frame_rule():
    w = load_golden("engine")["before"][:50]
    assert all(sy.leaf_frame(x, 5, None) == 0 for x in w)
    fr = [sy.leaf_frame(x, 12345, "full") for x in w]
    assert all(0 <= f < 480 for f in fr) and len(set(fr)) > 20
    z = pk.rand(12345 ^ sy.SYMMETRY_SALT, pk.canon_hash(w[0], pk.KEY_EXACT))
    assert fr[0] == ((z >> 32) * 480) >> 32
    assert sy.leaf_frame(w[0], 12345, "board") == ((z >> 32) * 4) >> 32
    # the frame reads the canonical words only: the rng key and counters do not move it
    w2 = w[0].copy()
    w2[24:28] = [1, 2, 3, 4]
    assert sy.leaf_frame(w2, 12345, "full") == fr[0]
    with pytest.raises(ValueError):
        sy.mode_code("rotate")
