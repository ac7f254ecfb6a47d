"""The Gumbel search's semantics on the C oracle (CPU only): the considered-visit table against a port of mctx's
sequential-halving schedule, the root's visits against that schedule, and the root's policy target and played action
against a numpy restatement of include/harmonies_b200.h ("Gumbel search")."""

import math

import numpy as np
import pytest

from oracle import oracle as orc
from tests import gumbel_oracle as go

FLT_MIN = float(np.finfo(np.float32).tiny)
SALT = 0x47554D42454C5F31


def mctx_sequence(m, n):
    """mctx seq_halving.get_sequence_of_considered_visits, verbatim in Python."""
    if m <= 1:
        return tuple(range(n))
    log2max = int(math.ceil(math.log2(m)))
    sequence, visits, num_considered = [], [0] * m, m
    while len(sequence) < n:
        extra = max(1, int(n / (log2max * num_considered)))
        for _ in range(extra):
            sequence.extend(visits[:num_considered])
            for i in range(num_considered):
                visits[i] += 1
        num_considered = max(2, num_considered // 2)
    return tuple(sequence[:n])


def _mix64(z):
    M = (1 << 64) - 1
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
    return z ^ (z >> 31)


def gumbel(key, a, scale):
    k = (key ^ SALT) & ((1 << 64) - 1)
    z = _mix64(k ^ _mix64((a + 0x9E3779B97F4A7C15) & ((1 << 64) - 1)))
    return scale * -math.log(-math.log(((z >> 11) + 0.5) * 2.0 ** -53))


def root_restatement(out, key, g):
    """(policy [143], action) from the oracle's root N, W, P and vhat, by the header's formulas."""
    edges = np.flatnonzero(out["child"] >= 0)
    N, W, P = out["N"][edges].astype(np.int64), out["W"][edges], out["P"][edges].astype(np.float64)
    ns = int(N.sum())
    pi = np.maximum(P / P.sum(), FLT_MIN)
    vis = N > 0
    q = np.where(vis, W / np.maximum(N, 1), 0.0)
    wq = (pi[vis] * q[vis]).sum() / pi[vis].sum() if vis.any() else 0.0
    vmix = (out["root_value"] + ns * wq) / (1 + ns)
    qc = np.where(vis, q, vmix)
    qc = (qc - qc.min()) / max(qc.max() - qc.min(), 1e-8)
    sigma = (np.float64(np.float32(g["c_visit"])) + N.max()) * np.float64(np.float32(g["c_scale"])) * qc
    logit = np.log(np.maximum(P, FLT_MIN))
    z = logit + sigma
    p = np.exp(z - z.max())
    policy = np.zeros(143, dtype=np.float64)
    policy[edges] = p / p.sum()
    gs = np.array([gumbel(key, int(a), float(np.float32(g["scale"]))) for a in edges])
    sc = np.where(N == N.max(), np.maximum(-1e9, gs + (logit - logit.max()) + sigma), -np.inf)
    return policy, int(edges[int(np.argmax(sc))])


def _roots(n, seed, steps=(0, 5, 23, 41)):
    out = []
    for i in range(n):
        s = orc.init_states(1, seed=seed + i)
        s, _, _ = orc.playout(s, max_steps=steps[i % len(steps)])
        out.append(s[0])
    return out


def test_considered_visit_table_is_mctx_schedule():
    for m in range(1, 33):
        for n in range(1, 401):
            assert tuple(go.considered_visits(m, n).tolist()) == mctx_sequence(m, n), (m, n)


@pytest.mark.parametrize("m,sims", [(4, 16), (16, 32), (16, 64), (8, 100), (2, 9)])
def test_root_visits_follow_sequential_halving(m, sims):
    for i, root in enumerate(_roots(6, 100 + m)):
        n_legal = int(sum(bin(int(w)).count("1") for w in orc.legal_mask(root[None])[0]))
        out = go.search(root, 1000 + i, sims, dict(m=m))
        assert out["rc"] == 0
        N = out["N"][out["child"] >= 0]
        if len(N) < n_legal:          # a self-loop move has no edge
            n_legal = len(N)
        k = min(m, n_legal)
        assert int(N.sum()) == sims - 1
        if sims >= m:
            assert int((N > 0).sum()) == k
        # the multiset of root visits is the one the schedule produces: simulation i visits an action with seq[i] visits
        counts = [0] * k
        for v in mctx_sequence(k, sims)[: sims - 1]:
            counts[counts.index(v)] += 1
        assert sorted(N[N > 0].tolist(), reverse=True) == sorted([c for c in counts if c], reverse=True)


@pytest.mark.parametrize("g", [dict(m=16), dict(m=4, scale=0.5), dict(m=16, c_visit=10.0, c_scale=1.0), dict(m=1)])
@pytest.mark.parametrize("sims", [2, 16, 17, 40])
def test_policy_target_and_action_match_restatement(g, sims):
    for i, root in enumerate(_roots(5, 7 * sims)):
        key = 0x1234 + 977 * i
        out = go.search(root, key, sims, g)
        assert out["rc"] == 0
        policy, action = root_restatement(out, key, dict(go.DEFAULTS, **g))
        assert np.abs(out["policy"] - policy).max() <= 1e-6
        assert abs(float(out["policy"].sum()) - 1.0) < 1e-5
        assert out["action"] == action


def test_greedy_m1_plays_argmax_prior():
    for i, root in enumerate(_roots(8, 300)):
        out = go.search(root, 55 + i, 12, dict(m=1, scale=0.0))
        edges = np.flatnonzero(out["child"] >= 0)
        assert out["action"] == int(edges[np.argmax(out["P"][edges])])
        assert out["N"][out["action"]] == 11


def test_zero_visit_root_is_gumbel_top1_of_prior():
    for i, root in enumerate(_roots(8, 400)):
        key = 99 + i
        out = go.search(root, key, 1, dict(m=16))
        edges = np.flatnonzero(out["child"] >= 0)
        assert out["N"].sum() == 0
        logit = np.log(np.maximum(out["P"][edges].astype(np.float64), FLT_MIN))
        g = np.array([gumbel(key, int(a), 1.0) for a in edges])
        assert out["action"] == int(edges[np.argmax(g + logit)])
        pi = np.maximum(out["P"][edges].astype(np.float64), FLT_MIN)
        assert np.abs(out["policy"][edges] - pi / pi.sum()).max() <= 1e-6


def test_unexpanded_and_terminal_roots():
    root = _roots(1, 5)[0]
    out = go.search(root, 1, 0, dict(m=16), num_sims=1)
    assert out["action"] == -1 and not out["policy"].any()
    over, _, _ = orc.playout(orc.init_states(1, seed=3), max_steps=1000)
    out = go.search(over[0], 1, 8, dict(m=16))
    assert out["action"] == -1 and not out["policy"].any() and out["N"].sum() == 0


def _one_move_root():
    for seed in range(200):
        s = orc.init_states(1, seed=seed)
        for _ in range(400):
            if int(orc.outcome(s)[0][0]):
                break
            if sum(bin(int(w)).count("1") for w in orc.legal_mask(s)[0]) == 1:
                return s[0]
            s, _ = orc.apply(s, orc.random_actions(s))
    return None


def test_one_edge_root_plays_it_one_hot():
    root = _one_move_root()
    if root is None:
        pytest.skip("no position with a single legal move in the sampled games")
    out = go.search(root, 7, 8, dict(m=16))
    edges = np.flatnonzero(out["child"] >= 0)
    assert len(edges) == 1
    assert out["action"] == int(edges[0]) and out["policy"][edges[0]] == 1.0 and out["policy"].sum() == 1.0
