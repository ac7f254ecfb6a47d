"""hz_playout's record I/O against the C oracle: a warp loads its 32 records with coalesced 16-byte loads and stores them
back through a shared-memory tile, so warps and blocks that are only partly inside the batch, views that start at any
record of a larger buffer, and records that do not move must all come back exactly as the oracle has them, with no
byte written outside the batch."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hb():
    from harmonies_alphazero_b200 import batched

    batched._lib.load()
    return batched


def host(states):
    return states.cpu().numpy().view(np.uint32)


def mixed_records(oracle, n, seed):
    """fresh games, games 1..60 actions in and finished games, in random order"""
    init = oracle.init_states(n, seed=seed)
    rng = np.random.default_rng(seed)
    cut = rng.integers(0, 90, size=n)
    out = init.copy()
    for m in np.unique(cut):
        sel = cut == m
        out[sel] = oracle.playout(init[sel], max_steps=int(m), n_threads=8)[0]
    return out


@pytest.mark.parametrize("n", [1, 31, 33, 63, 65, 65537])
def test_partial_warps_and_blocks(hb, oracle, n):
    init = oracle.init_states(n, seed=70 + n)
    st = hb.states_from_numpy(init)
    steps, total = hb.playout(st)
    ref, rsteps, rtotal = oracle.playout(init, n_threads=8)
    assert np.array_equal(host(st), ref)
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), rsteps)
    assert int(total.item()) == rtotal


@pytest.mark.parametrize("offset,n", [(1, 45), (3, 100), (37, 257), (64, 64)])
def test_offset_view_keeps_sentinels(hb, oracle, offset, n):
    """the batch is a view `offset` records into a buffer whose other records are random sentinel words"""
    init = mixed_records(oracle, n, seed=offset)
    rng = np.random.default_rng(100 + offset)
    buf_host = rng.integers(0, 2**32, size=(offset + n + 70, 32), dtype=np.uint64).astype(np.uint32)
    buf_host[offset:offset + n] = init
    buf = hb.states_from_numpy(buf_host)
    view = buf[offset:offset + n]
    assert view.is_contiguous() and view.data_ptr() % 128 == 0
    steps, total = hb.playout(view)
    ref, rsteps, rtotal = oracle.playout(init, n_threads=8)
    out = host(buf)
    assert np.array_equal(out[offset:offset + n], ref)
    assert np.array_equal(out[:offset], buf_host[:offset])
    assert np.array_equal(out[offset + n:], buf_host[offset + n:])
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), rsteps)
    assert int(total.item()) == rtotal


@pytest.mark.parametrize("n", [33, 4099])
def test_max_steps_zero_returns_records_unchanged(hb, oracle, n):
    init = mixed_records(oracle, n, seed=n)
    assert (init[:, 28:] == 0).all()
    st = hb.states_from_numpy(init)
    steps, total = hb.playout(st, max_steps=0)
    assert np.array_equal(host(st), init)
    assert not steps.cpu().numpy().any() and int(total.item()) == 0
    ref, _, _ = oracle.playout(init, max_steps=0, n_threads=8)
    assert np.array_equal(ref, init)
