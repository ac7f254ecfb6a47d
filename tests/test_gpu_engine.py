"""GPU parity tests of the engine kernels, through the C ABI (ctypes -> libharmonies_b200.so).

Three anchors: (1) the committed golden vectors produced by the Python reference,
(2) the C oracle on seeded inputs at sizes it finishes in seconds, (3) size-independent
properties at BASELINE.json's full sizes.  Everything is integer/byte work: bit-exact.
"""

import numpy as np
import pytest
import torch

from tests.conftest import load_golden
from harmonies_alphazero_b200 import constants as K
from harmonies_alphazero_b200 import packed as pk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hb():
    from harmonies_alphazero_b200 import batched

    batched._lib.load()  # fail loudly if the CUDA library is missing
    return batched


def dev(words):
    from harmonies_alphazero_b200 import batched

    return batched.states_from_numpy(words)


def host(states):
    return states.cpu().numpy().view(np.uint32)


def i16(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int16).copy()).cuda()


# ---- (1) golden vectors from the reference --------------------------------------------------
def test_golden_traces_explicit_draws(hb):
    g = load_golden("engine")
    st = dev(g["before"])
    assert np.array_equal(host(hb.legal_mask(st)), g["legal"])
    status = hb.apply(st, i16(g["action"]), i16(g["draw"]))
    assert (status == 0).all()
    new = host(st)
    assert np.array_equal(new[:, :24], g["after"][:, :24])
    assert np.array_equal(new[:, 27], g["after"][:, 27])
    assert (new[:, 28:] == 0).all()


def test_golden_traces_stream_draws(hb):
    g = load_golden("engine")
    sel = g["game_of"] >= int(g["n_python"])
    st = dev(g["before"][sel])
    assert np.array_equal(hb.random_actions(st).cpu().numpy(), g["action"][sel])
    status = hb.apply(st, i16(g["action"][sel]))
    assert (status == 0).all()
    assert np.array_equal(host(st)[:, :28], g["after"][sel][:, :28])


def test_golden_init_and_playout(hb):
    g = load_golden("engine")
    npy = int(g["n_python"])
    keys = g["keys"][npy:]
    st = hb.init_states(len(keys), keys=keys)
    assert np.array_equal(host(st)[:, :28], g["before"][g["starts"][npy:-1]][:, :28])
    steps, total = hb.playout(st)
    assert np.array_equal(steps.cpu().numpy(), g["lengths"][npy:])
    assert int(total.item()) == int(g["lengths"][npy:].sum())
    f = [pk.unpack_fields(w) for w in host(st)]
    assert [x["final_scores"] for x in f] == g["final_scores"][npy:].tolist()
    assert [x["winner"] for x in f] == g["winner"][npy:].tolist()
    over, oc = hb.outcome(st)
    assert over.all()
    assert oc.cpu().tolist() == [{0: 1, 1: -1, -1: 0}[w] for w in g["winner"][npy:].tolist()]


def test_golden_scoring_and_legal(hb):
    g = load_golden("scoring")
    st = dev(g["states"])
    sc, tm = hb.score(st, with_terms=True)
    assert np.array_equal(tm.cpu().numpy(), g["terms"])
    assert np.array_equal(sc.cpu().numpy(), g["totals"])
    assert np.array_equal(host(hb.legal_mask(st)), g["legal"])


def test_golden_encode_fp32_bit_exact(hb):
    g = load_golden("encode")
    st = dev(g["states"])
    b, gl = hb.encode(st)
    assert np.array_equal(b.cpu().numpy().view(np.uint32), g["board"].view(np.uint32))
    assert np.array_equal(gl.cpu().numpy().view(np.uint32), g["glob"].view(np.uint32))
    # channels-last holds the same logical tensor
    b2, gl2 = hb.encode(st, channels_last=True)
    assert b2.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(b2.contiguous(), b) and torch.equal(gl2, gl)
    # bf16 = round-to-nearest-even of the fp32 values, both layouts
    for cl in (False, True):
        b3, gl3 = hb.encode(st, dtype=torch.bfloat16, channels_last=cl)
        assert torch.equal(b3.contiguous(), b.to(torch.bfloat16)) and torch.equal(gl3, gl.to(torch.bfloat16))


# hz_encode renders whole 16-byte-aligned groups of 2 (fp32) / 4 (bf16) records with vector stores and every other
# record (the ragged tail, or all of them when the board is not aligned) with scalar ones.  The sizes cover fewer
# records than a group, one record past a group and, at 30,001, more groups than the 148*6 blocks x 8 warps of the
# grid-stride loop hold (28,416 bf16 / 14,208 fp32 records), so that it wraps.
ENCODE_SIZES = (1, 2, 3, 4, 5, 7, 9, 37, 4099, 30001)
ENCODE_KINDS = [(d, cl) for d in (torch.float32, torch.bfloat16) for cl in (False, True)]
SENTINEL = -7.0


def _offsets(dtype):
    """output offsets in elements: aligned, one element off, 8 bytes off"""
    return (0, 1, 8 // torch.empty(0, dtype=dtype).element_size())


@pytest.fixture(scope="module")
def encode_pool(hb):
    """32,524 records in a fixed shuffled order: games 0..49 actions deep (every phase, both players), games played
    to the end, the weird goldens and the encode goldens"""
    n, groups = 20000, 50
    st = hb.init_states(n, seed=606)
    per = n // groups
    for d in range(1, groups):
        hb.playout(st[d * per:(d + 1) * per], max_steps=d if d < groups - 1 else 1000)
    words = np.concatenate([host(st), load_golden("weird")["states"], load_golden("encode")["states"]])
    words = words[np.random.default_rng(606).permutation(len(words))]
    meta = words[:, 22] >> 24
    assert set((meta & 1).tolist()) == {0, 1} and set(((meta >> 1) & 7).tolist()) >= {0, 1, 2, 3, 4}
    return words


def _encode_into(hb, st, dtype, cl, off):
    """hz_encode into views at element offset `off` of sentinel-filled buffers; returns (board, glob, bbuf, gbuf)"""
    n = st.shape[0]
    bbuf = torch.full((off + n * 1330 + 64,), SENTINEL, dtype=dtype, device="cuda")
    gbuf = torch.full((off + n * 42 + 64,), SENTINEL, dtype=dtype, device="cuda")
    flat = bbuf[off:off + n * 1330]
    board = flat.view(n, 5, 7, 38).permute(0, 3, 1, 2) if cl else flat.view(n, 38, 5, 7)
    glob = gbuf[off:off + n * 42].view(n, 42)
    hb.encode(st, dtype=dtype, channels_last=cl, board=board, glob=glob)
    return board, glob, bbuf, gbuf


@pytest.mark.parametrize("dtype,cl", ENCODE_KINDS)
def test_encode_every_size_and_alignment_vs_oracle(hb, oracle, encode_pool, dtype, cl):
    """hz_encode == oracle.encode at every size and at outputs aligned, 1 element off and 8 bytes off: fp32 bit for
    bit, bf16 the round-to-nearest-even of the oracle's fp32, channels-last the same logical tensor; no byte outside
    the n records is written"""
    bits = torch.int32 if dtype == torch.float32 else torch.int16
    for n in ENCODE_SIZES:
        words = encode_pool[:n]
        st = dev(words)
        outs = []
        for off in _offsets(dtype):
            board, glob, bbuf, gbuf = _encode_into(hb, st, dtype, cl, off)
            for buf, end in ((bbuf, off + n * 1330), (gbuf, off + n * 42)):
                assert bool((buf[:off] == SENTINEL).all()) and bool((buf[end:] == SENTINEL).all()), (n, off)
            outs.append((board, glob))
        board, glob = outs[0]
        for b, g in outs[1:]:
            assert torch.equal(b.view(bits), board.view(bits)) and torch.equal(g.view(bits), glob.view(bits)), n
        for lo in range(0, n, 4096):
            hi = min(n, lo + 4096)
            ob, og = oracle.encode(words[lo:hi])
            want_b, want_g = torch.from_numpy(ob).to(dtype).view(bits), torch.from_numpy(og).to(dtype).view(bits)
            assert torch.equal(board[lo:hi].contiguous().view(bits).cpu(), want_b), (n, lo)
            assert torch.equal(glob[lo:hi].view(bits).cpu(), want_g), (n, lo)


@pytest.mark.parametrize("dtype,cl", ENCODE_KINDS)
def test_encode_is_one_launch(hb, encode_pool, dtype, cl):
    """hz_encode is one kernel launch for every non-empty batch, whatever its size and the output's alignment"""
    before = hb.launch_count()
    hb.encode(dev(encode_pool[:0]), dtype=dtype, channels_last=cl)
    assert hb.launch_count() == before
    launches = {}
    for n in ENCODE_SIZES:
        st = dev(encode_pool[:n])
        for off in _offsets(dtype):
            before = hb.launch_count()
            _encode_into(hb, st, dtype, cl, off)
            launches[(n, off)] = hb.launch_count() - before
    assert launches == {k: 1 for k in launches}


def test_golden_weird_states(hb):
    """non-standard states the reference accepts through initial_state: ragged piles, leftover
    hands, nearly empty bags (partial piles, multi-pile replenish, bag-empty end), stray flags"""
    g = load_golden("weird")
    st = dev(g["states"])
    assert np.array_equal(host(hb.legal_mask(st)), g["legal"])
    status = hb.apply(st, i16(g["action"]))
    assert np.array_equal(status.cpu().numpy(), g["status"])
    assert np.array_equal(host(st)[:, :28], g["after"][:, :28])
    # the fused playout must agree with the unfused kernels from these states too
    live = g["status"] == 0
    a, b = dev(g["after"][live]), dev(g["after"][live])
    hb.playout(a, max_steps=7)
    for _ in range(7):
        act = hb.random_actions(b)
        hb.apply(b, torch.where(act >= 0, act, torch.zeros_like(act)))
    stuck_ok = host(a)[:, :28] == host(b)[:, :28]
    assert stuck_ok.all()


def test_greedy_agent(hb, oracle):
    """hz_greedy_actions = choose_move_greedy (evaluation.py:137-196): reference goldens, then
    20,000 mid-game positions against the oracle, then whole greedy-vs-greedy games"""
    g = load_golden("greedy")
    assert np.array_equal(hb.greedy_actions(dev(g["states"])).cpu().numpy(), g["action"])
    st = hb.init_states(20000, seed=8)
    for lo, hi, d in [(0, 5000, 3), (5000, 10000, 18), (10000, 15000, 37), (15000, 20000, 55)]:
        sl = st[lo:hi].clone()
        hb.playout(sl, max_steps=d)
        st[lo:hi] = sl
    assert np.array_equal(hb.greedy_actions(st).cpu().numpy(), oracle.greedy_actions(host(st)))
    games = hb.init_states(512, seed=9)
    for _ in range(200):
        a = hb.greedy_actions(games)
        if bool((a < 0).all()):
            break
        hb.apply(games, torch.where(a >= 0, a, torch.zeros_like(a)))
    over, _ = hb.outcome(games)
    assert over.all()
    sc = hb.score(games).cpu().numpy()
    assert sc.mean() > 25          # greedy play scores far above random play (mean ~17)


def test_golden_equivalence_classes(hb):
    g = load_golden("equiv")
    st = dev(g["states"])
    for mode, cls in ((hb.KEY_EXACT, g["cls"]), (hb.KEY_REFERENCE, g["hcls"])):
        h = hb.canon_hash(st, mode).cpu().numpy().view(np.uint64)
        by_cls, by_hash = {}, {}
        for hi, ci in zip(h.tolist(), cls.tolist()):
            assert by_cls.setdefault(ci, hi) == hi
            assert by_hash.setdefault(hi, ci) == ci


# ---- (2) the C oracle on seeded inputs -------------------------------------------------------
def test_apply_error_codes_match_oracle(hb, oracle):
    """every (state, action) pair incl. all illegal ones: same status, state untouched"""
    g = load_golden("engine")
    rng = np.random.default_rng(5)
    idx = rng.choice(len(g["before"]), 300, replace=False)
    term = g["after"][((g["after"][:, 22] >> 25) & 7) == 4][:4]
    base = np.concatenate([g["before"][idx], term])
    states = np.repeat(base, 146, axis=0)
    actions = np.tile(np.arange(-1, 145, dtype=np.int16), len(base))
    want, wst = oracle.apply(states, actions)
    st = dev(states)
    status = hb.apply(st, i16(actions))
    assert np.array_equal(status.cpu().numpy(), wst)
    assert set(np.unique(wst).tolist()) >= {0, 1, 2, 3, 4, 5, 6}
    assert np.array_equal(host(st)[:, :28], want[:, :28])
    bad = wst != 0
    assert np.array_equal(host(st)[bad], states[bad])


def test_bad_explicit_draw(hb, oracle):
    g = load_golden("engine")
    rows = np.nonzero(g["draw"] != 0xFFFF)[0][:50]
    states = g["before"][rows].copy()
    states[:, 21] = 0
    states[:, 22] &= np.uint32(0xFFFF0000)  # empty bag: the recorded pile cannot be drawn
    want, wst = oracle.apply(states, g["action"][rows], g["draw"][rows])
    st = dev(states)
    status = hb.apply(st, i16(g["action"][rows]), i16(g["draw"][rows]))
    assert (wst == 7).all() and np.array_equal(status.cpu().numpy(), wst)
    assert np.array_equal(host(st), states)


def test_random_games_vs_oracle_stepwise(hb, oracle):
    """4096 seeded games, unfused K1+K2 loop against the oracle at every step"""
    n = 4096
    st = hb.init_states(n, seed=77, first_id=1000)
    ref = oracle.init_states(n, seed=77, first_id=1000)
    assert np.array_equal(host(st), ref)
    for step in range(80):
        mask = host(hb.legal_mask(st))
        assert np.array_equal(mask, oracle.legal_mask(ref))
        a = hb.random_actions(st)
        ra = oracle.random_actions(ref)
        assert np.array_equal(a.cpu().numpy(), ra)
        live = ra >= 0
        if not live.any():
            break
        a_dev = torch.where(a >= 0, a, torch.zeros_like(a))
        status = hb.apply(st, a_dev)
        ref2, rst = oracle.apply(ref, np.where(live, ra, 0))
        assert np.array_equal(status.cpu().numpy(), rst)
        ref = ref2
        assert np.array_equal(host(st), ref), step
    over, _ = hb.outcome(st)
    assert over.all()


def test_fused_playout_equals_unfused_and_oracle(hb, oracle):
    n = 20000
    st = hb.init_states(n, seed=123)
    init = host(st).copy()
    steps, total = hb.playout(st)
    ref, rsteps, rtotal = oracle.playout(init, n_threads=8)
    assert np.array_equal(host(st), ref)
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), rsteps)
    assert int(total.item()) == rtotal
    # bounded playout == the same number of unfused steps
    st2 = dev(init[:2048])
    hb.playout(st2, max_steps=13)
    st3 = dev(init[:2048])
    for _ in range(13):
        hb.apply(st3, hb.random_actions(st3))
    assert torch.equal(st2, st3)


def test_fused_playout_from_mixed_mid_game_states(hb, oracle):
    """neighbouring lanes at different depths: every warp holds both players and all four phases, so the fused
    kernel's per-step branch on the player (playout_step<P>) runs diverged; results must still equal the oracle's"""
    n, groups = 6144, 48
    st = hb.init_states(n, seed=4711)
    per = n // groups
    for d in range(groups):
        if d:
            hb.playout(st[d * per:(d + 1) * per], max_steps=d)          # group d is d actions into its game
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(5)).to(st.device)
    mixed = st[perm].contiguous()
    meta = host(mixed)[:, 22] >> 24
    assert len(set((meta[:32] & 1).tolist())) == 2 and len(set(((meta[:32] >> 1) & 7).tolist())) >= 3
    init = host(mixed).copy()
    steps, total = hb.playout(mixed)
    ref, rsteps, rtotal = oracle.playout(init, n_threads=8)
    assert np.array_equal(host(mixed), ref)
    assert np.array_equal(steps.cpu().numpy().astype(np.uint32), rsteps)
    assert int(total.item()) == rtotal


def test_host_buffer_api_equals_device_path(hb):
    """HostPlayout.run (pinned host in/out, chunked over streams) == hz_playout on device"""
    n = 10000
    st = hb.init_states(n, seed=321)
    pin_in = st.cpu().pin_memory()
    pin_out = torch.empty((n, 32), dtype=torch.int32).pin_memory()
    api = hb.HostPlayout(n, chunks=3)
    out = api.run(pin_in, pin_out)
    steps, total = hb.playout(st)
    assert torch.equal(out, st.cpu()) and int(api.total.item()) == int(total.item())
    assert torch.equal(api.steps.cpu(), steps.cpu())
    with pytest.raises(ValueError):
        api.run(st.cpu(), pin_out)          # not pinned
    # key-based call: fresh games from host keys, compact results back
    rng = np.random.default_rng(2)
    keys = rng.integers(-2**63, 2**63 - 1, size=n, dtype=np.int64)
    pin_keys = torch.from_numpy(keys).pin_memory()
    pin_res = torch.empty((n, 3), dtype=torch.int32).pin_memory()
    res = api.run_keys(pin_keys, pin_res).numpy().view(np.uint32)
    ref = hb.init_states(n, keys=keys.view(np.uint64))
    hb.playout(ref)
    w = host(ref)
    assert np.array_equal(res[:, 0], w[:, 22]) and np.array_equal(res[:, 1], w[:, 23]) and np.array_equal(res[:, 2], w[:, 27])
    # keys derived on the device from (seed, first_id): same games as hz_init_states(seed)
    r2, t2 = hb.playout_keys(None, n=n, seed=321, first_id=0, device="cuda", max_steps=1000)
    w2 = host(st)
    assert np.array_equal(r2.cpu().numpy().view(np.uint32), w2[:, [22, 23, 27]]) and int(t2.item()) == int(total.item())
    # the pipelined stream of batches returns what the one-batch call returns, batch by batch
    batches = [torch.from_numpy(rng.integers(-2**63, 2**63 - 1, size=n, dtype=np.int64)).pin_memory() for _ in range(7)]
    outs = [torch.empty((n, 3), dtype=torch.int32).pin_memory() for _ in range(7)]
    before = int(api.total.item())
    api.run_keys_many(batches, outs, depth=3)
    many_steps = int(api.total.item()) - before
    one = torch.empty((n, 3), dtype=torch.int32).pin_memory()
    acc = 0
    for kb, ob in zip(batches, outs):
        api.run_keys(kb, one)
        assert torch.equal(one, ob)
        acc += int(one[:, 2].sum())
    assert acc == many_steps
    with pytest.raises(ValueError):
        api.run_keys_many(batches, outs[:3])
    # the same buffer ring again with NEW contents: the second call captures the pipeline as a CUDA graph,
    # the third replays it; results must follow the new keys every time
    for rep in range(3):
        for kb in batches:
            kb.copy_(torch.from_numpy(rng.integers(-2**63, 2**63 - 1, size=n, dtype=np.int64)))
        api.run_keys_many(batches, outs, depth=3)
        for kb, ob in zip(batches, outs):
            api.run_keys(kb, one)
            assert torch.equal(one, ob), rep
    assert any(g not in (None, False) for g in api._graphs.values())
    # full-record stream
    recs = [hb.init_states(n, seed=500 + k).cpu().pin_memory() for k in range(5)]
    routs = [torch.empty((n, 32), dtype=torch.int32).pin_memory() for _ in range(5)]
    api.run_many(recs, routs, depth=2)
    for k in (0, 3, 4):
        ref = hb.init_states(n, seed=500 + k)
        hb.playout(ref)
        assert torch.equal(routs[k], ref.cpu())
    assert hb.playout_keys(torch.empty(0, dtype=torch.int64, device="cuda"))[0].shape == (0, 3)


def test_score_encode_hash_vs_oracle_on_random_positions(hb, oracle):
    n = 30000
    st = hb.init_states(n, seed=9)
    hb.playout(st, max_steps=1)  # warm
    rng = np.random.default_rng(1)
    # positions at random depths: play d_i steps by masking with max_steps per slice
    for lo, hi, d in [(0, 10000, 17), (10000, 20000, 41), (20000, 30000, 200)]:
        sl = st[lo:hi].clone()
        hb.playout(sl, max_steps=d)
        st[lo:hi] = sl
    words = host(st)
    sc, tm = hb.score(st, with_terms=True)
    osc, otm = oracle.score(words)
    assert np.array_equal(sc.cpu().numpy(), osc) and np.array_equal(tm.cpu().numpy(), otm)
    sub = rng.choice(n, 3000, replace=False)
    b, gl = hb.encode(st[torch.from_numpy(sub).cuda()].contiguous())
    ob, og = oracle.encode(words[sub])
    assert np.array_equal(b.cpu().numpy().view(np.uint32), ob.view(np.uint32))
    assert np.array_equal(gl.cpu().numpy().view(np.uint32), og.view(np.uint32))
    for mode in (0, 1):
        h = hb.canon_hash(st, mode).cpu().numpy().view(np.uint64)
        assert np.array_equal(h, oracle.canon_hash(words, mode))


# ---- (3) full-size properties (BASELINE.json configs[1], configs[2]) -----------------------
def test_full_size_playout_properties(hb):
    """65,536 concurrent games: every game ends, lengths in the structural range, stored
    final scores equal a fresh hz_score of the final boards, winner consistent, the wave is
    deterministic and independent of how games are batched (game id -> key)."""
    n = 65536
    st = hb.init_states(n, seed=2024)
    steps, total = hb.playout(st)
    over, oc = hb.outcome(st)
    assert over.all()
    s = steps.cpu().numpy()
    assert s.min() >= 56 and s.max() <= 160  # 14 turns minimum (21 hexes / 3 tiles), 40 maximum and s.sum() == int(total.item())
    w = host(st)
    stored = np.stack([(w[:, 23] & 0xFFFF).astype(np.int16), (w[:, 23] >> 16).astype(np.int16)], 1)
    assert np.array_equal(stored, hb.score(st).cpu().numpy())
    wc = (w[:, 22] >> 29) & 3
    expect = np.where(stored[:, 0] > stored[:, 1], 1, np.where(stored[:, 1] > stored[:, 0], 2, 3))
    assert np.array_equal(wc, expect)
    assert np.array_equal(oc.cpu().numpy(), np.where(wc == 1, 1, np.where(wc == 2, -1, 0)))
    # tile conservation: bag + piles + both boards = 120, hand empty at the end
    for x in w[:: 4099]:
        f = pk.unpack_fields(x)
        tiles = sum(f["tile_bag"].values()) + sum(len(p) for p in f["available_piles"])
        tiles += sum(len(s_) for b in f["player_boards"] for s_ in b.values())
        assert tiles == 120 and f["tiles_in_hand"] == []
    # sharding invariance: games 30000..30999 alone give the same records
    part = hb.init_states(1000, seed=2024, first_id=30000)
    hb.playout(part)
    assert np.array_equal(host(part), w[30000:31000])


def test_one_million_synthetic_positions(hb, oracle):
    """configs[2]: 1M full boards with <=3-high stacks: legal + score kernels; checked against
    the oracle on a 100k subsample and by symmetry (swapping the boards swaps the scores)."""
    n = 1_000_000
    rng = np.random.default_rng(31337)
    words = np.zeros((n, 32), dtype=np.uint32)
    shifts = np.arange(23, dtype=np.uint32)
    for p in range(2):
        h = rng.choice(np.array([1, 1, 2, 3], dtype=np.uint8), size=(n, 23))
        for lvl in range(3):
            t = rng.integers(1, 7, size=(n, 23), dtype=np.uint8)
            code = np.where(h > lvl, t, 0).astype(np.uint32)
            for b in range(3):
                words[:, p * 9 + lvl * 3 + b] = (((code >> b) & 1) << shifts).sum(axis=1, dtype=np.uint32)
    hand = rng.integers(0, 6, size=(n, 3))
    hc = np.zeros(n, dtype=np.uint32)
    for j in range(3):
        hc += (1 << (2 * hand[:, j])).astype(np.uint32)
    words[:, 20] = hc << 16
    words[:, 21] = 0x05050505
    words[:, 22] = 0x0505 | ((rng.integers(0, 2, n).astype(np.uint32) | (1 << 1)) << 24)
    st = dev(words)
    sc = hb.score(st).cpu().numpy()
    mask = host(hb.legal_mask(st))
    sub = rng.choice(n, 100_000, replace=False)
    osc, _ = oracle.score(words[sub])
    assert np.array_equal(sc[sub], osc)
    assert np.array_equal(mask[sub], oracle.legal_mask(words[sub]))
    swapped = words.copy()
    swapped[:, 0:9], swapped[:, 9:18] = words[:, 9:18], words[:, 0:9]
    sc2 = hb.score(dev(swapped)).cpu().numpy()
    assert np.array_equal(sc2, sc[:, ::-1])
    assert sc.max() < 200 and sc.min() >= 0


def test_scoring_component_stress(hb, oracle):
    """The loop-free scoring paths against the oracle's plain BFS on boards built to hit them:
    water- and field-heavy tops (components of every size, field rings with enclosed holes), a
    block of identical boards with several large water components (more queued components than
    the per-block water queue holds -> in-lane fallback), and height-1 boards of a single type."""
    rng = np.random.default_rng(77)
    n = 60_000
    shifts = np.arange(23, dtype=np.uint32)
    words = np.zeros((n, 32), dtype=np.uint32)
    # tile codes: water 1, plant 2, wood 3, stone 4, building 5, field 6
    mixes = [np.array([.70, .06, .06, .06, .06, .06]), np.array([.06, .06, .06, .06, .06, .70]),
             np.array([.45, .02, .02, .03, .03, .45]), np.array([.88, .02, .02, .03, .03, .02]),
             np.array([.02, .02, .02, .03, .03, .88])]
    for p in range(2):
        mix = rng.integers(0, len(mixes), n)
        top = np.zeros((n, 23), dtype=np.uint32)
        for m, pr in enumerate(mixes):
            sel = mix == m
            top[sel] = rng.choice(np.arange(1, 7, dtype=np.uint32), size=(int(sel.sum()), 23), p=pr / pr.sum())
        h = rng.choice(np.array([0, 1, 1, 1, 2, 3], dtype=np.uint8), size=(n, 23))     # some empty hexes too
        for lvl in range(3):
            below = rng.integers(1, 7, size=(n, 23), dtype=np.uint32)
            code = np.where(h == lvl + 1, top, np.where(h > lvl + 1, below, 0)).astype(np.uint32)
            for b in range(3):
                words[:, p * 9 + lvl * 3 + b] = (((code >> b) & 1) << shifts).sum(axis=1, dtype=np.uint32)
    # rows 20,000..24,095: one board with as many >= 5-hex water components as a search finds, repeated
    best, best_cnt = 0, -1
    for _ in range(4000):
        m = int(rng.integers(0, 1 << 23))
        rem, cnt = m, 0
        while rem:
            f = rem & -rem
            while True:
                nf = f
                for i in range(23):
                    if (f >> i) & 1:
                        nf |= K.NEIGHBOR_MASKS[i]
                nf &= m
                if nf == f:
                    break
                f = nf
            rem &= ~f
            cnt += bin(f).count("1") >= 5
        if cnt > best_cnt:
            best, best_cnt = m, cnt
    assert best_cnt >= 2
    words[20_000:24_096, 0:18] = 0
    words[20_000:24_096, 0] = best          # height-1 water (code 1) on the chosen hexes, both players
    words[20_000:24_096, 9] = best
    # rows 30,000..30,005: single-type full boards
    for k in range(6):
        words[30_000 + k, 0:18] = 0
        for b in range(3):
            if ((k + 1) >> b) & 1:
                words[30_000 + k, b] = words[30_000 + k, 9 + b] = 0x7FFFFF
    words[:, 21] = 0x05050505
    words[:, 22] = 0x0505 | (1 << 25)
    sc, tm = hb.score(dev(words), with_terms=True)
    osc, otm = oracle.score(words)
    assert np.array_equal(tm.cpu().numpy(), otm)
    assert np.array_equal(sc.cpu().numpy(), osc)
    assert otm[:, :, 2].max() >= 10 and otm[:, :, 4].max() >= 15      # several field components / long rivers occur


def test_edge_cases(hb, oracle):
    # empty batch
    e = torch.empty((0, 32), dtype=torch.int32, device="cuda")
    assert hb.legal_mask(e).shape == (0, 5)
    assert hb.score(e).shape == (0, 2)
    # ragged sizes around block boundaries
    for n in (1, 127, 128, 129, 1000):
        st = hb.init_states(n, seed=n)
        hb.playout(st)
        assert hb.outcome(st)[0].all()
    # stuck position: placement phase with an empty hand has no legal move and is not over
    s = pk.pack_fields([{}, {}], {"water": 3}, [], 0, [], "place_tile_2")
    st = dev(s[None])
    assert int(hb.random_actions(st)[0]) == -1 and (host(hb.legal_mask(st)) == 0).all()
    steps, _ = hb.playout(st)
    assert int(steps[0]) == 0 and not hb.outcome(st)[0].any()
    # partial pile: bag with 2 tiles left -> pile of 2; empty bag -> no new pile
    for bag in ({"water": 1, "field": 1}, {}):
        s = pk.pack_fields([{}, {}], bag, [["wood"] * 3] * 4, 1, ["stone"], "place_tile_3")
        st = dev(s[None])
        hb.apply(st, i16(np.array([5 + 23 * 3 + 4], dtype=np.int16)))
        want, wst = oracle.apply(s[None], [5 + 23 * 3 + 4])
        assert wst[0] == 0 and np.array_equal(host(st)[:, :28], want[:, :28])
        f = pk.unpack_fields(host(st)[0])
        assert len(f["available_piles"]) == (5 if bag else 4)
    # wrong dtype / shape is rejected before any launch
    with pytest.raises(TypeError):
        hb.legal_mask(torch.zeros((4, 32), dtype=torch.int64, device="cuda"))
