"""Batched self-play: the B200 replacement for the body of Trainer.execute_self_play_phase /
self_play_worker (trainer.py:62-134, 434-541).

Thousands of games live in one packed state tensor; every game owns one search tree; one
"simulation step" advances ALL trees by one simulation: hz_tree_select (PUCT descent + leaf
encoding) -> network forward on the whole batch of leaves -> hz_tree_expand_backup.  That
triple is captured once in a CUDA graph and replayed ``num_simulations`` times per move.
Finished games are replaced by fresh ones in place (continuous batching), so the network
batch stays full.

Output contract = the reference worker's (trainer.py:531-538): one example per action of
every completed game: (board f32[38,5,7], global f32[42], pi f32[143], z f32[1]) with the
state encoded BEFORE the search of that move, pi = root visit distribution, z = final
outcome from the mover's perspective (0 on a draw).  Examples are kept packed on the device
(128 B state + int16 visit counts) and expanded on demand.
"""

import time
from dataclasses import dataclass, field

import numpy as np
import torch

from . import batched as hb
from .tree import BatchedMCTS


@dataclass
class SelfPlayConfig:
    n_slots: int = 4096            # concurrent games on this GPU
    num_simulations: int = 100     # mcts_config["num_simulations"]
    cpuct: float = 2.0             # mcts_config["cpuct"]
    dirichlet_alpha: float = 0.4
    dirichlet_epsilon: float = 0.25
    turns_until_tau0: int = 15
    testing: bool = False          # True: no root noise, greedy moves (MCTS.py:308,400)
    key_mode: int = hb.KEY_REFERENCE
    seed: int = 0
    first_game_id: int = 0         # global id of this rank's first game (sharding)
    use_cuda_graph: bool = True
    leaves_per_step: int = 1       # K simulations in flight per tree and step; 1 = reference-exact search, >1 = virtual loss
    n_streams: int = 1             # >1: split the slots into groups on separate streams (overlap tree kernels with convs)
    max_nodes: int = 0             # per-tree node arena; 0 = worst case 1 + 69*sims
    max_moves: int = 200           # hard cap per game (structural maximum is 160 actions)
    compact_live: bool = True      # play(): keep the live games in a dense slot prefix and search only those (the game tail costs what it uses)
    eval_symmetry: str = None      # None, "board" or "full": the network sees each leaf in a random symmetry frame (hz_tree_set_symmetry)

    @classmethod
    def from_mcts_config(cls, mcts_config, **kw):
        """Reads the keys MCTS.py reads (SURVEY.md §5): num_simulations, cpuct,
        dirichlet_alpha, dirichlet_epsilon, turns_until_tau0, testing."""
        m = dict(
            num_simulations=int(mcts_config["num_simulations"]),
            cpuct=float(mcts_config["cpuct"]),
            dirichlet_alpha=float(mcts_config.get("dirichlet_alpha", 0.4)),
            dirichlet_epsilon=float(mcts_config.get("dirichlet_epsilon", 0.25)),
            turns_until_tau0=int(mcts_config.get("turns_until_tau0", 15)),
            testing=bool(mcts_config.get("testing", False)),
        )
        m.update(kw)
        return cls(**m)


@dataclass
class Trajectories:
    """Packed examples of completed games, on the device they were produced on."""
    states: torch.Tensor    # int32 [M, 32]  state before the search of that move (trainer.py:473)
    visits: torch.Tensor    # int16 [M, 143] root visit counts (pi = visits / sum)
    z: torch.Tensor         # float32 [M]    outcome from the mover's perspective (trainer.py:523-528)
    game_id: torch.Tensor   # int64 [M]
    move_no: torch.Tensor   # int32 [M]
    stats: dict = field(default_factory=dict)

    def __len__(self):
        return int(self.states.shape[0])

    def pi(self):
        v = self.visits.to(torch.float64)
        return (v / v.sum(dim=1, keepdim=True).clamp_min(1)).to(torch.float32)   # trainer.py:535

    def encode(self, dtype=torch.float32):
        """(board [M,38,5,7], glob [M,42]) via hz_encode — needs the tensors on a CUDA device."""
        return hb.encode(self.states.contiguous(), dtype=dtype)

    def to_reference_examples(self, last=None):
        """list[(board, global, pi, z)] of CPU tensors, exactly what self_play_worker returns
        and ReplayBuffer.extend consumes (trainer.py:127,531-538; buffer.py:55-67).  Every tensor
        owns its storage, like the reference's: buffer.save_buffer pickles the deque, and a VIEW
        into one big batch tensor would drag the whole batch into the pickle once per example.
        ``last`` = only the final ``last`` examples (what a deque(maxlen=last) keeps of an extend)."""
        n = len(self)
        if n == 0:
            return []
        lo = 0 if last is None else max(0, n - int(last))
        sub = self if lo == 0 else Trajectories(self.states[lo:], self.visits[lo:], self.z[lo:], self.game_id[lo:], self.move_no[lo:])
        board, glob = sub.encode()
        fields = [t.cpu().numpy() for t in (board, glob, sub.pi(), sub.z.view(-1, 1))]
        fn = torch.from_numpy
        return [tuple(fn(f[i].copy()) for f in fields) for i in range(n - lo)]

    def transform(self, sym):
        """A copy with every example mapped by a group element (symmetry.py): states T_g(state), visits
        x'[sigma_g(a)] = x[a], z and the ids unchanged.  sym: int or int[M] (0..479)."""
        from .symmetry import transform_actions, transform_states

        if len(self) == 0:
            return Trajectories(self.states.clone(), self.visits.clone(), self.z.clone(), self.game_id.clone(),
                                self.move_no.clone(), dict(self.stats))
        states = self.states.contiguous()
        return Trajectories(transform_states(states, sym), transform_actions(self.visits.contiguous(), sym, states),
                            self.z.clone(), self.game_id.clone(), self.move_no.clone(), dict(self.stats))

    def to(self, device):
        return Trajectories(self.states.to(device), self.visits.to(device), self.z.to(device),
                            self.game_id.to(device), self.move_no.to(device), dict(self.stats))


class SyntheticEvaluator:
    """Stands in for the network where the leaf evaluation has to be an exact, device-independent
    function of the position (parity tests against the reference's own self-play worker,
    tree-only measurements): priors and value come from hz_tree_fake_eval, the same function of
    the leaf's canonical hash as oracle/ref_harness.FakeModelManager.  Pass it as ``net``."""

    dtype = torch.float32
    tree_eval = True

    def __init__(self, device="cuda"):
        self.device = torch.device(device)

    def __call__(self, board, glob, out=None):
        raise RuntimeError("SyntheticEvaluator is evaluated on the tree (hz_tree_fake_eval), not on tensors")


class RolloutEvaluator:
    """Network-free evaluator: every leaf is valued by ``rollouts`` random playouts on the GPU (hz_tree_rollout_eval)
    and its priors are uniform over the legal moves.  Its strength is set by (simulations, rollouts) alone, so it is a
    fixed opponent for arena matches and gives iteration 0 real policy and value targets.  Pass it as ``net`` (self-play)
    or as either side of ``arena.play_match``.  rollouts: a power of two <= 64."""

    dtype = torch.float32

    def __init__(self, rollouts=32, device="cuda"):
        rollouts = int(rollouts)
        if rollouts < 1 or rollouts > 64 or rollouts & (rollouts - 1):
            raise ValueError("rollouts must be a power of two in 1..64")
        self.rollouts = rollouts
        self.device = torch.device(device)

    def __call__(self, board, glob, out=None):
        raise RuntimeError("RolloutEvaluator is evaluated on the tree (hz_tree_rollout_eval), not on tensors")


class _Group:
    """A contiguous range of slots with its own trees, static network buffers, CUDA graph and
    stream.  Two groups on two streams let one group's tree kernels (HBM/latency-bound) run
    under the other group's convolutions (tensor-bound)."""

    def __init__(self, owner, lo, hi):
        cfg, net, dev = owner.cfg, owner.net, owner.device
        self.o, self.lo, self.hi = owner, lo, hi
        n = hi - lo
        K = max(1, int(cfg.leaves_per_step))
        if cfg.num_simulations % K:
            raise ValueError("num_simulations must be a multiple of leaves_per_step")
        self.tree = BatchedMCTS(n, cfg.num_simulations, device=dev, key_mode=cfg.key_mode, max_nodes=cfg.max_nodes, leaves=K)
        self.tree.set_symmetry(cfg.eval_symmetry)     # before any capture: a graph keeps the mode it was captured with
        rows = n * K                  # the network sees K leaves per tree and step
        dt, cl = net.dtype, owner.channels_last
        self.tiles = bool(getattr(net, "wants_tiles", False))   # leaves go straight into the hand-written tower's input image
        if isinstance(net, RolloutEvaluator):                    # the leaves are never encoded
            self.board = self.glob = None
            self.logits = torch.zeros((rows, 143), dtype=torch.float32, device=dev)
            self.value = torch.zeros(rows, dtype=torch.float32, device=dev)
        elif self.tiles:
            self.board, self.glob, self.logits, self.value = net.leaf_buffers(rows)
        else:
            self.board = torch.empty((rows, 40 if owner.pad40 else 38, 5, 7), dtype=dt, device=dev,
                                     memory_format=torch.channels_last if cl else torch.contiguous_format).zero_()
            self.glob = torch.zeros((rows, 42), dtype=dt, device=dev)
            self.logits = torch.zeros((rows, 143), dtype=torch.float32, device=dev)
            self.value = torch.zeros(rows, dtype=torch.float32, device=dev)
        self.noise = None if cfg.testing else torch.ones((n, 143), dtype=torch.float32, device=dev)
        self.alpha = None if cfg.testing else torch.full((n, 143), cfg.dirichlet_alpha, dtype=torch.float32, device=dev)
        self.graph = None
        self.graph_version = 0
        self.stream = torch.cuda.Stream(device=dev) if owner.n_groups > 1 else None
        # [active trees, active leaf rows]: read on the device by the tree kernels and the hand-written network path,
        # so the captured graph follows it (hz_tree_set_active)
        self.n_active = torch.tensor([n, rows], dtype=torch.int32, device=dev)
        self.tree.set_active(self.n_active[0:1])

    def set_active(self, n_trees):
        K = self.tree.leaves
        self.n_active[0:1].fill_(int(n_trees))
        self.n_active[1:2].fill_(int(n_trees) * K)

    def sim_step(self):
        """one simulation for every tree of the group: select -> network (or rollouts) -> expand+backup"""
        o, t = self.o, self.tree
        if isinstance(o.net, RolloutEvaluator):
            t.select(o.cfg.cpuct)
            t.rollout_eval(self.logits, self.value, o.net.rollouts)
            t.expand_backup(self.logits, self.value, is_logits=False, noise=self.noise, eps=o.cfg.dirichlet_epsilon)
            return
        t.select(o.cfg.cpuct, self.board, self.glob, dtype=o.net.dtype, channels_last=o.channels_last, pad40=o.pad40, tiles=self.tiles)
        if getattr(o.net, "tree_eval", False):
            t.fake_eval(self.logits, self.value)       # priors, not logits
        elif self.tiles:
            o.net.forward_tiles(self.board, self.glob, self.glob.shape[0], out=(self.logits, self.value), n_active=self.n_active[1:2], tag=self.lo)
        elif o._net_takes_out:        # InferenceNet writes straight into the static buffers
            o.net(self.board, self.glob, out=(self.logits, self.value))
        else:
            logits, value = o.net(self.board, self.glob)
            self.logits.copy_(logits)
            self.value.copy_(value)
        t.expand_backup(self.logits, self.value, is_logits=not getattr(o.net, "tree_eval", False), noise=self.noise,
                        eps=o.cfg.dirichlet_epsilon)

    def capture(self):
        """Warm up (cuDNN algorithm selection must happen outside capture) and capture one
        simulation step in a CUDA graph."""
        dev = self.o.device
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(3):
                self.sim_step()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.sim_step()
        self.graph = g

    def prepare(self, states):
        self.tree.reset(states[self.lo:self.hi])
        if self.noise is not None:
            # unnormalised Dirichlet: i.i.d. Gamma(alpha); the expand kernel normalises over
            # the legal root moves (MCTS.py:314-316)
            self.noise.copy_(torch._standard_gamma(self.alpha)).clamp_min_(1e-30)


class BatchedSelfPlay:
    def __init__(self, net, cfg: SelfPlayConfig, device="cuda"):
        self.net, self.cfg = net, cfg
        self.device = torch.device(device)
        B = cfg.n_slots
        self.channels_last = net.device.type == "cuda"
        self.pad40 = self.channels_last and hasattr(net, "stem40")   # 40-channel input: no cuDNN padding pre-pass
        try:
            import inspect

            self._net_takes_out = "out" in inspect.signature(net.__call__).parameters
        except (TypeError, ValueError):
            self._net_takes_out = False
        self.n_groups = max(1, min(int(cfg.n_streams), B))
        cuts = [B * g // self.n_groups for g in range(self.n_groups + 1)]
        self.groups = [_Group(self, cuts[g], cuts[g + 1]) for g in range(self.n_groups)]
        self.sims_run = 0

    # single-group conveniences (profiling harnesses, tests)
    @property
    def tree(self):
        return self.groups[0].tree

    @property
    def graph(self):
        return self.groups[0].graph

    def _sim_step(self):
        for g in self.groups:
            g.sim_step()

    def search(self, states):
        """One full search per slot from ``states`` (get_best_action_and_pi up to the root
        statistics, MCTS.py:288-352)."""
        cfg = self.cfg
        main = torch.cuda.current_stream(self.device)
        for g in self.groups:
            g.prepare(states)
            if g.graph is not None and g.graph_version != getattr(self.net, "version", 0):
                g.graph = None                    # the network was reloaded: the captured launches point at the old weights
            if cfg.use_cuda_graph and g.graph is None:
                g.capture()
                g.graph_version = getattr(self.net, "version", 0)
                g.tree.reset(states[g.lo:g.hi])   # the warm-up/capture advanced the trees
        for g in self.groups:
            if g.stream is not None:
                g.stream.wait_stream(main)
        for _ in range(cfg.num_simulations // max(1, int(cfg.leaves_per_step))):
            for g in self.groups:
                if g.stream is None:
                    g.graph.replay() if g.graph is not None else g.sim_step()
                else:
                    with torch.cuda.stream(g.stream):
                        g.graph.replay() if g.graph is not None else g.sim_step()
        for g in self.groups:
            if g.stream is not None:
                main.wait_stream(g.stream)
        self.sims_run += cfg.num_simulations

    def root_policy(self):
        parts = [g.tree.root_policy() for g in self.groups]
        return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])

    def choose(self, u01=None, exploratory=None):
        return torch.cat([
            g.tree.choose(None if u01 is None else u01[g.lo:g.hi].contiguous(),
                          None if exploratory is None else exploratory[g.lo:g.hi].contiguous())
            for g in self.groups])

    def check_status(self):
        for g in self.groups:
            g.tree.check_status()

    # ---- whole games ---------------------------------------------------------------------
    def play(self, num_games, progress=None):
        """Play ``num_games`` complete games (ids first_game_id .. +num_games-1).  Returns
        Trajectories with ``stats`` (sims, seconds, sims_per_s, games, examples)."""
        cfg, dev, B = self.cfg, self.device, self.cfg.n_slots
        started = min(B, num_games)
        states = hb.init_states(B, device=dev, seed=cfg.seed, first_id=cfg.first_game_id)
        game_id = torch.arange(B, device=dev, dtype=torch.int64)        # local ids
        live = game_id < started
        outcome = torch.zeros(num_games, dtype=torch.int8, device=dev)
        finished = torch.zeros(num_games, dtype=torch.bool, device=dev)
        chunks, bad_status = [], torch.zeros((), dtype=torch.uint8, device=dev)
        live_sims = 0
        compact = cfg.compact_live and self.n_groups == 1
        for g in self.groups:
            g.set_active(g.hi - g.lo)             # (a previous call that raised may have left a smaller active prefix)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        step = 0
        searched_slots = 0
        while True:
            over, oc = hb.outcome(states)
            done = over.bool() & live
            n_done = int(done.sum().item())                      # one host sync per move
            if n_done:
                ids = game_id[done]
                outcome[ids] = oc[done]
                finished[ids] = True
                k = min(n_done, num_games - started)
                slots = torch.nonzero(done).flatten()
                if k:
                    fresh = hb.init_states(k, device=dev, seed=cfg.seed, first_id=cfg.first_game_id + started)
                    states[slots[:k]] = fresh
                    game_id[slots[:k]] = torch.arange(started, started + k, device=dev, dtype=torch.int64)
                    started += k
                live[slots[k:]] = False
            n_live = int(live.sum().item())
            if n_live == 0:
                break
            if compact:
                if n_done and n_live < B:
                    # live games first (stable): nothing is keyed by the slot index, the draws and the search
                    # streams depend on the game's own key only
                    order = torch.argsort((~live).to(torch.int8), stable=True)
                    states, game_id, live = states[order].contiguous(), game_id[order], live[order]
                self.groups[0].set_active(n_live)
            searched_slots += n_live if compact else B
            move_no = states[:, 27].clone()
            if int(move_no[live].max().item()) >= cfg.max_moves:
                raise RuntimeError("a game exceeded max_moves without ending")
            snap = states.clone()
            self.search(states)
            visits, _ = self.root_policy()
            expl = None
            u01 = None
            if not cfg.testing and cfg.turns_until_tau0 > 0:
                expl = (move_no < cfg.turns_until_tau0).to(torch.uint8)   # MCTS.py:399-402
                u01 = torch.rand(B, device=dev, dtype=torch.float32)
            actions = self.choose(u01, expl)
            # a root without visits (num_simulations <= leaves_per_step, or a search that only ever
            # reached the unexpanded root) has no move to offer: the reference then plays a random
            # legal move and records the all-zero visit vector (MCTS.py:382-392,425-433 — its uniform
            # fallback is written into an int array and truncates to 0)
            actions = torch.where(actions < 0, hb.random_actions(states), actions)
            actions = torch.where(live, actions, torch.full_like(actions, -1))
            status = hb.apply(states, actions)                   # the real move re-draws independently (trainer.py:502)
            bad_status = torch.maximum(bad_status, torch.where(live, status, torch.zeros_like(status)).max())
            chunks.append((snap, visits.to(torch.int16), game_id.clone(), move_no, live.clone()))
            live_sims += n_live * cfg.num_simulations
            step += 1
            if step % 8 == 0:
                self.check_status()
            if progress:
                progress(step, int(finished.sum().item()), num_games)
        for g in self.groups:
            g.set_active(g.hi - g.lo)
        self.check_status()
        if int(bad_status.item()) != 0:
            raise RuntimeError(f"engine rejected a searched move (status {int(bad_status.item())})")
        torch.cuda.synchronize(dev)
        secs = time.perf_counter() - t0
        if chunks:
            S = torch.cat([c[0] for c in chunks]); V = torch.cat([c[1] for c in chunks])
            G = torch.cat([c[2] for c in chunks]); M = torch.cat([c[3] for c in chunks]); L = torch.cat([c[4] for c in chunks])
            keep = L & finished[G.clamp_max(num_games - 1)]
            S, V, G, M = S[keep], V[keep], G[keep], M[keep]
            mover = ((S[:, 22] >> 24) & 1).to(torch.float32)
            z = outcome[G].to(torch.float32) * (1.0 - 2.0 * mover)   # trainer.py:523-528
        else:
            S = torch.empty((0, 32), dtype=torch.int32, device=dev); V = torch.empty((0, 143), dtype=torch.int16, device=dev)
            G = torch.empty(0, dtype=torch.int64, device=dev); M = torch.empty(0, dtype=torch.int32, device=dev)
            z = torch.empty(0, dtype=torch.float32, device=dev)
        stats = {"sims": live_sims, "seconds": secs, "sims_per_s": live_sims / secs if secs > 0 else 0.0,
                 "games": int(finished.sum().item()), "examples": int(S.shape[0]), "move_steps": step,
                 "searched_slots": searched_slots}
        return Trajectories(S, V, z, G + cfg.first_game_id, M, stats)
