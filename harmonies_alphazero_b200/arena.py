"""Batched arena evaluation (SURVEY.md §8 f3): the candidate-vs-best match of
Trainer.evaluate_model / play_one_eval_game (trainer.py:293-431) with all evaluation games
played concurrently on the GPU.

Reference semantics kept: the candidate plays player 0 in even games and player 1 in odd
games (trainer.py:318-324); every move is a fresh search with the network OF THE SIDE TO MOVE
(trainer.py:395-401) under ``mcts_config_eval`` (testing=True: no noise, greedy move,
config.py:67-78); the result is counted from the candidate's perspective and the win rate
excludes draws (trainer.py:338-342).
"""

import torch

from . import batched as hb
from .selfplay import RolloutEvaluator
from .tree import BatchedMCTS


def _search(tree, net, states, sims, cpuct, bufs):
    board, glob, logits, value = bufs
    tree.reset(states)
    if isinstance(net, RolloutEvaluator):
        for _ in range(sims // tree.leaves):
            tree.select(cpuct)
            tree.rollout_eval(logits, value, net.rollouts)
            tree.expand_backup(logits, value, is_logits=False)
        return
    tiles = board.dtype == torch.uint8
    pad40 = not tiles and board.shape[1] == 40
    for _ in range(sims // tree.leaves):
        tree.select(cpuct, board, glob, dtype=net.dtype, channels_last=True, pad40=pad40, tiles=tiles)
        if tiles:
            net.forward_tiles(board, glob, glob.shape[0], out=(logits, value))
        else:
            net(board, glob, out=(logits, value))
        tree.expand_backup(logits, value, is_logits=True)


GREEDY = "greedy"   # pass as either side to play the 1-ply greedy agent of evaluation.py instead of a network


def play_match(candidate_net, best_net, num_games, mcts_config_eval, device="cuda", seed=0, key_mode=hb.KEY_REFERENCE, leaves=1,
               symmetry=None):
    """Returns dict(candidate_wins, best_wins, draws, win_rate, games).  Each side is an
    InferenceNet on ``device``, ``arena.GREEDY`` (run_tournament of evaluation.py:7-65:
    AlphaZero vs the greedy agent, sides alternating by game index) or a
    ``selfplay.RolloutEvaluator`` (a network-free search of the same simulation count).  leaves > 1 switches the
    searches to the virtual-loss mode (K simulations in flight per tree): not the reference's
    visit counts any more, but a 30-game match then fills the network batch K times better.
    symmetry: None, "board" or "full": both sides' networks see every leaf in a random symmetry frame
    (BatchedMCTS.set_symmetry)."""
    dev = torch.device(device)
    sims, cpuct = int(mcts_config_eval["num_simulations"]), float(mcts_config_eval["cpuct"])
    # group 0: candidate is player 0 (even game indices); group 1: candidate is player 1
    sizes = [(num_games + 1) // 2, num_games // 2]
    result = {"candidate_wins": 0, "best_wins": 0, "draws": 0}
    for g, n in enumerate(sizes):
        if n == 0:
            continue
        states = hb.init_states(n, device=dev, seed=seed, first_id=0 if g == 0 else num_games)   # distinct games per group
        if sims % leaves:
            raise ValueError("num_simulations must be a multiple of leaves")
        searchers = [x for x in (candidate_net, best_net) if x is not GREEDY]
        nets = [x for x in searchers if not isinstance(x, RolloutEvaluator)]
        anynet = nets[0] if nets else None
        tree = bufs = None
        if searchers:                                                # greedy vs greedy needs no search arena
            tree = BatchedMCTS(n, sims, device=dev, key_mode=key_mode, leaves=leaves)
            tree.set_symmetry(symmetry)
            rows = n * leaves
            both_tiles = all(x not in nets or getattr(x, "wants_tiles", False) for x in (candidate_net, best_net))
            if anynet is None:                   # rollouts only: priors and values, no leaf encoding
                bufs = (None, None, torch.zeros((rows, 143), dtype=torch.float32, device=dev),
                        torch.zeros(rows, dtype=torch.float32, device=dev))
            elif both_tiles:                     # every network evaluates from the hand-written tower's input image
                bufs = anynet.leaf_buffers(rows)
            else:
                C = 40 if hasattr(anynet, "stem40") else 38
                bufs = (
                    torch.empty((rows, C, 5, 7), dtype=anynet.dtype, device=dev, memory_format=torch.channels_last).zero_(),
                    torch.zeros((rows, 42), dtype=anynet.dtype, device=dev),
                    torch.zeros((rows, 143), dtype=torch.float32, device=dev),
                    torch.zeros(rows, dtype=torch.float32, device=dev),
                )
        for _ in range(200):
            over, oc = hb.outcome(states)
            if bool(over.all()):
                break
            live = ~over.bool()
            # all live games of a group are in lockstep (fresh standard games: every game has
            # taken the same number of actions): same player to move
            movers = (states[live][:, 22] >> 24) & 1
            mover = int(movers[0].item())
            if not bool((movers == mover).all()):
                raise RuntimeError("arena games of one group are out of lockstep (different players to move)")
            net = candidate_net if mover == g else best_net
            if net is GREEDY:                                        # evaluation.py:137-196, one kernel
                actions = hb.greedy_actions(states)
            else:
                _search(tree, net, states, sims, cpuct, bufs)
                actions = tree.choose()                              # first max N: testing=True
            actions = torch.where(live, actions, torch.full_like(actions, -1))
            hb.apply(states, actions)
        if tree is not None:
            tree.check_status()          # status is sticky across resets: covers every search of the match
        over, oc = hb.outcome(states)
        if not bool(over.all()):
            raise RuntimeError("arena game did not finish")
        cand = oc.to(torch.int32) * (1 if g == 0 else -1)            # outcome is from player 0's view
        result["candidate_wins"] += int((cand > 0).sum().item())
        result["best_wins"] += int((cand < 0).sum().item())
        result["draws"] += int((cand == 0).sum().item())
    decided = result["candidate_wins"] + result["best_wins"]
    result["win_rate"] = result["candidate_wins"] / decided if decided else 0.0   # trainer.py:338-342
    result["games"] = num_games
    return result
