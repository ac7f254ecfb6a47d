"""Gumbel search against PUCT on one B200: the split of a simulation step and the time of whole searches.

4,096 trees, the default network in bf16 on the hand-written tower, eager launches, roots spread over the game.  The
two modes alternate for --rounds rounds; every phase is timed with CUDA events around its launches (select, network,
expand+backup; gumbel_root once per search).  Whole searches: Gumbel at n = 16, 32 and 100 (m = 16) and PUCT at 100
simulations, wall time of one search of all trees ending in a device synchronise.
Whole games: BatchedSelfPlay.play of --games games on the trees' slots (CUDA graph, live-prefix compaction), PUCT at 100
simulations and Gumbel at n = 16, 32 and 100 with m = 16; games/s and live sims/s.
Arena: Gumbel-n against PUCT-n at n = 8, 16 and 32, both sides RolloutEvaluator(32), --arena-games games, the candidate
(Gumbel) plays player 0 in even games and player 1 in odd ones; win/draw/loss from Gumbel's side.
Usage: python profiles/gumbel_bench.py [--trees 4096] [--rounds 6] [--games 8192] [--arena-games 256] [--json out.json]
"""

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from harmonies_alphazero_b200 import arena  # noqa: E402
from harmonies_alphazero_b200 import batched as hb  # noqa: E402
from harmonies_alphazero_b200 import selfplay as sp  # noqa: E402
from harmonies_alphazero_b200 import net as hznet
from harmonies_alphazero_b200 import tree as tr


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the record says so rather than guessing
        return f"unknown ({e})"


def roots_for(n, seed):
    st = hb.init_states(n, seed=seed)
    q = n // 4
    for i, d in enumerate((0, 20, 45, 70)):
        sl = st[i * q:(i + 1) * q].clone()
        hb.playout(sl, max_steps=d)
        st[i * q:(i + 1) * q] = sl
    return st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--games", type=int, default=8192)
    ap.add_argument("--arena-games", type=int, default=256)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    n = a.trees
    torch.manual_seed(0)
    model = hznet.AlphaZeroNet.from_config(hznet.DEFAULT_MODEL_CONFIG).eval()
    net = hznet.InferenceNet(model, device="cuda", tower="hand")
    board, glob, logits, value = net.leaf_buffers(n)
    roots = roots_for(n, 3)
    trees = {}
    for mode, sims in (("puct", 100), ("gumbel16", 16), ("gumbel32", 32), ("gumbel100", 100)):
        t = tr.BatchedMCTS(n, sims)
        if mode != "puct":
            t.set_gumbel(m=16, num_sims=sims)
        trees[mode] = (t, sims)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def search(mode, split=None):
        t, sims = trees[mode]
        t.reset(roots)
        for _ in range(sims):
            ev[0].record()
            t.select(2.0, board, glob, dtype=torch.bfloat16, tiles=True)
            ev[1].record()
            net.forward_tiles(board, glob, n, out=(logits, value))
            ev[2].record()
            t.expand_backup(logits, value, is_logits=True)
            ev[3].record()
            if split is not None:
                torch.cuda.synchronize()
                split["select"].append(ev[0].elapsed_time(ev[1]) * 1e3)
                split["network"].append(ev[1].elapsed_time(ev[2]) * 1e3)
                split["expand_backup"].append(ev[2].elapsed_time(ev[3]) * 1e3)
        if mode != "puct":
            ev[0].record()
            t.gumbel_root()
            ev[1].record()
            if split is not None:
                torch.cuda.synchronize()
                split["gumbel_root"].append(ev[0].elapsed_time(ev[1]) * 1e3)
        t.check_status()

    for mode in trees:            # warm-up of every shape
        search(mode)
    torch.cuda.synchronize()
    splits = {m: {k: [] for k in ("select", "network", "expand_backup", "gumbel_root")} for m in ("puct", "gumbel100")}
    whole = {m: [] for m in trees}
    for _ in range(a.rounds):
        for mode in ("puct", "gumbel100"):
            search(mode, splits[mode])
        for mode in trees:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            search(mode)
            torch.cuda.synchronize()
            whole[mode].append(time.perf_counter() - t0)
    med = lambda x: statistics.median(x) if x else None   # noqa: E731
    out = {
        "card": card(), "trees": n, "rounds": a.rounds, "network": "default, bf16, hand-written tower", "launches": "eager",
        "step_split_us_median": {m: {k: med(v) for k, v in s.items()} for m, s in splits.items()},
        "step_split_us_min_max": {m: {k: [min(v), max(v)] if v else None for k, v in s.items()} for m, s in splits.items()},
        "search_s_median": {m: med(v) for m, v in whole.items()},
        "search_s_all": whole,
        "sims_per_s": {m: n * trees[m][1] / med(v) for m, v in whole.items()},
    }
    del trees
    games = {}
    for name, search, sims in (("puct100", "puct", 100), ("gumbel16", "gumbel", 16), ("gumbel32", "gumbel", 32),
                               ("gumbel100", "gumbel", 100)):
        cfg = sp.SelfPlayConfig(n_slots=n, num_simulations=sims, search=search, gumbel_m=16, seed=1)
        sp.BatchedSelfPlay(net, cfg).play(min(n, 512))              # capture and warm-up outside the timed call
        st = sp.BatchedSelfPlay(net, cfg).play(a.games).stats
        games[name] = {"games_per_s": st["games"] / st["seconds"], "live_sims_per_s": st["sims_per_s"], "games": st["games"],
                       "seconds": st["seconds"], "examples": st["examples"]}
        print(name, games[name], flush=True)
    out["whole_games"] = games
    fights = {}
    for sims in (8, 16, 32):
        r = arena.play_match(sp.RolloutEvaluator(32), sp.RolloutEvaluator(32), a.arena_games,
                             {"num_simulations": sims, "cpuct": 2.0, "gumbel_m": 16}, seed=7, search=("gumbel", "puct"))
        fights[f"n{sims}"] = {"gumbel_wins": r["candidate_wins"], "draws": r["draws"], "puct_wins": r["best_wins"],
                              "games": r["games"]}
        print("arena", sims, fights[f"n{sims}"], flush=True)
    out["arena_gumbel_vs_puct_rollout32"] = fights
    print(json.dumps(out, indent=1))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
