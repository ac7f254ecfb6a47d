"""Measurements of the rollout evaluator (hz_tree_rollout_eval) on one GPU.

    python profiles/rollout_bench.py [--trees 4096] [--sims 100] [--rollouts 1,8,32,64] [--games 8192] [--slots 4096]
                                     [--strength-games 64] [--quick]

1. Search steps: --trees trees x --sims simulations from positions 8 actions into the game, per R in --rollouts.  One
   simulation step is three captured graphs (select / rollout eval / expand-backup), replayed back to back with CUDA
   events between them; reported: us per step and part, simulations/s, rollout actions/s (from total_steps).  The fused
   playout of 262,144 fresh games (hz_playout_keys, bench.py's engine leg) is timed in the same process for comparison.
2. Whole rollout-driven self-play games (R = 32, --sims simulations per move): games/s.
3. Strength: rollout MCTS (--sims simulations) against the 1-ply greedy agent and against the random-init default
   network (the same simulation count), --strength-games games per setting.  These are figures, not assertions.
--quick shrinks every size (a smoke run of the script itself).
"""

import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from harmonies_alphazero_b200 import arena  # noqa: E402
from harmonies_alphazero_b200 import batched as hb  # noqa: E402
from harmonies_alphazero_b200 import net as hznet  # noqa: E402
from harmonies_alphazero_b200 import selfplay as sp  # noqa: E402
from harmonies_alphazero_b200.tree import BatchedMCTS  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--trees", type=int, default=4096)
ap.add_argument("--sims", type=int, default=100)
ap.add_argument("--rollouts", default="1,8,32,64")
ap.add_argument("--games", type=int, default=8192)
ap.add_argument("--slots", type=int, default=4096)
ap.add_argument("--strength-games", type=int, default=64)
ap.add_argument("--searches", type=int, default=3, help="timed searches per R (after one untimed)")
ap.add_argument("--quick", action="store_true")
a = ap.parse_args()
if a.quick:
    a.trees, a.sims, a.games, a.slots, a.strength_games, a.searches = 64, 8, 16, 16, 4, 1

if not torch.cuda.is_available():
    sys.exit("rollout_bench.py measures the GPU and found none")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
dev = torch.device("cuda", 0)
torch.manual_seed(0)
out = {"trees": a.trees, "sims": a.sims}


# ---- the fused playout of fresh games, for comparison ------------------------------------------------------------
def playout_rate(n=262144, reps=10):
    keys = torch.arange(n, dtype=torch.int64, device=dev)
    res = torch.empty((n, 3), dtype=torch.int32, device=dev)
    tot = torch.zeros(1, dtype=torch.int64, device=dev)
    for _ in range(3):
        hb.playout_keys(keys, results=res, total=tot)
    torch.cuda.synchronize()
    tot.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        hb.playout_keys(keys, results=res, total=tot)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    return {"games": n, "us_per_launch": us, "actions_per_s": int(tot.item()) / reps / (us * 1e-6)}


out["k_playout_fresh_games"] = playout_rate(4096 if a.quick else 262144)
print("k_playout:", json.dumps(out["k_playout_fresh_games"]), flush=True)


# ---- search steps ---------------------------------------------------------------------------------------------------
def search_steps(R):
    n, sims = a.trees, a.sims
    roots = hb.init_states(n, device=dev, seed=404)
    hb.playout(roots, max_steps=8)
    t = BatchedMCTS(n, sims, device=dev, key_mode=hb.KEY_REFERENCE)
    policy = torch.zeros((n, 143), dtype=torch.float32, device=dev)
    value = torch.zeros(n, dtype=torch.float32, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    parts = [lambda: t.select(2.0), lambda: t.rollout_eval(policy, value, R, total),
             lambda: t.expand_backup(policy, value, is_logits=False)]
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        t.reset(roots)
        for _ in range(3):
            for f in parts:
                f()
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize()
    graphs = []
    for f in parts:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            f()
        graphs.append(g)
    acc = [0.0, 0.0, 0.0]
    steps_timed = 0
    actions = 0
    for rep in range(a.searches + 1):
        t.reset(roots)
        torch.cuda.synchronize()
        total.zero_()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(sims)]
        torch.cuda._sleep(2_000_000)          # the device waits while the host enqueues: device time, not launch latency
        for k in range(sims):
            ev[k][0].record()
            for j, g in enumerate(graphs):
                g.replay()
                ev[k][j + 1].record()
        torch.cuda.synchronize()
        t.check_status()
        if rep == 0:
            continue                          # warm-up search
        for k in range(sims):
            for j in range(3):
                acc[j] += ev[k][j].elapsed_time(ev[k][j + 1]) * 1e3
        steps_timed += sims
        actions += int(total.item())
    sel, rol, exp = (x / steps_timed for x in acc)
    step = sel + rol + exp
    return {"R": R, "us_per_step": step, "us_select": sel, "us_rollout_eval": rol, "us_expand_backup": exp,
            "sims_per_s": n / (step * 1e-6), "rollout_actions_per_s": actions / (acc[1] * 1e-6),
            "rollout_actions_per_step": actions / steps_timed}


out["search"] = []
for R in [int(x) for x in a.rollouts.split(",")]:
    r = search_steps(R)
    out["search"].append(r)
    print("search:", json.dumps(r), flush=True)


# ---- whole self-play games ------------------------------------------------------------------------------------------
cfg = sp.SelfPlayConfig(n_slots=a.slots, num_simulations=a.sims, seed=9)
drv = sp.BatchedSelfPlay(sp.RolloutEvaluator(32), cfg, device=dev)
drv.play(1)                                   # captures the step graph (kept by the driver)
torch.cuda.synchronize()
t0 = time.perf_counter()
traj = drv.play(a.games)
torch.cuda.synchronize()
secs = time.perf_counter() - t0
out["selfplay"] = {"R": 32, "games": traj.stats["games"], "slots": a.slots, "sims": a.sims, "seconds": secs,
                   "games_per_s": traj.stats["games"] / secs, "sims_per_s": traj.stats["sims_per_s"],
                   "examples": traj.stats["examples"]}
print("selfplay:", json.dumps(out["selfplay"]), flush=True)
del drv, traj

# ---- strength ------------------------------------------------------------------------------------------------------
mcfg = {"num_simulations": a.sims, "cpuct": 2.0, "testing": True}
model = hznet.AlphaZeroNet.from_config(hznet.DEFAULT_MODEL_CONFIG).eval()
default_net = hznet.InferenceNet(model, device=dev, dtype=torch.bfloat16)
out["strength"] = []
for R in (8, 32):
    for name, opp in (("greedy", arena.GREEDY), ("random-init default network", default_net)):
        t0 = time.perf_counter()
        r = arena.play_match(sp.RolloutEvaluator(R), opp, a.strength_games, mcfg, device=dev, seed=1)
        r.update({"rollouts": R, "opponent": name, "seconds": time.perf_counter() - t0})
        out["strength"].append(r)
        print("strength:", json.dumps(r), flush=True)

print(json.dumps(out))
