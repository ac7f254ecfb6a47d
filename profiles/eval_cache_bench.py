"""Leaf evaluation cache on/off: whole self-play games (SelfPlayConfig.eval_cache) and a step-level split.

Default network (random init, bf16, hand-written tower), cache-off and cache-on plays alternate in one process and their
trajectories must be identical.  Usage:
    python profiles/eval_cache_bench.py --sims 100 --games 8192 --slots 4096 --reps 3 [--symmetry board] [--split] --out f.json
"""

import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from harmonies_alphazero_b200 import batched as hb  # noqa: E402
from harmonies_alphazero_b200 import net as hnet  # noqa: E402
from harmonies_alphazero_b200 import selfplay as sp  # noqa: E402


def same(a, b):
    oa = torch.argsort(a.game_id * 1000 + a.move_no.to(torch.int64))
    ob = torch.argsort(b.game_id * 1000 + b.move_no.to(torch.int64))
    return all(torch.equal(x[oa], y[ob]) for x, y in ((a.states, b.states), (a.visits, b.visits), (a.z, b.z), (a.game_id, b.game_id)))


def step_split(inf, slots, sims, entries, steps=40):
    """Mean µs of select / tower + heads / fill / expand per step with the cache on (and select / network / expand with
    it off), from CUDA events, on the searches of mid-game positions after a warm first search."""
    res = {}
    states = hb.init_states(slots, seed=3)
    hb.playout(states, max_steps=25)
    for mode in ("off", "on"):
        cfg = sp.SelfPlayConfig(n_slots=slots, num_simulations=sims, use_cuda_graph=False, eval_cache=entries if mode == "on" else 0)
        g = sp.BatchedSelfPlay(inf, cfg).groups[0]
        t, o = g.tree, g.o
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        acc = [0.0] * 4
        n_eval = []
        for search in range(2):                     # search 0 fills the cache; search 1 (next move's root) is timed
            if search == 1:
                acts = t.choose()
                hb.apply(states, torch.where(acts < 0, hb.random_actions(states), acts))
            g.prepare(states)
            for k in range(min(steps, sims)):
                ev[0].record()
                if mode == "on":
                    t.select_cached(g.cache, cfg.cpuct, g.board, g.glob, g.logits, g.value, g.eval_rows, g.n_eval, dtype=inf.dtype, tiles=True)
                    ev[1].record()
                    g._evaluate((g.net_logits, g.net_value), g.n_eval)
                    ev[2].record()
                    g.cache.fill(g.net_logits, g.net_value, g.eval_rows, g.n_eval, g.logits, g.value)
                else:
                    t.select(cfg.cpuct, g.board, g.glob, dtype=inf.dtype, tiles=True)
                    ev[1].record()
                    g._evaluate((g.logits, g.value), g.n_active[1:2])
                    ev[2].record()
                ev[3].record()
                t.expand_backup(g.logits, g.value, is_logits=True, noise=g.noise, eps=cfg.dirichlet_epsilon)
                ev[4].record()
                torch.cuda.synchronize()
                if search == 1:
                    for i in range(4):
                        acc[i] += ev[i].elapsed_time(ev[i + 1]) * 1000.0
                    if mode == "on":
                        n_eval.append(int(g.n_eval.item()))
        n = min(steps, sims)
        res[mode] = dict(zip(("select_us", "network_us", "fill_us", "expand_us"), [a / n for a in acc]))
        if mode == "on":
            res[mode]["mean_n_eval"] = sum(n_eval) / len(n_eval)
    # the network alone at full and at reduced active counts
    rows = slots
    board, glob, lg, vl = inf.leaf_buffers(rows)
    na = torch.zeros(1, dtype=torch.int32, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res["network_by_rows_us"] = {}
    for k in (rows, int(rows * 0.9), int(rows * 0.8), int(rows * 0.7), rows // 2):
        na.fill_(k)
        for _ in range(3):
            inf.forward_tiles(board, glob, rows, out=(lg, vl), n_active=na)
        e0.record()
        for _ in range(20):
            inf.forward_tiles(board, glob, rows, out=(lg, vl), n_active=na)
        e1.record()
        torch.cuda.synchronize()
        res["network_by_rows_us"][k] = e0.elapsed_time(e1) * 1000.0 / 20
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sims", type=int, default=100)
    ap.add_argument("--games", type=int, default=8192)
    ap.add_argument("--slots", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--entries", type=int, default=0, help="0: slots * sims * 2")
    ap.add_argument("--symmetry", default=None)
    ap.add_argument("--split", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.manual_seed(0)
    inf = hnet.InferenceNet(hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval(), device="cuda")
    assert inf.wants_tiles
    entries = a.entries or a.slots * a.sims * 2
    base = dict(n_slots=a.slots, num_simulations=a.sims, seed=1, eval_symmetry=a.symmetry)
    players = {"off": sp.BatchedSelfPlay(inf, sp.SelfPlayConfig(**base)),
               "on": sp.BatchedSelfPlay(inf, sp.SelfPlayConfig(**base, eval_cache=entries))}
    runs, ref = {"off": [], "on": []}, None
    for rep in range(a.reps):
        for mode in ("off", "on"):
            torch.manual_seed(100 + rep)
            t0 = time.perf_counter()
            tr = players[mode].play(a.games)
            secs = time.perf_counter() - t0
            if mode == "off":
                ref = tr
            else:
                assert same(ref, tr), "cache-on trajectories differ from cache-off"
            r = dict(seconds=secs, sims_per_s=tr.stats["sims_per_s"], games_per_s=tr.stats["games"] / tr.stats["seconds"])
            if mode == "on":
                r.update(tr.stats["eval_cache"])
            runs[mode].append(r)
            print(mode, rep, json.dumps(r), flush=True)
    out = dict(sims=a.sims, games=a.games, slots=a.slots, symmetry=a.symmetry, entries=entries, identical=True, runs=runs,
               gpu=torch.cuda.get_device_name(0))
    for mode in ("off", "on"):
        v = sorted(x["sims_per_s"] for x in runs[mode])
        out[f"median_sims_per_s_{mode}"] = v[len(v) // 2]
    out["speedup"] = out["median_sims_per_s_on"] / out["median_sims_per_s_off"]
    if a.split:
        out["step_split"] = step_split(inf, a.slots, a.sims, entries)
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
