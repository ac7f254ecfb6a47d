"""What random-frame leaf evaluation and the bulk symmetry transforms cost.

1. One simulation step of self-play at 4,096 trees (default net, hand-written tower, bf16, eager launches), with the
   leaf-frame mode off, "board" and "full" alternated in one run: every round sets the mode, resets the trees, grows
   them with 30 untimed simulations and then times 20 steps with CUDA events.
2. hz_sym_states and hz_sym_actions (int16 visits, fp32 policies) at 1 M rows against a device copy of the same bytes.

    python profiles/symmetry_step.py [--games 4096] [--rounds 6] [--out result.json]
"""

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from harmonies_alphazero_b200 import batched as hb  # noqa: E402
from harmonies_alphazero_b200 import net as hznet  # noqa: E402
from harmonies_alphazero_b200 import selfplay as sp  # noqa: E402
from harmonies_alphazero_b200 import symmetry as sy  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--games", type=int, default=4096)
ap.add_argument("--rounds", type=int, default=6)
ap.add_argument("--rows", type=int, default=1 << 20)
ap.add_argument("--out", default=None)
a = ap.parse_args()

assert torch.cuda.is_available(), "needs a CUDA device"
dev = torch.device("cuda", 0)
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
except Exception:  # noqa: BLE001
    gpu = torch.cuda.get_device_name(dev)
out = {"gpu": gpu, "games": a.games}


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


# ---- 1. simulation step ----------------------------------------------------------------------------
torch.manual_seed(0)
model = hznet.AlphaZeroNet.from_config(hznet.DEFAULT_MODEL_CONFIG).eval()
inf = hznet.InferenceNet(model, device=dev, dtype=torch.bfloat16, tower="hand")
cfg = sp.SelfPlayConfig(n_slots=a.games, num_simulations=64, use_cuda_graph=False, seed=77)
drv = sp.BatchedSelfPlay(inf, cfg, device=dev)
g = drv.groups[0]
states = hb.init_states(a.games, device=dev, seed=77)
hb.playout(states, max_steps=8)
modes = [None, "board", "full"]
steps = {str(m): [] for m in modes}
for r in range(a.rounds):
    for m in (modes if r % 2 == 0 else modes[::-1]):
        g.tree.set_symmetry(m)                  # a search runs in one mode (hz_tree_set_symmetry)
        g.prepare(states)
        for _ in range(30):
            drv._sim_step()
        torch.cuda.synchronize()
        for _ in range(20):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(400_000)      # the GPU stays busy while the host enqueues: device time, not launch latency
            e0.record()
            drv._sim_step()
            e1.record()
            torch.cuda.synchronize()
            steps[str(m)].append(e0.elapsed_time(e1) * 1e3)
        g.tree.check_status()
out["step_us_median"] = {k: median(v) for k, v in steps.items()}
out["step_us_all"] = steps
base = out["step_us_median"]["None"]
out["step_cost_vs_off_pct"] = {k: 100.0 * (v - base) / base for k, v in out["step_us_median"].items()}

# select / expand alone, mode by mode (the two kernels the mode touches), same warm trees
parts = {}
for m in modes:
    g.tree.set_symmetry(m)
    g.prepare(states)
    for _ in range(30):
        drv._sim_step()
    sel, exp = [], []
    for _ in range(20):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        torch.cuda._sleep(400_000)
        e0.record()
        g.tree.select(cfg.cpuct, g.board, g.glob, dtype=inf.dtype, channels_last=True, pad40=drv.pad40, tiles=g.tiles)
        e1.record()
        inf.forward_tiles(g.board, g.glob, g.glob.shape[0], out=(g.logits, g.value))
        torch.cuda.synchronize()
        torch.cuda._sleep(400_000)
        e2b = torch.cuda.Event(enable_timing=True)
        e2b.record()
        g.tree.expand_backup(g.logits, g.value, is_logits=True, noise=g.noise, eps=cfg.dirichlet_epsilon)
        e2.record()
        torch.cuda.synchronize()
        sel.append(e0.elapsed_time(e1) * 1e3)
        exp.append(e2b.elapsed_time(e2) * 1e3)
    parts[str(m)] = {"select_us": median(sel), "expand_backup_us": median(exp)}
out["kernels_us_median"] = parts
del drv, g

# ---- 2. bulk transforms at 1 M rows ---------------------------------------------------------------------
n = a.rows
st = hb.init_states(n, device=dev, seed=5)
hb.playout(st, max_steps=40)
sym = torch.randint(0, 480, (n,), device=dev).to(torch.int16)
dst = torch.empty_like(st)
visits = torch.randint(0, 50, (n, 143), device=dev, dtype=torch.int16)
pol = torch.rand((n, 143), device=dev)
vout, pout = torch.empty_like(visits), torch.empty_like(pol)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # 256 MB: evicts the 126 MB L2 between passes


def bulk(fn, reps=20):
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return median(ts)


for _ in range(2):
    sy.transform_states(st, sym, out=dst)
    sy.transform_actions(visits, sym, st)
b = {}
b["sym_states_us"] = bulk(lambda: sy.transform_states(st, sym, out=dst))
b["copy_states_us"] = bulk(lambda: dst.copy_(st))
b["sym_actions_i16_us"] = bulk(lambda: hb._lib.check(hb._lib.load().hz_sym_actions(
    visits.data_ptr(), n, 2, sym.data_ptr(), st.data_ptr(), 0, vout.data_ptr(), torch.cuda.current_stream().cuda_stream)))
b["copy_i16_us"] = bulk(lambda: vout.copy_(visits))
b["sym_actions_f32_us"] = bulk(lambda: hb._lib.check(hb._lib.load().hz_sym_actions(
    pol.data_ptr(), n, 0, sym.data_ptr(), st.data_ptr(), 0, pout.data_ptr(), torch.cuda.current_stream().cuda_stream)))
b["copy_f32_us"] = bulk(lambda: pout.copy_(pol))
b["rows"] = n
b["states_GBps"] = 2 * 128 * n / (b["sym_states_us"] * 1e3)
b["copy_states_GBps"] = 2 * 128 * n / (b["copy_states_us"] * 1e3)
out["bulk"] = b

s = json.dumps(out)
print(s)
if a.out:
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")
