"""Phase timeline of one hz_playout wave, measured on the device (-DHZ_PLAYOUT_TIMELINE builds of hz_engine.cu).

Builds two profiling libraries from this tree's sources, both with the time stamps compiled in:
  one_trip_tables  the default: the block's neighbour LUT and rand table fetched in one round trip (fetch_tables)
  looped_tables    -DHZ_PLAYOUT_LOOPED_TABLES: the looped copies of build_nbr_lut / build_rand_table, four round trips
                   in a row (the prologue before fetch_tables; without the time stamps its k_playout is the same SASS)
and runs one L2-flushed wave of `n` fresh games on each, after warm-up waves.  Each warp's lowest active lane writes
%globaltimer and clock64 at kernel entry, tables ready, records in registers, the end of every round of play_random,
the end of play_random, after partial_scores, after resolve_water and after the store (k_playout in hz_engine.cu).
Phase durations come from clock64 differences inside a warp (same SM), converted with the SM clock measured against
%globaltimer; cross-SM times use %globaltimer.  Reports the median and p99 of every phase over the warps, the split of
the median and of the last warp, and the number of warps in each phase over time on the slowest SM.

    python profiles/playout_timeline.py [--games 65536] [--libdir DIR] [--build-only] [--json FILE]

The libraries go to DIR (default: a directory under the system temp dir) and are rebuilt when older than the sources.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from harmonies_alphazero_b200 import build  # noqa: E402

VARIANTS = {"one_trip_tables": [], "looped_tables": ["-DHZ_PLAYOUT_LOOPED_TABLES"]}
EVENTS = ["entry", "tables", "records", "played", "partial", "resolved", "stored"]
TL_ROUND, TL_ROUNDS, TL_WORDS = len(EVENTS), 24, 64       # as in hz_engine.cu


def build_variant(libdir, name, flags):
    lib = os.path.join(libdir, f"libhz_timeline_{name}.so")
    srcs = [os.path.join(build.CSRC, f) for f in ("hz_abi.cu", "hz_engine.cu")]
    deps = [os.path.join(build.CSRC, f) for f in os.listdir(build.CSRC)] + [os.path.abspath(__file__)]
    if os.path.exists(lib) and all(os.path.getmtime(d) <= os.path.getmtime(lib) for d in deps):
        return lib
    cmd = [build._nvcc()] + build.NVCC_FLAGS + ["-DHZ_PLAYOUT_TIMELINE"] + flags + ["-shared", "-o", lib] + srcs
    subprocess.run(cmd, check=True)
    return lib


def run_wave(lib_path, n, warmup):
    import torch

    lib = C.CDLL(lib_path)
    vp, i64 = C.c_void_p, C.c_int64
    lib.hz_init_states.argtypes = [vp, i64, vp, C.c_uint64, C.c_uint64, vp]
    lib.hz_playout.argtypes = [vp, i64, C.c_int, vp, vp, vp]
    lib.hz_playout_set_timeline.argtypes = [vp, C.c_longlong]
    dev = torch.device("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    states = torch.empty((n, 32), dtype=torch.int32, device=dev)
    steps = torch.empty(n, dtype=torch.int32, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB of L2
    n_warps = (n + 31) // 32
    tl = torch.zeros((n_warps, TL_WORDS), dtype=torch.int64, device=dev)

    def wave(seed):
        assert lib.hz_init_states(states.data_ptr(), n, None, seed, 0, stream) == 0
        flush.fill_(seed & 255)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        assert lib.hz_playout(states.data_ptr(), n, 1000, steps.data_ptr(), total.data_ptr(), stream) == 0
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3

    for w in range(warmup):
        wave(100 + w)
    assert lib.hz_playout_set_timeline(tl.data_ptr(), n_warps) == 0
    total.zero_()
    us = wave(1000)
    assert lib.hz_playout_set_timeline(None, 0) == 0
    checksum = int(states.to(torch.int64).sum().item()) ^ int(total.item())
    return us, tl.cpu().numpy().view(np.uint64).astype(np.int64), checksum


def pct(x, q):
    x = x[~np.isnan(x)]
    return float(np.percentile(x, q)) if len(x) else float("nan")


def analyse(us, raw):
    smid = raw[:, 0]
    gt = {e: raw[:, 1 + 2 * i] for i, e in enumerate(EVENTS)}
    ck = {e: raw[:, 2 + 2 * i] for i, e in enumerate(EVENTS)}
    rgt = np.stack([raw[:, 1 + 2 * (TL_ROUND + r)] for r in range(TL_ROUNDS)], 1)
    rck = np.stack([raw[:, 2 + 2 * (TL_ROUND + r)] for r in range(TL_ROUNDS)], 1)
    n_rounds = (rgt > 0).sum(1)
    ghz = float(np.median((ck["stored"] - ck["entry"]) / (gt["stored"] - gt["entry"])))     # SM cycles per ns

    def dur(a, b, sel=True):                        # us per warp from clock64 (same SM); NaN where sel is false
        return np.where(sel, (b - a) / ghz / 1e3, np.nan)

    full = n_rounds >= 7
    last_round = rck[np.arange(len(raw)), np.maximum(n_rounds - 1, 0)]
    phases = {
        "prologue (entry -> tables ready)": dur(ck["entry"], ck["tables"]),
        "record load (tables ready -> records in registers)": dur(ck["tables"], ck["records"]),
        "rounds 1-7": dur(ck["records"], rck[:, 6], full),
    }
    prev = ck["records"]
    for r in range(10):
        sel = n_rounds > r
        phases[f"round {r + 1}"] = dur(prev, rck[:, r], sel)
        prev = np.where(sel, rck[:, r], prev)
    phases["rounds 8+ (round 7 -> end of play_random)"] = dur(rck[:, 6], ck["played"], full)
    phases["end of the loop (last round -> end of play_random)"] = dur(last_round, ck["played"], n_rounds > 0)
    phases["final scoring (partial_scores)"] = dur(ck["played"], ck["partial"])
    phases["resolve_water + block barriers"] = dur(ck["partial"], ck["resolved"])
    phases["store"] = dur(ck["resolved"], ck["stored"])
    phases["scoring and store"] = dur(ck["played"], ck["stored"])
    phases["warp lifetime (entry -> stored)"] = dur(ck["entry"], ck["stored"])
    t0 = gt["entry"].min()
    end = (gt["stored"] - t0) / 1e3
    w = int(np.argmax(gt["stored"]))                 # the last warp to finish
    out = {
        "event_us": us, "warps": int(len(raw)), "sm_clock_ghz": ghz,
        "span_us": float((gt["stored"].max() - t0) / 1e3),
        "entry_spread_us": float((gt["entry"].max() - t0) / 1e3),
        "warp_end_us": {"median": pct(end, 50), "p99": pct(end, 99), "max": float(end.max())},
        "rounds_per_warp": {str(int(k)): int(v) for k, v in zip(*np.unique(n_rounds, return_counts=True))},
        "phases": {k: {"median": pct(v, 50), "p99": pct(v, 99), "last_warp": None if np.isnan(v[w]) else float(v[w]),
                       "warps": int((~np.isnan(v)).sum())} for k, v in phases.items()},
        "last_warp": {"warp": w, "sm": int(smid[w]), "rounds": int(n_rounds[w]),
                      "entry_after_first_us": float((gt["entry"][w] - t0) / 1e3)},
    }
    # warps per phase over time on the slowest SM (the one whose last warp stores last), in its own clock
    sm = int(smid[w])
    on = np.flatnonzero(smid == sm)
    c0 = ck["entry"][on].min()
    rel = lambda x: (x[on] - c0) / ghz / 1e3                         # noqa: E731
    bounds = [("prologue", rel(ck["entry"])), ("load", rel(ck["tables"])), ("rounds 1-7", rel(ck["records"])),
              ("round 8", np.where(n_rounds[on] >= 7, rel(rck[:, 6]), rel(ck["played"]))),
              ("round 9+", np.where(n_rounds[on] >= 8, rel(rck[:, 7]), rel(ck["played"]))),
              ("scoring", rel(ck["played"])), ("store", rel(ck["resolved"])), ("done", rel(ck["stored"]))]
    names = [b[0] for b in bounds]
    starts = np.stack([b[1] for b in bounds], 1)
    horizon = float(starts[:, -1].max())
    series = []
    for t in np.arange(0.0, horizon + 1.0, 1.0):
        phase = (starts <= t).sum(1) - 1                             # -1: not started yet
        series.append([round(float(t), 2)] + [int((phase == i).sum()) for i in range(len(names))])
    out["slowest_sm"] = {"sm": sm, "warps": int(len(on)), "columns": ["t_us"] + names, "series": series}
    return out


def print_report(name, r):
    print(f"== {name}: wave {r['event_us']:.2f} us (CUDA events, timeline build), {r['warps']} warps, "
          f"SM clock {r['sm_clock_ghz']:.3f} GHz, first entry -> last store {r['span_us']:.2f} us, "
          f"entries spread over {r['entry_spread_us']:.2f} us")
    we = r["warp_end_us"]
    print(f"   warp end after first entry: median {we['median']:.2f}  p99 {we['p99']:.2f}  max {we['max']:.2f} us; "
          f"loop iterations per warp {r['rounds_per_warp']}")
    print(f"   {'phase':56s} {'median':>8s} {'p99':>8s} {'last warp':>10s}  warps")
    for k, v in r["phases"].items():
        lw = "" if v["last_warp"] is None else f"{v['last_warp']:.2f}"
        print(f"   {k:56s} {v['median']:8.2f} {v['p99']:8.2f} {lw:>10s}  {v['warps']}")
    s = r["slowest_sm"]
    print(f"   warps per phase over time on the slowest SM ({s['sm']}, {s['warps']} warps, its own clock):")
    print("   " + " ".join(f"{c:>10s}" for c in s["columns"]))
    for row in s["series"]:
        print("   " + " ".join(f"{x:10}" for x in row))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=65536)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--libdir", default=os.path.join(tempfile.gettempdir(), "hz_playout_timeline"))
    ap.add_argument("--build-only", action="store_true")
    ap.add_argument("--json", help="write the reports (and nothing else) to this file")
    a = ap.parse_args()
    os.makedirs(a.libdir, exist_ok=True)
    libs = {name: build_variant(a.libdir, name, flags) for name, flags in VARIANTS.items()}
    if a.build_only:
        print("\n".join(libs.values()))
        return
    reports, sums = {}, {}
    for name, lib in libs.items():
        us, raw, sums[name] = run_wave(lib, a.games, a.warmup)
        reports[name] = analyse(us, raw)
        reports[name]["checksum"] = sums[name]
        print_report(name, reports[name])
    print("checksums:", sums, "identical" if len(set(sums.values())) == 1 else "DIFFERENT")
    if a.json:
        with open(a.json, "w") as f:
            json.dump(reports, f, indent=1)


if __name__ == "__main__":
    main()
