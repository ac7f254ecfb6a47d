"""Times the hand-written tower (csrc/hz_tower.cu) against the cuDNN tower on the same box:
per 3x3 residual convolution and for the whole stem + 8-block tower, at the self-play batch
(4,096 boards) and a 4x batch.  CUDA events on the launching stream, warm-up, L2 flushed between
timed iterations for the single-layer numbers (the whole tower's working set exceeds nothing: its
activations live in L2 in both implementations, which is the regime self-play runs in).

usage: python profiles/tower_bench.py [--boards 4096] [--iters 20] [--json out.json]
"""

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from harmonies_alphazero_b200 import net as hnet  # noqa: E402


def timeit(fn, iters, flush=None):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return {"us_min": ts[0], "us_med": ts[len(ts) // 2]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--boards", type=int, default=4096)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    torch.manual_seed(0)
    model = hnet.AlphaZeroNet.from_config(hnet.DEFAULT_MODEL_CONFIG).eval()
    hand = hnet.InferenceNet(model, tower="hand")
    lib = hnet.InferenceNet(model, tower="cudnn")
    B = a.boards
    board = torch.zeros((B, 40, 5, 7), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
    board[:, :38] = (torch.rand((B, 38, 5, 7), device="cuda") < 0.15).to(torch.bfloat16)
    glob = torch.rand((B, 42), device="cuda").to(torch.bfloat16)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = {"boards": B, "gpu": torch.cuda.get_device_name(0)}
    dense_flop = 2.0 * B * 35 * 9 * 128 * 128
    # one residual convolution (128 -> 128, residual + ReLU)
    ht = hand.hand
    n_pad = (B + 15) // 16 * 16
    buf = ht._buffers(n_pad)
    hand.tower_out(board)      # fills the tile buffers with real activations
    c1, c2 = ht.blocks[0]
    r = timeit(lambda: ht.conv(buf["a"], 2, c2, buf["b"], buf["c"], n_pad), a.iters, flush)
    r["dense_equiv_tflops"] = dense_flop / r["us_min"] / 1e6
    r["executed_tflops"] = dense_flop * 247 / 315 / r["us_min"] / 1e6
    out["hand_conv_l2_flushed"] = r
    r = timeit(lambda: ht.conv(buf["a"], 2, c2, buf["b"], buf["c"], n_pad), a.iters)
    r["dense_equiv_tflops"] = dense_flop / r["us_min"] / 1e6
    out["hand_conv_warm"] = r
    # attribution: the same launch with parts switched off (results are garbage, timing only)
    attr = {}
    for flags, name in ((1, "no_mma"), (2, "no_epilogue_mem"), (4, "no_weight_copies"), (8, "no_act_copies"), (12, "no_copies"),
                        (3, "no_mma_no_epi_mem"), (13, "copies_off_mma_off"), (15, "barriers_only")):
        ht.lib.hz_tower_set_debug(flags)
        attr[name] = timeit(lambda: ht.conv(buf["a"], 2, c2, buf["b"], buf["c"], n_pad), a.iters)["us_min"]
    ht.lib.hz_tower_set_debug(0)
    out["hand_conv_attribution_us"] = attr
    # role timeline of CTA 0 (SM clocks) for the fused all-layers launch
    def trace_run(fn, n_stage=600, n_rows=200):
        tr = torch.zeros(4096, dtype=torch.int64, device="cuda")
        ht.lib.hz_tower_set_trace(tr.data_ptr())
        fn()
        torch.cuda.synchronize()
        ht.lib.hz_tower_set_trace(None)
        t = tr.cpu().numpy().astype("int64")
        t0 = int(t[0])
        rel = lambda v: int(v - t0) if v else None  # noqa: E731
        stages = [(rel(t[16 + 3 * i]), rel(t[16 + 3 * i + 1]), rel(t[16 + 3 * i + 2])) for i in range(n_stage) if t[16 + 3 * i + 2]]
        rows = [tuple(rel(t[2700 + 4 * j + k]) for k in range(4)) for j in range(n_rows) if t[2700 + 4 * j + 3]]
        waits = [b - a for a, b, _ in stages]
        issues = [c - b for _, b, c in stages]
        cyc, ns = rel(t[1]), int(t[3] - t[2])
        return {"total_cycles": cyc, "total_ns": ns, "sm_ghz": cyc / ns if ns else None, "n_stages": len(stages),
                "mma_wait_cycles_total": sum(waits), "mma_issue_cycles_total": sum(issues), "mma_wait_max": max(waits) if waits else None,
                "stage_period_avg": (stages[-1][2] - stages[0][0]) / len(stages) if stages else None,
                "stages(before_wait,after_wait,after_issue)": stages, "weight_issue": [rel(t[2000 + i]) for i in range(n_stage) if t[2000 + i]],
                "act_issue": [rel(t[3600 + i]) for i in range(64) if t[3600 + i]],
                "epilogue_rows(before_wait,after_wait,after_tmem_ld,after_stores)": rows,
                "epilogue_wait_total": sum(r[1] - r[0] for r in rows), "epilogue_work_total": sum(r[3] - r[1] for r in rows)}

    x0t = hand.hand.x0_buffer(B)
    hand.hand.to_tiles(board, 40, True, x0t)
    out["trace_fused"] = trace_run(lambda: hand.hand.forward_tiles(x0t, B))
    ht.lib.hz_tower_set_debug(14)
    out["trace_fused_mma_only"] = trace_run(lambda: hand.hand.forward_tiles(x0t, B))
    ht.lib.hz_tower_set_debug(0)
    out["trace_summary"] = {k: {kk: vv for kk, vv in out[k].items() if not isinstance(vv, list)} for k in ("trace_fused", "trace_fused_mma_only")}
    hand.tower_out(board)
    x = lib.tower_out(board)
    r = timeit(lambda: lib._conv_relu(x, lib.blocks[0][1], 1, residual=x), a.iters, flush)
    r["dense_equiv_tflops"] = dense_flop / r["us_min"] / 1e6
    out["cudnn_conv_l2_flushed"] = r
    r = timeit(lambda: lib._conv_relu(x, lib.blocks[0][1], 1, residual=x), a.iters)
    r["dense_equiv_tflops"] = dense_flop / r["us_min"] / 1e6
    out["cudnn_conv_warm"] = r
    # whole tower and whole forward (tower + heads), CUDA graph replay like self-play
    for name, net in (("hand", hand), ("cudnn", lib)):
        logits = torch.zeros((B, 143), dtype=torch.float32, device="cuda")
        value = torch.zeros(B, dtype=torch.float32, device="cuda")
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                net(board, glob, out=(logits, value))
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            net(board, glob, out=(logits, value))
        r = timeit(g.replay, a.iters)
        r["net_tflops"] = hnet.flops_per_position() * B / r["us_min"] / 1e6
        out[name + "_forward_graph"] = r
        gt = torch.cuda.CUDAGraph()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            net.tower_out(board)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        with torch.cuda.graph(gt):
            net.tower_out(board)
        out[name + "_tower_graph"] = timeit(gt.replay, a.iters)
    # attribution of the fused all-layers launch (eager; results are garbage with a switch on)
    x0 = hand.hand.x0_buffer(B)
    hand.hand.to_tiles(board, 40, True, x0)
    fa = {}
    for flags, name in ((0, "full"), (4, "no_weight_copies"), (8, "no_act_copies"), (2, "no_epilogue_mem"), (12, "no_copies"), (14, "mma_only"), (1, "no_mma")):
        ht.lib.hz_tower_set_debug(flags)
        fa[name] = timeit(lambda: hand.hand.forward_tiles(x0, B), a.iters)["us_min"]
    ht.lib.hz_tower_set_debug(0)
    out["hand_tower_fused_attribution_us"] = fa
    lh, vh = hand(board, glob)
    ll, vl = lib(board, glob)
    out["max_logit_diff_hand_vs_cudnn"] = float((lh - ll).abs().max())
    out["max_value_diff_hand_vs_cudnn"] = float((vh - vl).abs().max())
    print(json.dumps(out, indent=1))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
