"""Training-propagation timing of the two backward precisions: forward (saving activations) + backward per step, fp32 FFMA backward against
the tensor-core bf16x3 backward, on cfg2, cfg4, cfg5_rgcn and the 100 000-node default batch (workloads.py).

Method of bench.py: inputs resident in HBM, L2 flushed by a 256 MiB write (untimed) before every timed step, CUDA events around each
step, the two precisions alternated step by step in one process on one engine (so clocks and thermal state are shared).  Also reports
launches per backward, the largest per-piece difference between the two precisions' gradients (relative to the piece's max |fp32
value|), whether two bf16x3 backward calls give identical bits, and the card's name and power limit read in the same run.

    python tools/bench_backward.py --steps 20 --warmup 3 --out DIR      -> DIR/bench_backward.json (nothing is written in the tree)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = ["cfg2", "cfg4", "cfg5_rgcn", "default_batch_100k_nodes"]


def card_info():
    import torch
    info = {"name": torch.cuda.get_device_name(), "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as ex:   # the numbers stay valid without it; say why the power limit is missing
        info["nvidia_smi"] = "unavailable: %s" % ex
    return info


def pieces(key, g, D, R):
    from tests.test_gpu_backward_edges import gradient_pieces
    return gradient_pieces(key, g, D, R)


def max_piece_diff(a, b, key, D, R):
    """max over pieces of max|a - b| / max|b piece| (pieces whose fp32 value is all zero must match exactly: reported as 0 or inf)"""
    worst = 0.0
    for (_, pa), (_, pb) in zip(pieces(key, a, D, R), pieces(key, b, D, R)):
        m = float(np.max(np.abs(pb))) if pb.size else 0.0
        d = float(np.max(np.abs(pa - pb))) if pb.size else 0.0
        worst = max(worst, d / m if m > 0 else (0.0 if d == 0 else float("inf")))
    return worst


def run_config(name, steps, warmup, flush_buf, fwd_precision):
    import torch
    from gated_graph_neural_network_samples_b200 import workloads
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine, residual_inputs_of_layer
    w = workloads.build(name)
    p, T = w["engine_params"], w["num_edge_types"]
    D = int(p["hidden_size"])
    eng = PropagationEngine(p, T, precision=fwd_precision)
    dev_w = [{k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in lw.items()} for lw in w["weights"]]
    eng.set_weights(dev_w)
    eng.set_save_for_backward(True)
    eng.set_graph_sparse(w["adjacency_lists"], w["num_incoming_edges_per_type"])
    h0 = torch.from_numpy(w["h0"]).cuda()
    out = torch.empty_like(h0)
    d_out = torch.from_numpy(np.random.default_rng(3).normal(size=w["h0"].shape).astype(np.float32)).cuda()
    d_h0 = torch.empty_like(h0)
    grads = {bp: [{k: torch.zeros_like(v) for k, v in lw.items()} for lw in dev_w] for bp in ("fp32", "bf16x3")}
    launches = {}

    def step(bp):
        eng.forward(h0, out)
        eng.set_backward_precision(bp)
        eng.backward(d_out, grads[bp], d_h0)

    for _ in range(max(warmup, 1)):
        for bp in ("fp32", "bf16x3"):
            step(bp)
            launches[bp] = eng.last_launch_count
    torch.cuda.synchronize()
    ev = {bp: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)] for bp in ("fp32", "bf16x3")}
    for i in range(steps):
        for bp in ("fp32", "bf16x3"):   # alternated: both see the same clocks
            flush_buf.fill_(1)
            ev[bp][i][0].record()
            step(bp)
            ev[bp][i][1].record()
    torch.cuda.synchronize()
    eng.sync_check()
    ms = {bp: [a.elapsed_time(b) for a, b in ev[bp]] for bp in ev}

    # accuracy and reproducibility on one forward: fresh zeroed buffers per precision
    eng.forward(h0, out)
    res = {}
    for bp in ("fp32", "bf16x3", "bf16x3 again"):
        g = [{k: torch.zeros_like(v) for k, v in lw.items()} for lw in dev_w]
        d = torch.empty_like(h0)
        eng.set_backward_precision(bp.split()[0])
        eng.backward(d_out, g, d)
        res[bp] = (d, g)
    eng.sync_check()
    diff = {"d_h0": max_piece_diff(res["bf16x3"][0].cpu().numpy(), res["fp32"][0].cpu().numpy(), "d_h0", D, 0)}
    for l, (a, b) in enumerate(zip(res["bf16x3"][1], res["fp32"][1])):
        R = len(residual_inputs_of_layer(p, l))
        for k in b:
            diff["layer %d %s" % (l, k)] = max_piece_diff(a[k].cpu().numpy(), b[k].cpu().numpy(), k, D, R)
    same = bool(torch.equal(res["bf16x3"][0], res["bf16x3 again"][0])) and all(
        torch.equal(la[k], lb[k]) for la, lb in zip(res["bf16x3"][1], res["bf16x3 again"][1]) for k in la)
    med = {bp: float(np.median(v)) for bp, v in ms.items()}
    return {"config": name, "V": w["V"], "M": w["M"], "hidden_size": D, "edge_types": T, "layer_timesteps": p["layer_timesteps"],
            "forward_plan": eng.plan, "steps": steps,
            "ms_forward_plus_backward": {bp: {"median": med[bp], "min": float(np.min(v)), "mean": float(np.mean(v))} for bp, v in ms.items()},
            "speedup_bf16x3_over_fp32": med["fp32"] / med["bf16x3"],
            "launches_per_backward": launches,
            "max_piece_rel_diff_bf16x3_vs_fp32": max(diff.values()), "per_gradient_rel_diff": diff,
            "bf16x3_bit_reproducible": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--forward-precision", default="bf16x3")
    ap.add_argument("--out", required=True, help="output directory for bench_backward.json")
    args = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    result = {"card": card_info(), "method": "forward(save) + backward per step, L2 flushed (256 MiB write, untimed) before each step, CUDA events, "
                                            "fp32 and bf16x3 backward alternated step by step on one engine",
              "forward_precision": args.forward_precision, "configs": []}
    for name in args.configs.split(","):
        r = run_config(name, args.steps, args.warmup, flush_buf, args.forward_precision)
        print(json.dumps({k: r[k] for k in ("config", "ms_forward_plus_backward", "speedup_bf16x3_over_fp32", "launches_per_backward",
                                            "max_piece_rel_diff_bf16x3_vs_fp32", "bf16x3_bit_reproducible")}), flush=True)
        result["configs"].append(r)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_backward.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
