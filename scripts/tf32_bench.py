#!/usr/bin/env python
"""TF32 precision against bf16 and cuDNN TF32 on the benchmark's nets (chess 16x128 b1024, go-9 20x256 b4096, go-19 40x256 b8192).

For every net, in one process: the staged step (kzb_time_staged, L2 flushed before every step) of the bf16 and the TF32 network,
alternated bf16 / TF32 / bf16 / TF32; per-launch times (kzb_profile_staged) for the tower's share; fp32 on chess only; and the cuDNN
TF32 NCHW tower (bench.gpu_comparator) on the same weights and batch.  Tower TFLOP/s are algorithmic (no padding), against the
data-sheet dense TF32 rate of one B200 (1,125 TFLOP/s) and against our own bf16 rate.  Prints the card name and power limit and
writes the JSON to --out (default profiles/tf32_bench.json).
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from kzero_b200 import netgen  # noqa: E402
from kzero_b200.network import B200Network, PRECISION_BF16, PRECISION_FP32, PRECISION_TF32, mapper_for  # noqa: E402

TF32_DENSE_TFLOPS = 1125.0  # HGX B200 data sheet, one GPU, dense
CONFIGS = [("chess", 16, 128, 1024), ("go-9", 20, 256, 4096), ("go-19", 40, 256, 8192)]
NAMES = {PRECISION_BF16: "bf16", PRECISION_TF32: "tf32", PRECISION_FP32: "fp32"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown (no nvidia-smi)"
    return q.stdout.strip().split("\n")[0] if q.returncode == 0 else "unknown"


def tower_flops(spec, depth, ch, batch):
    return batch * (2.0 * spec.area * 9 * spec.input_channels * ch + depth * 2 * (2.0 * spec.area * 9 * ch * ch))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--comparator-iters", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "tf32_bench.json"))
    args = ap.parse_args()
    gpu = card()
    print(f"card: {gpu}", flush=True)
    results = {"card": gpu, "steps": args.steps, "l2": "flushed before every timed step", "tf32_dense_tflops_datasheet": TF32_DENSE_TFLOPS,
               "configs": {}}
    for game, depth, ch, batch in CONFIGS:
        spec = netgen.game_spec(game)
        weights = {}
        onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=0, weights_out=weights)
        bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, batch, seed=1)
        flops = tower_flops(spec, depth, ch, batch)
        precisions = [PRECISION_BF16, PRECISION_TF32] + ([PRECISION_FP32] if game == "chess" else [])
        nets = {}
        for prec in precisions:
            net = B200Network(mapper_for(spec), onnx_bytes, batch, precision=prec)
            for _ in range(2):
                net.evaluate_packed(bits, scalars, mv_idx, mv_off)
            net.stage_packed(bits, scalars, mv_idx, mv_off)
            net.time_staged(2, True)
            nets[prec] = net
        step_ms = {p: [] for p in precisions}
        for _ in range(2):  # bf16 / TF32 / bf16 / TF32 (fp32 once, chess only)
            for prec in (PRECISION_BF16, PRECISION_TF32):
                step_ms[prec] += [float(v) for v in nets[prec].time_staged(args.steps, True)]
        if PRECISION_FP32 in nets:
            step_ms[PRECISION_FP32] = [float(v) for v in nets[PRECISION_FP32].time_staged(max(2, args.steps // 2), True)]
        row = {"depth": depth, "channels": ch, "batch": batch, "tower_algorithmic_flops": flops, "precisions": {}}
        for prec in precisions:
            names, ms = nets[prec].profile_staged(True)
            tower = float(sum(m for n, m in zip(names, ms) if bench.TOWER_STEP(n)))
            med = float(np.median(step_ms[prec]))
            row["precisions"][NAMES[prec]] = {
                "ms_per_step_median": med, "ms_per_step_min": float(min(step_ms[prec])), "ms_per_step_all": step_ms[prec],
                "positions_per_s": batch / (med * 1e-3), "tower_ms_profiled": tower,
                "tower_tflops_algorithmic": flops / (tower * 1e-3) / 1e12, "launches_per_eval": nets[prec].launches_per_eval(),
                "conv_mode": int(nets[prec].info().conv_mode)}
        for net in nets.values():
            net.close()
        bf, tf = row["precisions"]["bf16"], row["precisions"]["tf32"]
        tf["tower_share_of_tf32_datasheet"] = tf["tower_tflops_algorithmic"] / TF32_DENSE_TFLOPS
        tf["tower_rate_vs_our_bf16"] = tf["tower_tflops_algorithmic"] / bf["tower_tflops_algorithmic"]
        tf["step_time_vs_bf16"] = tf["ms_per_step_median"] / bf["ms_per_step_median"]
        cfg = {"depth": depth, "channels": ch, "batch": batch}
        row["cudnn"] = bench.gpu_comparator(cfg, spec, weights, 0, args.comparator_iters, variants=("tf32_nchw",))
        cud = row["cudnn"]["variants"].get("tf32_nchw", {})
        if "ms_per_tower" in cud:
            tf["tower_vs_cudnn_tf32"] = cud["ms_per_tower"] / tf["tower_ms_profiled"]
        results["configs"][f"{game} {depth}x{ch} b{batch}"] = row
        print(json.dumps({game: {k: {kk: vv for kk, vv in v.items() if kk != "ms_per_step_all"} for k, v in row["precisions"].items()},
                          "cudnn_tf32_ms_per_tower": cud.get("ms_per_tower")}), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1) + "\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
