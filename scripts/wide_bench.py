#!/usr/bin/env python
"""Towers wider than 256 channels against the 256-wide go-9 net and against cuDNN on the same shapes.

Nets: go-9 20x384 b4096, go-19 20x384 b4096, chess 16x384 b1024, chess 10x512 b1024 and, as the control, go-9 20x256 b4096.  For
every net, in one process: the staged bf16 step (kzb_time_staged, L2 flushed before every step); per-launch times
(kzb_profile_staged, L2 flushed) for the tower's share and the per-launch profile; algorithmic tower TFLOP/s (real channels, no
padding); the cuDNN bf16 channels_last tower (bench.gpu_comparator) on the same weights and batch; TF32 on go-9 20x384.  Prints the
card name and power limit and writes the JSON to --out (default profiles/wide_bench.json).
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
from kzero_b200.network import B200Network, PRECISION_BF16, PRECISION_TF32, mapper_for  # noqa: E402

CONTROL = ("go-9", 20, 256, 4096)
CONFIGS = [("go-9", 20, 384, 4096), ("go-19", 20, 384, 4096), ("chess", 16, 384, 1024), ("chess", 10, 512, 1024), CONTROL]
TF32_ON = ("go-9", 20, 384, 4096)
NAMES = {PRECISION_BF16: "bf16", PRECISION_TF32: "tf32"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown (no nvidia-smi)"
    return q.stdout.strip().split("\n")[0] if q.returncode == 0 else "unknown"


def tower_flops(spec, depth, ch, batch):
    return batch * (2.0 * spec.area * 9 * spec.input_channels * ch + depth * 2 * (2.0 * spec.area * 9 * ch * ch))


def measure(net, batch, flops, steps, profiles):
    step_ms = [float(v) for v in net.time_staged(steps, True)]
    runs = [net.profile_staged(True) for _ in range(profiles)]
    names = runs[0][0]
    per_launch = [float(np.mean([ms[i] for _, ms in runs])) for i in range(len(names))]
    tower = float(sum(m for n, m in zip(names, per_launch) if bench.TOWER_STEP(n)))
    med = float(np.median(step_ms))
    return {"ms_per_step_median": med, "ms_per_step_min": float(min(step_ms)), "positions_per_s": batch / (med * 1e-3),
            "tower_ms_profiled": tower, "tower_share_of_step": tower / float(sum(per_launch)),
            "tower_tflops_algorithmic": flops / (tower * 1e-3) / 1e12, "launches_per_eval": net.launches_per_eval(),
            "conv_mode": int(net.info().conv_mode), "per_launch_ms": dict(zip(names, per_launch))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--profiles", type=int, default=3, help="profiled steps averaged per net")
    ap.add_argument("--comparator-iters", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "wide_bench.json"))
    args = ap.parse_args()
    gpu = card()
    print(f"card: {gpu}", flush=True)
    results = {"card": gpu, "steps": args.steps, "l2": "flushed before every timed and every profiled step", "configs": {}}
    for game, depth, ch, batch in CONFIGS:
        spec = netgen.game_spec(game)
        weights = {}
        onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=0, weights_out=weights)
        bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, batch, seed=1)
        flops = tower_flops(spec, depth, ch, batch)
        row = {"depth": depth, "channels": ch, "batch": batch, "tower_algorithmic_flops": flops, "precisions": {}}
        for prec in [PRECISION_BF16] + ([PRECISION_TF32] if (game, depth, ch, batch) == TF32_ON else []):
            with B200Network(mapper_for(spec), onnx_bytes, batch, precision=prec) as net:
                for _ in range(2):
                    net.evaluate_packed(bits, scalars, mv_idx, mv_off)
                net.stage_packed(bits, scalars, mv_idx, mv_off)
                net.time_staged(2, True)
                row["precisions"][NAMES[prec]] = measure(net, batch, flops, args.steps, args.profiles)
        cfg = {"depth": depth, "channels": ch, "batch": batch}
        row["cudnn"] = bench.gpu_comparator(cfg, spec, weights, 0, args.comparator_iters, variants=("bf16_channels_last",))
        cud = row["cudnn"]["variants"].get("bf16_channels_last", {})
        bf = row["precisions"]["bf16"]
        if "ms_per_tower" in cud:
            bf["tower_speedup_vs_cudnn_bf16"] = cud["ms_per_tower"] / bf["tower_ms_profiled"]
        results["configs"][f"{game} {depth}x{ch} b{batch}"] = row
        print(json.dumps({f"{game} {depth}x{ch} b{batch}": {k: {kk: vv for kk, vv in v.items() if kk != "per_launch_ms"}
                                                            for k, v in row["precisions"].items()},
                          "cudnn_bf16_ms_per_tower": cud.get("ms_per_tower")}), flush=True)
    control = results["configs"]["%s %dx%d b%d" % CONTROL]["precisions"]["bf16"]["tower_tflops_algorithmic"]
    for row in results["configs"].values():
        row["precisions"]["bf16"]["tower_rate_vs_go9_20x256"] = row["precisions"]["bf16"]["tower_tflops_algorithmic"] / control
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1) + "\n")
    print(json.dumps({k: {"tower_tflops": round(v["precisions"]["bf16"]["tower_tflops_algorithmic"], 1),
                          "vs_control": round(v["precisions"]["bf16"]["tower_rate_vs_go9_20x256"], 3),
                          "vs_cudnn_bf16": v["precisions"]["bf16"].get("tower_speedup_vs_cudnn_bf16")}
                      for k, v in results["configs"].items()}), flush=True)
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
