#!/usr/bin/env python
"""A/B of two builds of the library on the row path's launches: the head 1x1 convs (scalar_conv, policy_conv2, att_conv*), the
tower layers and the staged step.

Each tree is a copy of the repository with its libkzb200.so built.  One worker process per (tree, repeat) runs every config, and
the repeats alternate the order of the trees, so both builds see the same machine state.  Per config and worker: the staged step
(kzb_time_staged, L2 flushed before every step) and the per-launch times (kzb_profile_staged, L2 flushed, averaged over
--profiles steps); the outputs of one packed evaluation are compared bit for bit between the trees.  Prints the card name and
power limit and writes the JSON to --out.

    python scripts/head_conv_ab.py --trees OLD_TREE . --labels parent new --reps 3 --out profiles/head_conv_ab.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent

# name -> (game, depth, channels, batch, precision, environment)
CONFIGS = {
    "go-9 20x256 b4096 bf16": ("go-9", 20, 256, 4096, "bf16", {}),
    "go-9 20x256 b4096 tf32": ("go-9", 20, 256, 4096, "tf32", {}),
    "go-19 40x256 b8192 bf16": ("go-19", 40, 256, 8192, "bf16", {}),
    "go-19 40x256 b8192 tf32": ("go-19", 40, 256, 8192, "tf32", {}),
    "chess 16x128 b1024 bf16 KZB_NO_HEADS8=1": ("chess", 16, 128, 1024, "bf16", {"KZB_NO_HEADS8": "1"}),
    "chess 16x128 b1024 tf32": ("chess", 16, 128, 1024, "tf32", {}),
    "chess-att 16x128 b1024 bf16": ("chess-att", 16, 128, 1024, "bf16", {}),
}


def tower_step(name):
    return name == "tower8" or name.startswith("conv_first") or name.startswith("block")


def head_step(name):
    return name in ("scalar_conv", "policy_conv2") or name.startswith("att_conv")


def worker(tree, steps, profiles, dump_dir):
    sys.path.insert(0, str(Path(tree).resolve()))
    from kzero_b200 import _abi, netgen
    from kzero_b200.network import B200Network, PRECISION_BF16, PRECISION_TF32, mapper_for

    print(f"  library {_abi.lib_path()}", file=sys.stderr, flush=True)
    out = {"configs": {}}
    for i, (name, (game, depth, ch, batch, prec, env)) in enumerate(CONFIGS.items()):
        os.environ.update(env)  # read when the network is created
        spec = netgen.game_spec(game)
        onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=0)
        inputs = netgen.synthetic_positions(spec, batch, seed=1)
        with B200Network(mapper_for(spec), onnx_bytes, batch, precision=PRECISION_TF32 if prec == "tf32" else PRECISION_BF16) as net:
            for _ in range(2):
                values, probs = net.evaluate_packed(*inputs)
            np.savez(Path(dump_dir) / f"{i}.npz", values=values, probs=probs)
            net.stage_packed(*inputs)
            net.time_staged(2, True)
            step_ms = [float(v) for v in net.time_staged(steps, True)]
            runs = [net.profile_staged(True) for _ in range(profiles)]
            launches = net.launches_per_eval()
        for k in env:
            del os.environ[k]
        names = runs[0][0]
        per_launch = {n: float(np.mean([ms[j] for _, ms in runs])) for j, n in enumerate(names)}
        out["configs"][name] = {"step_ms": step_ms, "per_launch_ms": per_launch, "launches_per_eval": launches}
        print(f"  {name}: step median {np.median(step_ms):.3f} ms", file=sys.stderr, flush=True)
    print(json.dumps(out))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown (no nvidia-smi)"
    return q.stdout.strip().split("\n")[0] if q.returncode == 0 else "unknown"


def spread(xs):
    return {"min": float(min(xs)), "max": float(max(xs)), "mean": float(np.mean(xs))}


def summarize(runs, labels):
    """per config: for the staged step (median of each repeat), the tower (sum of its launches), every head conv and every
    tower layer, the min / max / mean over the repeats of each tree"""
    summary = {}
    for name in CONFIGS:
        row = {}
        for lab in labels:
            reps = [r["configs"][name] for r in runs[lab]]
            names = list(reps[0]["per_launch_ms"])
            r = {"step_ms": spread([float(np.median(x["step_ms"])) for x in reps]),
                 "tower_ms": spread([sum(v for n, v in x["per_launch_ms"].items() if tower_step(n)) for x in reps]),
                 "launches_per_eval": reps[0]["launches_per_eval"]}
            for n in names:
                if head_step(n) or tower_step(n):
                    r[n] = spread([x["per_launch_ms"][n] for x in reps])
            row[lab] = r
        old, new = row[labels[0]], row[labels[1]]
        layers = [n for n in old if tower_step(n)]
        row["tower_layers_slower_than_parent_max"] = [n for n in layers if new[n]["mean"] > old[n]["max"]]
        row["step_slower_than_parent_max"] = new["step_ms"]["mean"] > old["step_ms"]["max"]
        row["head_ratio_new_over_old"] = {n: new[n]["mean"] / old[n]["mean"] for n in old if head_step(n)}
        summary[name] = row
    return summary


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs=2, help="two repository copies, each with its library built")
    ap.add_argument("--labels", nargs=2, default=["old", "new"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--profiles", type=int, default=3, help="profiled steps averaged per config and worker")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "head_conv_ab.json"))
    ap.add_argument("--worker", metavar="TREE", help=argparse.SUPPRESS)
    ap.add_argument("--dump", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        worker(args.worker, args.steps, args.profiles, args.dump)
        return
    if not args.trees:
        ap.error("--trees is required")
    gpu = card()
    print(f"card: {gpu}", flush=True)
    labels = list(args.labels)
    runs = {lab: [] for lab in labels}
    same = {}
    with tempfile.TemporaryDirectory() as tmp:
        for rep in range(args.reps):
            order = [0, 1] if rep % 2 == 0 else [1, 0]
            for t in order:
                dump = Path(tmp) / f"{t}_{rep}"
                dump.mkdir()
                print(f"rep {rep}: {labels[t]} ({args.trees[t]})", flush=True)
                r = subprocess.run([sys.executable, __file__, "--worker", args.trees[t], "--dump", str(dump), "--steps", str(args.steps),
                                    "--profiles", str(args.profiles)], stdout=subprocess.PIPE, text=True, check=True)
                runs[labels[t]].append(json.loads(r.stdout.strip().split("\n")[-1]))
        # outputs of the first repeat: bit for bit the same in both trees?
        for i, name in enumerate(CONFIGS):
            a, b = (np.load(Path(tmp) / f"{t}_0" / f"{i}.npz") for t in (0, 1))
            same[name] = {k: bool(np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32))) for k in ("values", "probs")}
            same[name]["max_abs_diff"] = {k: float(np.abs(a[k] - b[k]).max()) for k in ("values", "probs")}
    result = {"card": gpu, "builds": labels, "reps": args.reps, "steps": args.steps, "profiles": args.profiles,
              "l2": "flushed before every timed and every profiled step", "order": "repeats alternate which tree runs first",
              "outputs_bit_identical": same, "summary": summarize(runs, labels), "runs": runs}
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    for name, row in result["summary"].items():
        o, n = row[labels[0]], row[labels[1]]
        heads = "  ".join(f"{k} {o[k]['mean']:.4f}->{n[k]['mean']:.4f}" for k in row["head_ratio_new_over_old"])
        print(f"{name}: step {o['step_ms']['mean']:.3f} [{o['step_ms']['min']:.3f}, {o['step_ms']['max']:.3f}] -> "
              f"{n['step_ms']['mean']:.3f} [{n['step_ms']['min']:.3f}, {n['step_ms']['max']:.3f}] ms; tower {o['tower_ms']['mean']:.3f} -> "
              f"{n['tower_ms']['mean']:.3f} ms; {heads}; layers above the parent's max: {len(row['tower_layers_slower_than_parent_max'])}; "
              f"outputs identical: {same[name]['values'] and same[name]['probs']}", flush=True)
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
