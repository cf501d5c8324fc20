"""Development probe (GPU): the heuristic labelers over the 48-scene default job of bench.py (c3 workload), scene by
scene through gen_pseudo_label_box2mask / gen_pseudo_label against one gen_pseudo_labels_heuristic_batch call per
pass of 16 scenes, for the methods box2mask and dist.  CUDA events around every pass, one warm-up job per arm, the
two arms alternate over the repetitions; the labels of both arms must be identical.  Prints one JSON line with the
card's name and power limit.

    python tests/heuristic_probe.py [--reps 5] [--scenes 16] [--total-scenes 48]
"""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import make_input, scene_ids  # noqa: E402
from gapro_b200.gen_ps import to_scene_inputs  # noqa: E402
from gapro_b200.gen_ps_utils import (gen_pseudo_label, gen_pseudo_label_box2mask,  # noqa: E402
                                     gen_pseudo_labels_heuristic_batch)


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), f"--query-gpu={q}",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm = [x.strip() for x in out.split(",")]
    except (OSError, ValueError, subprocess.SubprocessError):
        name, power, sm = torch.cuda.get_device_name(), None, None
    return {"name": name, "power_limit": power, "sm_max_clock": sm}


def per_scene(scenes, method):
    out = []
    for s in scenes:
        args = (s.coords_float, s.spp, s.instance_cls, s.instance_box, s.instance_box_volume)
        out.append(gen_pseudo_label_box2mask(*args) if method == "box2mask" else
                   gen_pseudo_label(*args, heuristic_rule=method))
    return out


def batched(scenes, method):
    return gen_pseudo_labels_heuristic_batch(scenes, method=method, instance_classes=18, dataset_name="scannetv2")


def run_job(fn, passes, method):
    """The whole job pass by pass; returns (ms per pass, labels of every scene)."""
    ms, labels = [], []
    for scenes in passes:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        labels += fn(scenes, method)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms, labels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scenes", type=int, default=16, help="scenes per pass")
    ap.add_argument("--total-scenes", type=int, default=48)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "heuristic_probe needs a CUDA device"
    dev = torch.device("cuda:0")
    ids = scene_ids(SimpleNamespace(mode="strong", total_scenes=args.total_scenes, scenes=args.scenes), 1)
    scenes = [to_scene_inputs(make_input(i, "c3"), dev) for i in ids]
    passes = [scenes[i:i + args.scenes] for i in range(0, len(scenes), args.scenes)]
    torch.cuda.synchronize()
    result = {"probe": "heuristic labelers, per-scene calls vs one batched call per pass",
              "workload": "c3 (bench.py default job)", "scenes": len(scenes), "scenes_per_pass": args.scenes,
              "points": int(sum(s.coords_float.shape[0] for s in scenes)), "reps": args.reps,
              "card": card(), "methods": {}}
    for method in ("box2mask", "dist"):
        arms = {"per_scene": per_scene, "batched": batched}
        labels = {}
        for name, fn in arms.items():              # warm-up: every shape of the timed window
            labels[name] = run_job(fn, passes, method)[1]
        times = {name: [] for name in arms}
        for _ in range(args.reps):
            for name, fn in arms.items():
                ms, _ = run_job(fn, passes, method)
                times[name].append(sum(ms))
        same = all(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
                   for a, b in zip(labels["per_scene"], labels["batched"]))
        med = {name: float(np.median(t)) for name, t in times.items()}
        result["methods"][method] = {
            "identical": bool(same),
            "job_ms_median": med, "job_ms_all": {k: [round(x, 3) for x in v] for k, v in times.items()},
            "scenes_per_s": {k: len(scenes) / (v / 1e3) for k, v in med.items()},
            "speedup_batched": med["per_scene"] / med["batched"],
        }
    print(json.dumps(result))
    if not all(m["identical"] for m in result["methods"].values()):
        sys.exit("per-scene and batched labels differ")


if __name__ == "__main__":
    main()
