#!/usr/bin/env python
"""Throughput of a batch whose envs differ in size, next to the homogeneous batches it is made of.

One batch of 2048 C2' envs (QuadAssembly: 4 quads, 15 separated phototaxis kilobots) plus 2048 C3-like envs (50
kilobots, one L-form / triangle / circle object) -- padded to 4 objects + 50 kilobots, so every env runs on 32-lane
groups -- against the two homogeneous batches (C2' alone: 8-lane groups; C3-like alone: 32-lane groups) stepped back
to back.  Light actions, device-resident path (kb_step), CUDA events around `--steps` env-steps after `--warmup`.
Prints one JSON line with kilobot-steps/s of each, the GPU name and its power limit.

    python tools/mixed_batch_bench.py [--envs 2048] [--steps 20] [--warmup 5] [--repeats 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gym_kilobots_b200 import _native as native  # noqa: E402
from gym_kilobots_b200 import scenarios as SC  # noqa: E402


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:
        power = None
    return name, power


def timed(nb, acts, steps, warmup):
    """seconds per env-step (device events around `steps` env-steps)"""
    import torch
    for t in range(warmup):
        nb.step_device(acts[t % len(acts)])
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for t in range(steps):
        nb.step_device(acts[t % len(acts)])
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / 1e3 / steps


def build(scenario):
    import torch
    nb = native.NativeBatch(scenario.scenes, scenario.num_envs, scenario.env_scene, scenario.max_contacts)
    nb.reset(scenario.body_pose, scenario.light_state)
    acts = torch.as_tensor(SC.random_actions(2, scenario.num_envs, 8, seed=5), device=nb.device)
    return nb, acts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=2048, help="envs of each size")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    E = args.envs
    c2 = SC.c2_quad_assembly(E, seed=0, degenerate=False)
    c3 = SC.c3_shapes(E, seed=0)
    specs = c2.scenes + c3.scenes
    es = np.concatenate([np.zeros(E, np.int32), 1 + c3.env_scene]).astype(np.int32)
    poses = list(c2.body_pose) + list(c3.body_pose)
    mixed = SC.Scenario("C2'+C3", specs, es, SC.stack_poses(specs, es, poses),
                        np.concatenate([c2.light_state, c3.light_state]), max(c2.max_contacts, c3.max_contacts))
    kb = {"mixed": E * (15 + 50), "C2'": E * 15, "C3": E * 50}
    batches = {"mixed": build(mixed), "C2'": build(c2), "C3": build(c3)}
    times = {k: [] for k in batches}
    for _ in range(args.repeats):   # alternate the batches: other work on the host shares the GPU
        for k, (nb, acts) in batches.items():
            times[k].append(timed(nb, acts, args.steps, args.warmup))
    best = {k: min(v) for k, v in times.items()}
    status = {k: int(np.count_nonzero(nb.get_status())) for k, (nb, _) in batches.items()}
    name, power = gpu_info()
    homog = best["C2'"] + best["C3"]
    out = {
        "gpu": name, "power_limit_w": power, "envs_per_size": E, "steps": args.steps, "repeats": args.repeats,
        "lanes_per_env": {k: nb.launch_config()["lanes_per_env"] for k, (nb, _) in batches.items()},
        "ms_per_env_step": {k: round(v * 1e3, 4) for k, v in best.items()},
        "kilobot_steps_per_s": {k: kb[k] / v for k, v in best.items()},
        "homogeneous_back_to_back": {"ms_per_env_step": round(homog * 1e3, 4),
                                     "kilobot_steps_per_s": kb["mixed"] / homog},
        "mixed_over_back_to_back_time": best["mixed"] / homog,
        "envs_with_status_bits": status,
    }
    print(json.dumps(out))


if __name__ == "__main__":
    main()
