#!/usr/bin/env python
"""Generic vs specialised step kernel (csrc/kb_jit.h) on the same scenario in one process.

For each workload a KB_JIT=0 handle (kb_step_kernel<LPE>, layout from the kernel parameters) and a KB_JIT=1 handle
(compiled at kb_create for the batch's layout) are stepped alternately for --rounds rounds; each round times --steps
env-steps of each handle, one CUDA event pair per launch, with the L2 overwritten (a 256 MB buffer written) before
every timed step.  Prints the median ms per env-step of each kernel, its spread over the rounds (min..max of the
round medians), the speed-up, the compile times and the GPU's name and power limit, then one JSON line.

    python tools/jit_bench.py [--rounds 5] [--steps 10] [--workloads c2,c3,c5]
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

WORKLOADS = {"c2": lambda: SC.c2_quad_assembly(4096), "c3": lambda: SC.c3_shapes(8192), "c5": lambda: SC.c5_small(1 << 20)}


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


def make(sc, jit):
    os.environ["KB_JIT"] = jit
    try:
        nb = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    finally:
        del os.environ["KB_JIT"]
    nb.reset(sc.body_pose, sc.light_state)
    return nb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default="c2,c3,c5")
    args = ap.parse_args()
    import torch
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")   # 256 MB: twice the L2
    name, power = gpu_info()
    result = {"gpu": name, "power_limit_w": power, "workloads": {}}
    for wl in args.workloads.split(","):
        sc = WORKLOADS[wl]()
        nbs = {"generic": make(sc, "0"), "specialised": make(sc, "1")}
        cfg = nbs["specialised"].launch_config()
        assert cfg["specialised"], cfg["jit_reason"]
        acts = torch.as_tensor(SC.random_actions(sc, sc.num_envs, 8, seed=5), device="cuda")
        for nb in nbs.values():
            for t in range(args.warmup):
                nb.step_device(acts[t % len(acts)])
        times = {k: [] for k in nbs}
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for r in range(args.rounds):
            for k, nb in nbs.items():
                for t in range(args.steps):
                    flush.fill_(float(t))
                    ev[t][0].record()
                    nb.step_device(acts[t % len(acts)])
                    ev[t][1].record()
                torch.cuda.synchronize()
                times[k].append(float(np.median([a.elapsed_time(b) for a, b in ev])))
        row = {k: {"median_ms": float(np.median(v)), "min_ms": min(v), "max_ms": max(v)} for k, v in times.items()}
        row["speedup"] = row["generic"]["median_ms"] / row["specialised"]["median_ms"]
        row["envs"] = sc.num_envs
        row["lanes_per_env"] = cfg["lanes_per_env"]
        row["jit_ms"] = cfg["jit_ms"]
        result["workloads"][wl] = row
        print("%-3s %7d envs  <%2d>  generic %.4f ms (%.4f..%.4f)  specialised %.4f ms (%.4f..%.4f)  x%.3f  compile %.0f ms"
              % (wl, sc.num_envs, cfg["lanes_per_env"], row["generic"]["median_ms"], row["generic"]["min_ms"],
                 row["generic"]["max_ms"], row["specialised"]["median_ms"], row["specialised"]["min_ms"],
                 row["specialised"]["max_ms"], row["speedup"], cfg["jit_ms"]), flush=True)
        del nbs
    print("GPU: %s, power limit %s W" % (name, power))
    print(json.dumps(result))


if __name__ == "__main__":
    main()
