#!/usr/bin/env python
"""Cost of the actuation model (include/kb_b200.h kb_set_actuation): the env-step with the model off and on.

For each workload two handles of the same scenario are stepped alternately for --rounds rounds: one without a model
(the step kernel as it always was) and one with every part of the model switched on (gains, drift, dead kilobots and
per-sub-step noise on speed and turn rate).  Each round times --steps env-steps of each handle, one CUDA event pair per
launch, with the L2 overwritten (a 256 MB buffer written) before every timed step.  Prints the median ms per env-step
of each variant, its spread over the rounds (min..max of the round medians), the ratio on / off, which kernels ran and
the GPU's name and power limit, then one JSON line.

    python tools/actuation_bench.py [--rounds 5] [--steps 10] [--workloads c2,c5,c3,c4]
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
from gym_kilobots_b200.scene import ActuationSpec  # noqa: E402

WORKLOADS = {"c2": lambda: SC.c2_quad_assembly(4096), "c5": lambda: SC.c5_small(1 << 20),
             "c3": lambda: SC.c3_shapes(8192), "c4": lambda: SC.c4_swarm(256)}
MODEL = ActuationSpec(seed=1, gain_v_lo=0.8, gain_v_hi=1.2, gain_w_lo=0.8, gain_w_hi=1.2, drift_w=0.05, noise_v=0.1,
                      noise_w=0.1, p_dead=0.02)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default="c2,c5,c3,c4")
    args = ap.parse_args()
    import torch
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")   # 256 MB: twice the L2
    name, power = gpu_info()
    result = {"gpu": name, "power_limit_w": power, "workloads": {}}
    for wl in args.workloads.split(","):
        sc = WORKLOADS[wl]()
        nbs = {}
        for k in ("off", "on"):
            nb = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
            if k == "on":
                nb.set_actuation(MODEL)
            nb.reset(sc.body_pose, sc.light_state)
            nbs[k] = nb
        cfgs = {k: nb.launch_config() for k, nb in nbs.items()}
        assert cfgs["on"]["actuation"] and not cfgs["off"]["actuation"]
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
        row["on_over_off"] = row["on"]["median_ms"] / row["off"]["median_ms"]
        row["envs"] = sc.num_envs
        row["lanes_per_env"] = cfgs["off"]["lanes_per_env"]
        row["specialised"] = {k: c["specialised"] for k, c in cfgs.items()}
        row["jit_reason_on"] = cfgs["on"]["jit_reason"]
        result["workloads"][wl] = row
        print("%-3s %7d envs  <%3d>  off %.4f ms (%.4f..%.4f)  on %.4f ms (%.4f..%.4f)  on/off %.3f  specialised %s"
              % (wl, sc.num_envs, row["lanes_per_env"], row["off"]["median_ms"], row["off"]["min_ms"], row["off"]["max_ms"],
                 row["on"]["median_ms"], row["on"]["min_ms"], row["on"]["max_ms"], row["on_over_off"], row["specialised"]),
              flush=True)
        del nbs
    print("GPU: %s, power limit %s W" % (name, power))
    print(json.dumps(result))


if __name__ == "__main__":
    main()
