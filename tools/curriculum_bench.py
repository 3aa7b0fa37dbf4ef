#!/usr/bin/env python
"""Cost of a size curriculum with scenes drawn on the device, next to its parts and to the host route.

A steady-state auto-reset loop like bench.py's: episodes of 50 env-steps at staggered phases, so that every env-step
one masked reset rebuilds the envs whose episode ends (E / 50 of them) and then all envs take one `step_device`.
Three Yaml configurations with one random object and a circular light at the object; 10, 20 and 40 kilobots.

  (a) curriculum  KilobotsVecEnv.from_configurations(configs, E, weights=[1, 1, 1]): every reset draws the env's
                  configuration and scene inside the reset kernel (kb_set_sampler_mix), masks follow on the device
  (b) alone       each configuration as its own batch of E envs (from_configuration, kb_set_sampler)
  (c) host route  the same mix built by from_envs from E YamlKilobotsEnv objects; every step vec.resample(done_host)
                  re-draws the finished envs in Python and reset_done(done, pose, light) copies the poses up

Reports ms per env-step split into reset and step (CUDA events for (a) / (b): one pair around each reset and each
step; host clock with a device synchronise for (c), which synchronises anyway), the sampled-reset kernel time alone
(CUDA events around kb_reset_sampled launches), the GPU name and its power limit.  Prints one JSON line.

    python tools/curriculum_bench.py [--envs 4096] [--steps 200] [--host-steps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gym_kilobots_b200 import scenarios as SC  # noqa: E402
from gym_kilobots_b200.envs import KilobotsVecEnv, YamlKilobotsEnv  # noqa: E402

EP_LEN = 50
SIZES = (10, 20, 40)
CONF = """
!EvalEnv
width: 1.0
height: 1.0
resolution: 600
objects:
  - !ObjectConf {idx: 0, color: null, shape: square, width: .1, height: .1, init: random, symmetry: null}
light: !LightConf {type: circular, init: object, radius: .2}
kilobots: !KilobotsConf {num: %d, mean: light, std: .1}
"""


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


def configs():
    return [yaml.load(CONF % n, Loader=yaml.Loader) for n in SIZES]


def masks(E, device):
    import torch
    ids = torch.arange(E, device=device)
    return [((ids + t) % EP_LEN == 0).to(torch.uint8) for t in range(EP_LEN)]


def device_loop(vec, steps):
    """steady state with sampled resets: (ms reset, ms step, ms sampled-reset kernel) per env-step"""
    import torch
    E = vec.num_envs
    ms = masks(E, vec.batch.device)
    acts = torch.as_tensor(SC.random_actions(vec.scenario, E, 16, seed=5), device=vec.batch.device)
    vec.reset()
    for t in range(EP_LEN):   # untimed: spread the phases
        vec.reset_done(ms[t])
        vec.step_device(acts[t % len(acts)])
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    for t in range(steps):
        ev[t][0].record()
        vec.reset_done(ms[t % EP_LEN])
        ev[t][1].record()
        vec.step_device(acts[t % len(acts)])
        ev[t][2].record()
    ev[-1][2].synchronize()
    reset = sum(e[0].elapsed_time(e[1]) for e in ev) / steps
    step = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
    # the sampled-reset launches alone (the same masks, no step in between)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for t in range(steps):
        vec.batch.reset_sampled(ms[t % EP_LEN])
    k1.record()
    k1.synchronize()
    return reset, step, k0.elapsed_time(k1) / steps


def host_loop(vec, steps):
    """the same loop through resample(done_host) + reset_done(done, pose, light): host clock, synchronised"""
    import torch
    E = vec.num_envs
    ms = masks(E, vec.batch.device)
    ms_host = [m.cpu().numpy().astype(bool) for m in ms]
    acts = torch.as_tensor(SC.random_actions(vec.scenario, E, 16, seed=5), device=vec.batch.device)
    vec.reset()
    for t in range(EP_LEN):
        pose, light = vec.resample(ms_host[t])
        vec.reset_done(ms[t], pose, light)
        vec.step_device(acts[t % len(acts)])
    torch.cuda.synchronize()
    reset = step = 0.0
    for t in range(steps):
        t0 = time.perf_counter()
        pose, light = vec.resample(ms_host[t % EP_LEN])
        vec.reset_done(ms[t % EP_LEN], pose, light)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        vec.step_device(acts[t % len(acts)])
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        reset += t1 - t0
        step += t2 - t1
    return reset * 1e3 / steps, step * 1e3 / steps


def row(reset, step, kernel=None, vec=None):
    out = {"ms_per_env_step": round(reset + step, 4), "reset_ms": round(reset, 4), "step_ms": round(step, 4)}
    if kernel is not None:
        out["sampled_reset_kernel_ms"] = round(kernel, 4)
    if vec is not None:
        out["lanes_per_env"] = vec.batch.launch_config()["lanes_per_env"]
        out["envs_with_status_bits"] = int(np.count_nonzero(vec.batch.get_status()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=200, help="timed env-steps of (a) and (b)")
    ap.add_argument("--host-steps", type=int, default=20, help="timed env-steps of (c)")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    E = args.envs
    confs = configs()
    out = {"envs": E, "episode_len_env_steps": EP_LEN, "resets_per_env_step": E / EP_LEN, "kilobots": list(SIZES),
           "objects": 1, "steps": args.steps, "host_steps": args.host_steps}

    vec = KilobotsVecEnv.from_configurations(confs, E, weights=[1.0, 1.0, 1.0], seed=args.seed, allow_status_flags=True)
    out["a_curriculum"] = row(*device_loop(vec, args.steps), vec=vec)
    vec.close()

    alone, weighted = {}, 0.0
    for n, conf in zip(SIZES, confs):
        v = KilobotsVecEnv.from_configuration(conf, E, seed=args.seed, allow_status_flags=True)
        r = device_loop(v, args.steps)
        alone[str(n)] = row(*r, vec=v)
        weighted += (r[0] + r[1]) / len(SIZES)
        v.close()
    out["b_alone"] = alone
    out["b_alone_equal_weight_mean_ms_per_env_step"] = round(weighted, 4)

    np.random.seed(args.seed)
    envs = [YamlKilobotsEnv(configuration=confs[e % len(confs)]) for e in range(E)]
    vec = KilobotsVecEnv.from_envs(envs, allow_status_flags=True)
    out["c_host_route"] = row(*host_loop(vec, args.host_steps), vec=vec)
    vec.close()

    name, power = gpu_info()
    out["gpu"], out["power_limit_w"] = name, power
    print(json.dumps(out))


if __name__ == "__main__":
    main()
