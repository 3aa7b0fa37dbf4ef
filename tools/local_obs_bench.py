#!/usr/bin/env python
"""local_obs_bench.py -- cost of the per-kilobot local observation (kb_local_observation) against the env-step it
follows and against a straightforward PyTorch formulation of its neighbour part.

    python tools/local_obs_bench.py [--reps 30] [--configs c2,c3,c4,c5,mixed] [--out FILE.json]

Batches: the C2 / C3 / C4 / C5 sizes of bench.py and a mixed batch (10 / 40 / 100 kilobots); K = 8 neighbours within
0.1 m (plus the object and light parts where the batch has them).  Per rep, the variants run alternately, each timed by
CUDA events around its own launches, with L2 overwritten (a 256 MB write) before every timed pass:
  local   kb_local_observation
  step    kb_step of the same batch (zero light action)
  torch   the neighbour part in PyTorch on the step's obs tensors: torch.cdist + topk per env, chunked to 1 GiB
The GPU's name and power limit are printed with the numbers (median and min over the reps, milliseconds).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gym_kilobots_b200 import _native  # noqa: E402
from gym_kilobots_b200 import scenarios as SC  # noqa: E402
from gym_kilobots_b200.scene import LocalObsSpec  # noqa: E402

K, RADIUS = 8, 0.1


def _mixed(per):
    sizes = (10, 40, 100)
    homs = [SC.swarm_corner(per, n=n, spread=.05, corner=False, seed=i) for i, n in enumerate(sizes)]
    specs = [h.scenes[0] for h in homs]
    E = 3 * per
    env_scene = (np.arange(E) % 3).astype(np.int32)
    poses = [homs[e % 3].body_pose[e // 3] for e in range(E)]
    light = np.stack([homs[e % 3].light_state[e // 3] for e in range(E)])
    return SC.Scenario("mixed", specs, env_scene, SC.stack_poses(specs, env_scene, poses), light)


CONFIGS = {
    "c2": lambda: SC.c2_quad_assembly(4096),
    "c3": lambda: SC.c3_shapes(8192),
    "c4": lambda: SC.c4_swarm(256),
    "c5": lambda: SC.c5_small(1 << 20),
    "mixed": lambda: _mixed(256),
}


def torch_neighbours(torch, kb, k, radius, chunk_bytes=1 << 30):
    """count + K nearest (x, y, distance, 1) in each kilobot's frame: cdist + topk per env, chunked over the envs."""
    E, N, _ = kb.shape
    out = torch.empty((E, N, 1 + 4 * k), dtype=torch.float32, device=kb.device)
    step = max(1, chunk_bytes // (4 * N * N * 3))
    eye = torch.eye(N, dtype=torch.bool, device=kb.device)
    kk = min(k, max(N - 1, 1))
    for e0 in range(0, E, step):
        x = kb[e0:e0 + step]
        p = x[..., :2]
        d = torch.cdist(p, p)
        d = d.masked_fill(eye | torch.isnan(d), float("inf"))
        hit = d <= radius
        val, idx = torch.topk(d, kk, dim=-1, largest=False)
        q = torch.gather(p.unsqueeze(1).expand(-1, N, -1, -1), 2, idx.unsqueeze(-1).expand(-1, -1, -1, 2)) - p.unsqueeze(2)
        c, s = torch.cos(x[..., 2]).unsqueeze(-1), torch.sin(x[..., 2]).unsqueeze(-1)
        ok = (val <= radius).unsqueeze(-1)
        slot = torch.stack([c * q[..., 0] + s * q[..., 1], -s * q[..., 0] + c * q[..., 1], val, torch.ones_like(val)], -1)
        slot = torch.where(ok, slot, torch.zeros_like(slot))
        o = out[e0:e0 + step]
        o[..., 0] = hit.sum(-1).float()
        o[..., 1:] = 0
        o[..., 1:1 + 4 * kk] = slot.reshape(*slot.shape[:2], 4 * kk)
    return out


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception as e:  # the name from torch below still identifies the card
        name, power = None, "unknown (%s)" % type(e).__name__
    return name, power


def run(name, reps, torch):
    sc = CONFIGS[name]()
    nb = _native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    spec = LocalObsSpec(RADIUS, max_neighbours=K, objects=nb.M > 0, light=nb.L > 0)
    nb.reset(sc.body_pose, sc.light_state)
    act = torch.zeros((nb.E, max(nb.A, 1)), dtype=torch.float64, device=nb.device)[:, :nb.A]
    act = act.contiguous() if nb.A else None
    flush = torch.empty(64 << 20, dtype=torch.float32, device=nb.device)   # 256 MB: more than the 126 MB L2
    variants = {
        "local": lambda: nb.local_observation(spec),
        "step": lambda: nb.step_device(act),
        "torch": lambda: torch_neighbours(torch, nb.obs_kilobots, K, RADIUS),
    }
    for f in variants.values():   # warm-up of every shape in the timed window
        f()
        f()
    torch.cuda.synchronize()
    ev = {k: [] for k in variants}
    for _ in range(reps):
        for k, f in variants.items():
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            ev[k].append((a, b))
    torch.cuda.synchronize()
    ms = {k: np.array([a.elapsed_time(b) for a, b in v]) for k, v in ev.items()}
    res = {"config": name, "envs": nb.E, "kilobots": nb.N, "objects": nb.M, "D": nb.local_observation_dim(spec),
           "kernel": "grid (CTA per env)" if nb.B > 64 else "warp per env"}
    for k, v in ms.items():
        res[k + "_ms_median"] = float(np.median(v))
        res[k + "_ms_min"] = float(v.min())
    res["local_over_step"] = res["local_ms_median"] / res["step_ms_median"]
    res["torch_over_local"] = res["torch_ms_median"] / res["local_ms_median"]
    nb.close()
    del flush
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--configs", default="c2,c3,c4,c5,mixed")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("local_obs_bench.py measures on the GPU: no CUDA device visible")
    name, power = gpu_info()
    head = {"gpu": name or torch.cuda.get_device_name(0), "power_limit": power, "K": K, "radius_m": RADIUS,
            "reps": args.reps, "l2": "overwritten (256 MB) before every timed pass"}
    print(json.dumps(head), flush=True)
    rows = []
    for c in args.configs.split(","):
        r = run(c, args.reps, torch)
        rows.append(r)
        print(json.dumps(r), flush=True)
    print("%-6s %8s %5s %4s  %10s %10s %10s  %9s %9s" % ("config", "envs", "N", "D", "local ms", "step ms", "torch ms",
                                                         "local/step", "torch/local"))
    for r in rows:
        print("%-6s %8d %5d %4d  %10.4f %10.3f %10.3f  %9.4f %9.1f" % (
            r["config"], r["envs"], r["kilobots"], r["D"], r["local_ms_median"], r["step_ms_median"], r["torch_ms_median"],
            r["local_over_step"], r["torch_over_local"]))
    print("GPU: %s, power limit %s" % (head["gpu"], power))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"device": head, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
