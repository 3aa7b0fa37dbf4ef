#!/usr/bin/env python
"""bench.py -- throughput of the batched KilobotsEnv.step hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c2p|c3|c5|c1]
                    [--dump-outputs DIR]

A "step" is one `KilobotsEnv.step` (10 physics sub-steps of 0.1 s, gym_kilobots/envs/kilobots_env.py:161-215)
for EVERY environment of the batch.  Default workload (BASELINE.json configs[1]): 4096 envs x 15
PhototaxisKilobots + 4 CornerQuads + circular gradient light (QuadAssemblyKilobotsEnv) per GPU.
Weak scaling: every rank owns its own 4096 environments; no data-path collective (NCCL only
all-reduces the timing and the episode statistics).

One JSON line on stdout (rank 0).  `value` = kilobot-steps/s with all inputs resident in HBM,
`e2e` = the same metric through KilobotsVecEnv.step with HOST numpy buffers (pinned staging,
H2D + D2H inside the timed region).  `--impl reference` times the CPU oracle (oracle/, a Box2D
restatement -- pybox2d itself is not installable here) on all host cores on a bounded sample.

Scenes and actions are seeded, so the same arguments give the same inputs on every run.  `--dump-outputs DIR` writes
what the last of the K timed steps returned (observations, reward, done, status) as DIR/<name>.npy, so that two
builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from gym_kilobots_b200 import _abi as abi  # noqa: E402
from gym_kilobots_b200 import scenarios as SC  # noqa: E402

METRIC = "kilobot-steps/s"
UNIT = "kilobot-steps/s"


def build_scenario(name, num_envs, env_offset=0):
    if name == "c2":
        return SC.c2_quad_assembly(num_envs, seed=0, env_offset=env_offset, degenerate=True)
    if name == "c2p":
        return SC.c2_quad_assembly(num_envs, seed=0, env_offset=env_offset, degenerate=False)
    if name == "c3":
        return SC.c3_shapes(num_envs, seed=0, env_offset=env_offset)
    if name == "c4":
        return SC.c4_swarm(num_envs, seed=0, env_offset=env_offset)
    if name == "c5":
        return SC.c5_small(num_envs, seed=0, env_offset=env_offset)
    if name == "c1":
        return SC.c1_single_env(num_envs, seed=0, env_offset=env_offset)
    raise SystemExit("unknown workload %s" % name)


# envs per GPU; C5 is BASELINE.json's "throughput sweep 1M envs x 4 kilobots at 1/2/4/8 GPUs": 2^20 envs in TOTAL,
# split over the ranks (strong scaling); every other workload keeps its per-GPU batch (weak scaling)
DEFAULT_ENVS = {"c2": 4096, "c2p": 4096, "c3": 8192, "c4": 256, "c5": 1 << 20, "c1": 1}
TOTAL_FIXED = {"c5"}


def envs_per_gpu(workload, world, override=0):
    if override:
        return override
    return DEFAULT_ENVS[workload] // world if workload in TOTAL_FIXED else DEFAULT_ENVS[workload]


def workload_desc(workload, E, world):
    return {
        "c2": "C2 QuadAssemblyKilobotsEnv: %d envs x (15 PhototaxisKilobot + 4 CornerQuad 0.15m + CircularGradientLight r=0.2) per GPU, reference spawn" % E,
        "c2p": "C2' QuadAssembly scene, non-degenerate spawn, %d envs x 15 kilobots per GPU" % E,
        "c3": "C3: %d envs x (50 PhototaxisKilobot + LForm/Triangle/Circle object) per GPU" % E,
        "c4": "C4 large-swarm stress: %d envs x 1024 PhototaxisKilobot (32x32 lattice, light r=0.8, zero action) per GPU" % E,
        "c5": "C5 throughput sweep: %d envs x (4 PhototaxisKilobot + Quad) in total = %d per GPU, N(L0, 0.03^2) rejection-separated spawn" % (E * world, E),
        "c1": "C1 single env: 10 PhototaxisKilobot + Quad + CircularGradientLight",
    }[workload]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def algorithmic_bytes_per_env_step(N, M, P, C, A, L):
    """SURVEY.md 8(d): minimal persistent state read+written once per env-step, action in, obs out."""
    return 2.0 * (32 * (N + M) + 16 * N + 16 * P + 40 * C + 32) + 4 * A + (12 * (N + M) + 4 * L + 8)


def algorithmic_flops_per_env_step(N, M, pair_tests, points, pos_iters_per_island_step, substeps=10):
    """SURVEY.md 8(d) F_alg, per env-step (sums over the sub-steps are passed in as per-substep means)."""
    return substeps * (76 * N + 60 * M + 12 * pair_tests + points * (102 + 620 + 80 * pos_iters_per_island_step))


def measured_traffic(workload, envs):
    """dram__bytes_read.sum + dram__bytes_write.sum per kb_step launch, a CITATION of the committed `ncu --set full`
    capture of this workload (profiles/traffic.json, written from the .ncu-rep by tools/ncu_summary.py) -- not
    measured in this run.  Returned only if the capture was taken at the same number of envs."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            t = json.load(f).get(workload)
    except Exception:
        return None
    if isinstance(t, dict) and t.get("envs") == envs:
        return {"bytes": t["bytes"], "source": "profiles/traffic.json (%s; cited, not measured in this run)" % t.get("capture", "ncu --set full")}
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, outputs):
    """Write the outputs of one env-step as out_dir/<name>.npy (float32, or float64 where the step returns float64).
    When they exceed DUMP_MAX_BYTES, the same fixed, seeded sample of envs is kept from every array."""
    outputs = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in outputs.items()}
    E = len(outputs["reward"])
    per_env = sum(v.nbytes for v in outputs.values()) // E
    keep = (DUMP_MAX_BYTES - 4096 * len(outputs)) // per_env   # 4 KB per file for the .npy header
    if keep < E:
        envs = np.sort(np.random.default_rng(0).choice(E, keep, replace=False))
        outputs = {k: v[envs] for k, v in outputs.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in outputs.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def time_oracle(workload, sample_envs, steps, warmup, threads, dump_dir=None):
    """CPU oracle on the host cores: kilobot-steps/s on a bounded sample of the workload.  With dump_dir, the outputs
    of the last timed step are written there (dump_outputs)."""
    from oracle import kbo
    kbo.build()
    sc = build_scenario(workload, sample_envs)
    ob = kbo.OracleBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts, threads=threads)
    ob.reset(sc.body_pose, sc.light_state)
    acts = SC.random_actions(sc, sc.num_envs, steps + warmup)
    for t in range(warmup):
        ob.step(acts[t])
    t0 = time.perf_counter()
    for t in range(warmup, warmup + steps):
        out = ob.step(acts[t])
    dt = time.perf_counter() - t0
    if dump_dir is not None:
        dump_outputs(dump_dir, out)
    N = sc.scenes[0].num_kilobots
    return sc.num_envs * steps * N / dt, dt / steps, N


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    E = envs_per_gpu(args.workload, world, args.envs)
    sample = min(E, args.ref_envs)
    value, sec_per_step, N = time_oracle(args.workload, sample, args.steps, args.warmup, threads, args.dump_outputs)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_desc(args.workload, E, world), "sample_envs": sample,
                   "same_config": sample == E,
                   "note": "CPU arm: the first %d envs of the workload (same scene, spawn and action draws), "
                           "throughput-normalised; it uses the SAME host cores at every --gpus N" % sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d envs of the workload x %d env-steps, oracle/libkbo.so (Box2D restatement; "
                                   "pybox2d is not installable offline, profiles/box2d_install_r02.log), one thread "
                                   "per core" % (sample, args.steps)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


class Rig:
    """Process-wide plumbing of one bench run: rank / device / NCCL group / L2-flush buffer."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)  # > 126 MB L2

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return vals
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return tuple(float(x) for x in t)

    def gather(self, val):
        if self.world == 1:
            return [float(val)]
        t = self.torch.tensor([val], dtype=self.torch.float64, device=self.dev)
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(x[0]) for x in out]

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def measure(rig, workload, E, steps, warmup, cpu_envs, steady_steps=0, sampler=None, dump_dir=None):
    """One workload on this rank's GPU: device-resident leg (CUDA events per step, L2 flushed between steps), the
    end-to-end leg through KilobotsVecEnv.step with host buffers, optionally a steady-state leg with staggered
    auto-resets, and (rank 0) the roofline / cpu_baseline objects.  Returns the result dict on rank 0, else None.
    With dump_dir, rank 0 writes what the last timed step of the device-resident leg returned (dump_outputs)."""
    torch = rig.torch
    from gym_kilobots_b200.envs import KilobotsVecEnv
    dev, world, rank = rig.dev, rig.world, rig.rank
    sc = build_scenario(workload, E, env_offset=rank * E)
    env = KilobotsVecEnv(sc, device=rig.local_rank, allow_status_flags=True)   # flags are counted and reported below
    env.reset()
    b = env.batch
    total = steps + warmup
    acts_h = torch.from_numpy(SC.random_actions(sc, E, total, seed=1 + rank)).pin_memory().numpy()   # pinned host inputs
    acts_d = torch.as_tensor(acts_h, dtype=torch.float64, device=dev)

    # ---------------- device-resident leg
    for t in range(warmup):
        env.step_device(acts_d[t])
    cnt0 = b.counters().astype(np.float64).sum(0)
    rig.barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    wall0 = time.perf_counter()
    for i in range(steps):
        rig.flush.zero_()  # L2 flush between timed iterations (not inside the event pair)
        starts[i].record()
        obs, rew, done, info = env.step_device(acts_d[warmup + i])
        ends[i].record()
    rig.barrier()
    wall = time.perf_counter() - wall0
    if dump_dir is not None and rank == 0:
        # the step's output tensors are re-used by every later step: copy them out before the next leg
        dump_outputs(dump_dir, {"kilobots": obs["kilobots"].cpu().numpy(), "objects": obs["objects"].cpu().numpy(),
                                "light": obs["light"].cpu().numpy(), "reward": rew.cpu().numpy(),
                                "done": done.cpu().numpy(), "status": info["status"].cpu().numpy()})
    step_ms = np.array([s.elapsed_time(e) for s, e in zip(starts, ends)])
    my_elapsed = float(step_ms.sum()) * 1e-3
    cnt1 = b.counters().astype(np.float64).sum(0)
    # episode statistics of the whole job: device-side reduction + NCCL all-reduce (the only collective of the path)
    job_stats = env.all_reduce_episode_stats()

    # ---------------- end-to-end leg: public API, host buffers.  Same episode and the same step indices as the
    # device-resident leg (reset, W untimed steps through the host path, then the K timed ones), so that the two
    # numbers differ by the host<->device path only
    env.reset()
    for t in range(warmup):
        env.step(acts_h[t])
    rig.barrier()
    e0 = time.perf_counter()
    for i in range(steps):
        obs, rew, done, info = env.step(acts_h[warmup + i])
    torch.cuda.synchronize(dev)
    my_e2e = time.perf_counter() - e0
    h2d, d2h = env.host_io_bytes()

    # ---------------- steady-state leg: hundreds of env-steps with auto-reset.  Episodes of `ep_len` env-steps with
    # staggered phases: every step the envs with (env id + t) % ep_len == 0 are rebuilt by a masked kb_reset launch
    # (fresh bodies + settle step) before the step -- all episode phases are present at once, as in a long rollout
    steady = None
    if steady_steps > 0:
        ep_len = 50
        pose_d = torch.as_tensor(sc.body_pose, dtype=torch.float64, device=dev)
        light_d = torch.as_tensor(sc.light_state, dtype=torch.float64, device=dev)
        ids = torch.arange(E, device=dev)
        masks = [((ids + t) % ep_len == 0).to(torch.uint8) for t in range(ep_len)]
        env.reset()
        for t in range(ep_len):   # untimed: spread the phases
            env.batch.reset(pose_d, light_d, None, masks[t % ep_len])
            env.step_device(acts_d[t % total])
        rig.barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for t in range(steady_steps):
            env.batch.reset(pose_d, light_d, None, masks[t % ep_len])
            env.step_device(acts_d[t % total])
        s1.record()
        rig.barrier()
        (steady_s,) = rig.max_over_ranks(s0.elapsed_time(s1) * 1e-3)
        flagged = int((b.get_status() != 0).sum())
        steady = {"steps": steady_steps, "episode_len_env_steps": ep_len, "resets_per_step": E / ep_len,
                  "ms_per_step": steady_s / steady_steps * 1e3, "value": E * world * steady_steps * b.N / steady_s,
                  "unit": UNIT, "launches_per_step": 2, "envs_with_status_flags_rank0": flagged,
                  "note": "one masked kb_reset launch + one kb_step launch per step, timed as one CUDA-event pair around "
                          "all steps (no L2 flush inside: the %.1f MB of state stay L2-resident, as in a real rollout)"
                          % (E * b.state_bytes_per_env / 1e6)}
    if sampler is not None:
        # keep the GPU under the same load (untimed) until the clock sampler has seen it for at least ~0.6 s
        t_load = time.perf_counter()
        while time.perf_counter() - t_load < 0.6:
            for _ in range(20):
                env.step_device(acts_d[warmup])
            torch.cuda.synchronize(dev)

    elapsed, e2e_elapsed = rig.max_over_ranks(my_elapsed, my_e2e)
    per_rank_ms = rig.gather(my_elapsed / steps * 1e3)
    per_rank_e2e_ms = rig.gather(my_e2e / steps * 1e3)
    N, M = b.N, b.M
    env_steps_total = float(E * world * steps)
    env_steps_s = env_steps_total / elapsed
    out = None
    if rank == 0:
        d = cnt1 - cnt0
        sub = max(d[abi.COUNTER_NAMES.index("substeps")], 1.0)
        C_mean = d[abi.COUNTER_NAMES.index("contacts")] / sub
        pts = d[abi.COUNTER_NAMES.index("points")] / sub
        lvls = d[abi.COUNTER_NAMES.index("levels")] / sub
        isl = max(d[abi.COUNTER_NAMES.index("islands")] / sub, 1e-9)
        pit = d[abi.COUNTER_NAMES.index("pos_iters")] / sub
        ptests = d[abi.COUNTER_NAMES.index("pair_tests")] / sub
        peaks, peak_src = measured_peaks()
        bytes_env = algorithmic_bytes_per_env_step(N, M, b.P, C_mean, b.A, b.L)
        launch_s = float(step_ms.mean()) * 1e-3
        achieved = bytes_env * E / launch_s / 1e9
        flops_env = algorithmic_flops_per_env_step(N, M, ptests, pts, pit / isl)
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
        lc = b.launch_config()
        traffic = measured_traffic(workload, E)
        t_hbm = bytes_env * E / (peaks["hbm_gbs"] * 1e9)
        t_fp32 = flops_env * E / (fp32_peak * 1e12)
        roof = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic["bytes"] if traffic else None,
                "traffic_source": (traffic["source"] if traffic else None), "peak_source": peak_src,
                "kernel": lc.pop("kernel"), "launch": lc,
                "algorithmic_bytes_per_env_step": bytes_env, "launch_ms": launch_s * 1e3,
                "note": "state I/O is a few KB per env-step against tens of thousands of warp-instructions of "
                        "sequential-impulse solving: the kernel is bound by dependent-issue latency, not by HBM "
                        "(DESIGN.md section 5); frac_of_max_roofline = max(T_hbm, T_fp32) / T_measured (SURVEY 8d)",
                "frac_of_max_roofline": max(t_hbm, t_fp32) / launch_s,
                "fp32": {"algorithmic_flops_per_env_step": flops_env,
                         "achieved_tflops": flops_env * E / launch_s / 1e12, "peak_tflops": fp32_peak,
                         "frac": flops_env * E / launch_s / 1e12 / fp32_peak,
                         "note": "non-tensor FP32 issue roofline (SURVEY 8d); no dense contraction on this path"}}
        cpu_n = min(E, cpu_envs)
        cpu_steps = max(2, steps)
        cpu_val, cpu_sec, _ = time_oracle(workload, cpu_n, cpu_steps, 1, 1)
        out = {
            "workload": workload, "value": env_steps_s * N, "unit": UNIT, "ms_per_step": float(step_ms.mean()),
            "scaling": "strong" if workload in TOTAL_FIXED else "weak",
            "config": {"workload": workload_desc(workload, E, world), "envs_per_gpu": E, "envs_total": E * world,
                       "kilobots_per_env": N, "objects_per_env": M,
                       "substeps_per_step": sc.scenes[0].steps_per_action,
                       "l2": "256 MiB device buffer zeroed between timed steps (L2 flush, outside the event pairs)",
                       "parallelism": "env-sharded x%d" % world},
            "env_steps_per_s": env_steps_s, "substeps_per_s": env_steps_s * sc.scenes[0].steps_per_action,
            "wall_s_timed_region": wall, "per_rank_ms": per_rank_ms, "per_rank_e2e_ms": per_rank_e2e_ms,
            "e2e": {"value": env_steps_total * N / e2e_elapsed, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h),
                    "api": "KilobotsVecEnv.step(pinned numpy actions) -> kb_step_host (H2D + kernel + D2H into pinned numpy; "
                           "large batches are pipelined in chunks on two side streams)"},
            "gpu_launches": int(steps),
            "roofline": roof,
            "cpu_baseline": {"value": cpu_val, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": "%d envs of the workload x %d env-steps (%.1f s), oracle/libkbo.so single thread (Box2D "
                                       "restatement; pybox2d not installable offline)" % (cpu_n, cpu_steps, cpu_sec * cpu_steps)},
            "episode_stats_all_reduced": job_stats,
            "sim_stats": {"contacts_per_substep": C_mean, "manifold_points_per_substep": pts,
                          "gs_levels_per_substep": lvls, "islands_per_substep": isl,
                          "pos_iters_per_island": pit / isl, "toi_events": d[abi.COUNTER_NAMES.index("toi_events")],
                          "envs_with_status_flags": job_stats["envs_with_status"]},
        }
        if steady is not None:
            out["steady_state"] = steady
    env.close()
    del env, acts_d
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    rig = Rig()
    world = rig.world
    # clocks / throttle reasons are sampled from the first warm-up step of the headline workload to the end of its
    # load tail (the timed region of a default run is only ~25 ms, shorter than nvidia-smi's sampling period)
    sampler = ClockSampler(rig.local_rank)
    sampler.start()
    E = envs_per_gpu(args.workload, world, args.envs)
    head = measure(rig, args.workload, E, args.steps, args.warmup, args.cpu_envs, steady_steps=args.steady_steps,
                   sampler=sampler, dump_dir=args.dump_outputs)
    clocks = sampler.stop()
    sweep = []
    if args.sweep:
        for wl in args.sweep.split(","):
            if wl == args.workload:
                continue
            r = measure(rig, wl, envs_per_gpu(wl, world), max(5, args.steps // 2), max(3, args.warmup // 2),
                        min(args.cpu_envs, {"c4": 8, "c3": 128, "c5": 4096}.get(wl, 256)))
            if r is not None:
                sweep.append(r)
    if rig.rank == 0:
        out = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
               "scaling": head["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "clocks": clocks}
        out.update({k: v for k, v in head.items() if k not in ("value", "unit", "ms_per_step", "scaling", "workload")})
        if sweep:
            out["sweep"] = sweep
        print(json.dumps(out))
    rig.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(DEFAULT_ENVS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the workload's)")
    ap.add_argument("--cpu-envs", type=int, default=2048, help="sample size of the cpu_baseline leg (envs, one thread)")
    ap.add_argument("--ref-envs", type=int, default=4096, help="sample size of --impl reference (envs, all host cores)")
    ap.add_argument("--steady-steps", type=int, default=200,
                    help="env-steps of the steady-state leg with staggered auto-resets (0 = skip)")
    ap.add_argument("--sweep", default="c5,c3,c4",
                    help="extra workloads measured after the headline one and reported under 'sweep' ('' = none)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline workload returned (rank 0's envs) as "
                         "DIR/<name>.npy; a fixed sample of the envs if that exceeds 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
