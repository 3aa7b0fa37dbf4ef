"""Loader of the CUDA library (csrc/libkb_b200.so) and the batched handle built on it.

PyTorch is plumbing here: it owns device tensors and streams; every byte of simulation work happens
inside hand-written sm_100a kernels reached through the C-ABI of include/kb_b200.h.  There is no
CPU fallback -- if the library is missing or no B200 is visible this module raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _abi as abi

_CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
_LIB_PATH = os.path.join(_CSRC, "libkb_b200.so")
_lib = None
_fn = None


class NativeLibraryError(RuntimeError):
    pass


class KbStatusError(RuntimeError):
    """An env raised a KB_STATUS_* bit: its contact / solver capacity overflowed (pairs or constraints were
    dropped, the physics is no longer the reference's) or a pose became non-finite."""


def describe_status(status):
    status = np.asarray(status)
    bad = np.flatnonzero(status != 0)
    names = ((abi.KB_STATUS_CONTACT_OVERFLOW, "contact-list overflow"), (abi.KB_STATUS_NONFINITE, "non-finite pose"),
             (abi.KB_STATUS_SOLVER_OVERFLOW, "solver-capacity overflow"))
    bits = int(np.bitwise_or.reduce(status[bad])) if len(bad) else 0
    what = ", ".join(n for b, n in names if bits & b)
    return "%d env(s) flagged (%s), first env %d; raise max_contacts (or pass max_contacts=-1 for every proxy pair)" % (
        len(bad), what, int(bad[0]) if len(bad) else -1)


def build(force=False):
    """Compile csrc/kb_b200.cu for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    if force or not os.path.exists(_LIB_PATH):
        subprocess.check_call(["make", "-C", _CSRC, "libkb_b200.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


def load():
    """dlopen the product library; never falls back to anything else."""
    global _lib, _fn
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise NativeLibraryError(
                "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the Kilobots step)" % _LIB_PATH)
        _lib = C.CDLL(_LIB_PATH)
        _fn = abi.bind(_lib, "kb_")
    return _lib, _fn


def exported_symbols():
    return ["kb_" + n for n in list(abi.PROTOTYPES) + list(abi.PRODUCT_ONLY)]


def jit_step_source(scenes, max_contacts=0, compile=False):
    """(source, log, compile_ms) of the specialised step kernel kb_create would build for a lane-group batch of
    `scenes`; with compile=True it is also compiled with NVRTC, and log holds ptxas's resource report.  No GPU needed."""
    load()
    scenes = list(scenes) if isinstance(scenes, (list, tuple)) else [scenes]
    descs = (abi.KbSceneDesc * len(scenes))()
    keep = []
    for i, s in enumerate(scenes):
        descs[i], k = s.to_desc()
        keep.append(k)
    src = C.create_string_buffer(1 << 16)
    log = C.create_string_buffer(1 << 20)
    ms = C.c_double(0.0)
    _check(_fn["jit_step_source"](descs, len(scenes), max_contacts, int(compile), src, len(src), log, len(log),
                                  C.byref(ms)), "kb_jit_step_source")
    return src.value.decode(), log.value.decode(), ms.value


def _check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what, rc, _fn["last_error"]().decode()))


def _hptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class NativeBatch:
    """E environments resident on one B200, stepped by one kernel launch per action."""

    def __init__(self, scenes, num_envs, env_scene=None, max_contacts=0, device=0):
        import torch

        self.torch = torch
        if not torch.cuda.is_available():
            raise NativeLibraryError("no CUDA device visible: the Kilobots step has no CPU fallback")
        load()
        if not isinstance(scenes, (list, tuple)):
            scenes = [scenes]
        self.scenes = list(scenes)
        self.device = torch.device("cuda", device)
        descs = (abi.KbSceneDesc * len(scenes))()
        self._keep = []
        for i, s in enumerate(scenes):
            d, keep = s.to_desc()
            descs[i] = d
            self._keep.append(keep)
        es = None if env_scene is None else np.ascontiguousarray(env_scene, dtype=np.int32)
        h = C.c_void_p()
        _check(_fn["create"](descs, len(scenes), _hptr(es), num_envs, max_contacts, device, C.byref(h)), "kb_create")
        self.h = h
        dims = abi.KbDims()
        _check(_fn["get_dims"](self.h, C.byref(dims)), "kb_get_dims")
        self.E, self.B, self.M, self.N = dims.num_envs, dims.num_bodies, dims.num_objects, dims.num_kilobots
        self.P, self.C, self.L, self.A = dims.num_proxies, dims.max_contacts, dims.light_state_dim, dims.action_dim
        self.state_bytes_per_env = dims.state_bytes_per_env
        dev = self.device
        self.obs_kilobots = torch.zeros((self.E, self.N, 3), dtype=torch.float32, device=dev)
        self.obs_objects = torch.zeros((self.E, self.M, 3), dtype=torch.float32, device=dev)
        self.obs_light = torch.zeros((self.E, self.L), dtype=torch.float64, device=dev)
        self.reward = torch.zeros(self.E, dtype=torch.float32, device=dev)
        self.done = torch.zeros(self.E, dtype=torch.uint8, device=dev)
        self.status = torch.zeros(self.E, dtype=torch.int32, device=dev)

    def close(self):
        if getattr(self, "h", None):
            _fn["destroy"](self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- device-resident API (tensors in, tensors out, asynchronous on the current stream)
    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, x, dtype, shape):
        torch = self.torch
        if x is None:
            return None
        t = torch.as_tensor(x, dtype=dtype)
        if t.device != self.device:
            t = t.to(self.device)
        return t.contiguous().reshape(shape)

    def reset(self, body_pose, light_state=None, kb_velocity=None, mask=None):
        torch = self.torch
        pose = self._dev(body_pose, torch.float64, (self.E, self.B, 3))
        light = self._dev(light_state, torch.float64, (self.E, self.L)) if self.L > 0 else None
        vel = self._dev(kb_velocity, torch.float64, (self.E, self.N, 2))
        m = self._dev(mask, torch.uint8, (self.E,))
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        _check(_fn["reset"](self.h, ptr(m), ptr(pose), ptr(light), ptr(vel), self._stream()), "kb_reset")
        self._keep_reset = (pose, light, vel, m)

    def step_device(self, action=None, mode=None):
        """One env-step for all E envs; returns the (re-used) device output tensors."""
        torch = self.torch
        if action is None:
            if mode is None:
                mode = abi.KB_ACTION_NONE
            act = None
        else:
            if mode is None:
                mode = abi.KB_ACTION_LIGHT
            n = 2 * self.N if mode == abi.KB_ACTION_KILOBOTS else self.A
            act = self._dev(action, torch.float64, (self.E, n))
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else None
        _check(_fn["step"](self.h, p(act), mode, p(self.obs_kilobots), p(self.obs_objects), p(self.obs_light),
                           p(self.reward), p(self.done), p(self.status), self._stream()), "kb_step")
        self._keep_step = act
        return self.obs_kilobots, self.obs_objects, self.obs_light, self.reward, self.done, self.status

    def step(self, action=None, mode=None):
        """numpy-returning convenience wrapper (same dict as the oracle driver)."""
        k, o, l, r, d, s = self.step_device(action, mode)
        self.torch.cuda.synchronize(self.device)
        return {"kilobots": k.cpu().numpy(), "objects": o.cpu().numpy(), "light": l.cpu().numpy(),
                "reward": r.cpu().numpy(), "done": d.cpu().numpy(), "status": s.cpu().numpy()}

    def step_host(self, action, mode, out):
        """kb_step_host: HOST numpy buffers in and out, copies inside the call (end-to-end path)."""
        act = None if action is None else np.ascontiguousarray(action, dtype=np.float64)
        _check(_fn["step_host"](self.h, _hptr(act), mode, _hptr(out.get("kilobots")), _hptr(out.get("objects")),
                                _hptr(out.get("light")), _hptr(out.get("reward")), _hptr(out.get("done")),
                                _hptr(out.get("status")), self._stream()), "kb_step_host")
        return out

    # ---- introspection (host numpy, synchronising)
    def bodies(self):
        out = np.zeros((self.E, self.B, abi.KB_BODY_STATE_FLOATS), np.float32)
        _check(_fn["get_bodies"](self.h, _hptr(out)), "kb_get_bodies")
        return out

    def set_poses(self, pose, body_mask=None):
        """Body.set_pose for the bodies flagged in body_mask [E,B] (None = all)."""
        pose = np.ascontiguousarray(pose, dtype=np.float64).reshape(self.E, self.B, 3)
        m = None if body_mask is None else np.ascontiguousarray(body_mask, dtype=np.uint8).reshape(self.E, self.B)
        _check(_fn["set_poses_masked"](self.h, _hptr(pose), _hptr(m)), "kb_set_poses_masked")

    def get_status(self):
        """Sticky per-env status words (host int32 [E]; synchronises)."""
        out = np.zeros(self.E, np.int32)
        _check(_fn["get_status"](self.h, _hptr(out)), "kb_get_status")
        return out

    def body_counts(self):
        """(objects [E], kilobots [E]) host int32: the counts of the scene each env was last reset with (before its
        first reset: its scene at creation).  Object j < objects[e] is body j, kilobot k < kilobots[e] is body M + k;
        the other body indices up to B are absent (include/kb_b200.h kb_create, padded body layout)."""
        obj = np.zeros(self.E, np.int32)
        kb = np.zeros(self.E, np.int32)
        _check(_fn["get_body_counts"](self.h, _hptr(obj), _hptr(kb)), "kb_get_body_counts")
        return obj, kb

    # ---- on-device scene sampling at reset (csrc/kb_sample.cuh)
    def set_sampler(self, spec):
        """spec: sampler.SceneSampler (or anything with to_abi() -> (KbSampleSpec, keep-alive))."""
        s, keep = spec.to_abi()
        _check(_fn["set_sampler"](self.h, C.byref(s)), "kb_set_sampler")
        self._sampler_keep = keep

    def set_sampler_mix(self, mix):
        """mix: sampler.SamplerMix (or anything with to_abi() -> (KbSampleSpec[K], K, weights or None, keep-alive))."""
        specs, k, weights, keep = mix.to_abi()
        _check(_fn["set_sampler_mix"](self.h, specs, k, weights), "kb_set_sampler_mix")
        self._sampler_keep = keep

    def current_scenes(self, out=None):
        """The scene each env was last reset with, as a DEVICE int32 [E] tensor (asynchronous, current stream)."""
        if out is None:
            out = self.torch.empty(self.E, dtype=self.torch.int32, device=self.device)
        _check(_fn["current_scenes"](self.h, C.c_void_p(out.data_ptr()), self._stream()), "kb_current_scenes")
        return out

    def reset_sampled(self, mask=None):
        """kb_reset with poses / light states drawn inside the reset kernel; mask: device or host uint8 [E] or None."""
        m = self._dev(mask, self.torch.uint8, (self.E,))
        _check(_fn["reset_sampled"](self.h, None if m is None else C.c_void_p(m.data_ptr()), self._stream()), "kb_reset_sampled")
        self._keep_reset = (m,)

    def get_sampled(self):
        """(body_pose [E,B,3], light_state [E,L], env_scene [E], episodes [E]) of the last sampled resets (host)."""
        pose = np.zeros((self.E, self.B, 3), np.float64)
        light = np.zeros((self.E, max(self.L, 1)), np.float64)
        scene = np.zeros(self.E, np.int32)
        ep = np.zeros(self.E, np.uint32)
        _check(_fn["get_sampled"](self.h, _hptr(pose), _hptr(light), _hptr(scene), _hptr(ep)), "kb_get_sampled")
        return pose, light[:, :self.L], scene, ep

    def set_env_scene(self, env_scene):
        es = np.ascontiguousarray(env_scene, dtype=np.int32).reshape(self.E)
        _check(_fn["set_env_scene"](self.h, _hptr(es)), "kb_set_env_scene")

    def reduce_episode_stats(self, out=None):
        """Rank-local sums of the episode statistics as a DEVICE float64[KB_REDUCED_STATS] tensor (asynchronous):
        the operand of the NCCL all-reduce in KilobotsVecEnv.all_reduce_episode_stats."""
        if out is None:
            out = self.torch.zeros(abi.KB_REDUCED_STATS, dtype=self.torch.float64, device=self.device)
        _check(_fn["reduce_episode_stats"](self.h, C.c_void_p(out.data_ptr()), self._stream()), "kb_reduce_episode_stats")
        return out

    def contacts(self):
        pairs = np.zeros((self.E, self.C, 4), np.int32)
        count = np.zeros(self.E, np.int32)
        _check(_fn["get_contacts"](self.h, _hptr(pairs), _hptr(count)), "kb_get_contacts")
        return pairs, count

    def impulses(self):
        out = np.zeros((self.E, self.C, 4), np.float32)
        _check(_fn["get_impulses"](self.h, _hptr(out)), "kb_get_impulses")
        return out

    def counters(self):
        out = np.zeros((self.E, abi.KB_NUM_COUNTERS), np.uint64)
        _check(_fn["get_counters"](self.h, _hptr(out)), "kb_get_counters")
        return out

    def proxies(self):
        out = np.zeros((self.E, self.P, 4), np.float32)
        _check(_fn["get_proxies"](self.h, _hptr(out)), "kb_get_proxies")
        return out

    def controllers(self):
        ctrl = np.zeros((self.E, self.N, 4), np.float64)
        light = np.zeros((self.E, max(self.L, 1)), np.float64)
        _check(_fn["get_controllers"](self.h, _hptr(ctrl), _hptr(light)), "kb_get_controllers")
        return ctrl, light[:, :self.L]

    def mass_data(self):
        out = np.zeros((len(self.scenes), self.B, 4), np.float32)
        _check(_fn["get_mass_data"](self.h, _hptr(out)), "kb_get_mass_data")
        return out

    # ---- task layer (extension: on-device reward / done / episode statistics / flat observation)
    def set_task(self, task, targets=None):
        """task: scene.TaskSpec; targets: [E,3] (x m, y m, theta) or None to keep the current ones."""
        t = task.to_def()
        tg = None if targets is None else np.ascontiguousarray(targets, dtype=np.float64).reshape(self.E, 3)
        _check(_fn["set_task"](self.h, C.byref(t), _hptr(tg)), "kb_set_task")

    def episode_stats(self):
        out = np.zeros((self.E, abi.KB_EPISODE_STATS), np.float64)
        _check(_fn["get_episode_stats"](self.h, _hptr(out)), "kb_get_episode_stats")
        return out

    def bind_flat_observation(self, enable=True):
        """Device tensor f32[E, 2N+L+4M] in YamlKilobotsEnv.observation_space order, refreshed by every step."""
        if not enable:
            self.obs_flat = None
            _check(_fn["bind_flat_observation"](self.h, None), "kb_bind_flat_observation")
            return None
        dim = _fn["flat_observation_dim"](self.h)
        self.obs_flat = self.torch.zeros((self.E, dim), dtype=self.torch.float32, device=self.device)
        _check(_fn["bind_flat_observation"](self.h, C.c_void_p(self.obs_flat.data_ptr())), "kb_bind_flat_observation")
        return self.obs_flat

    # ---- per-kilobot local observations (csrc/kb_local.cuh)
    def local_observation_dim(self, spec):
        """Row width D of scene.LocalObsSpec `spec` on this batch (raises if the batch cannot provide a part)."""
        d = spec.to_def()
        D = _fn["local_observation_dim"](self.h, C.byref(d))
        _check(min(D, 0), "kb_local_observation_dim")
        return D

    def local_observation(self, spec, mask=None, out=None):
        """Device float32 [E, Nmax, D]: each kilobot's neighbours, objects and light in its own frame, from the state after
        the last call on the current stream (asynchronous, no synchronisation).  mask: uint8 / bool [E] (device or
        host) or None; the rows of unmasked envs are left as they were.  Without `out` the result goes to a buffer
        kept per spec, so a later call with the same spec overwrites it."""
        torch = self.torch
        if out is None:
            cache = self.__dict__.setdefault("_local_out", {})
            out = cache.get(spec)
            if out is None:
                out = torch.full((self.E, self.N, self.local_observation_dim(spec)), float("nan"), dtype=torch.float32,
                                 device=self.device)   # (rows a masked call has not written yet)
                cache[spec] = out
        elif (out.dtype != torch.float32 or out.device != self.device or not out.is_contiguous()
              or tuple(out.shape) != (self.E, self.N, self.local_observation_dim(spec))):
            raise ValueError("out must be a contiguous float32 tensor [E, Nmax, D] on the batch's device")
        m = self._dev(mask, torch.uint8, (self.E,))
        d = spec.to_def()
        _check(_fn["local_observation"](self.h, C.byref(d), None if m is None else C.c_void_p(m.data_ptr()),
                                        C.c_void_p(out.data_ptr()), self._stream()),
               "kb_local_observation")
        self._keep_local = m
        return out

    def render(self, env_ids=(0,), width=1200, height=900):
        """uint8 CUDA tensor [len(env_ids), height, width, 3]: the picture KilobotsEnv.render would draw
        (kilobots_env.py:221-275; default size = screen_size :22), rasterised on the device."""
        ids = np.ascontiguousarray(env_ids, dtype=np.int32).reshape(-1)
        out = self.torch.empty((len(ids), height, width, 3), dtype=self.torch.uint8, device=self.device)
        _check(_fn["render"](self.h, _hptr(ids), len(ids), width, height, C.c_void_p(out.data_ptr()), self._stream()),
               "kb_render")
        return out

    def host_layout(self):
        """(offsets of kilobots, objects, light, reward, status, done; total bytes) of the packed host block."""
        off = (C.c_int64 * 6)()
        total = C.c_int64()
        _check(_fn["get_host_layout"](self.h, off, C.byref(total)), "kb_get_host_layout")
        return [int(x) for x in off], int(total.value)

    def launch_config(self):
        cfg = abi.KbLaunchConfig()
        _check(_fn["get_launch_config"](self.h, C.byref(cfg)), "kb_get_launch_config")
        out = {k: int(getattr(cfg, k)) for k, _ in cfg._fields_ if k not in ("specialised", "jit_ms", "jit_reason")}
        out["specialised"] = bool(cfg.specialised)
        out["jit_ms"] = round(float(cfg.jit_ms), 1)
        out["jit_reason"] = cfg.jit_reason.decode()
        out["kernel"] = ("kb_swarm_step_kernel (one CTA per env)" if out["lanes_per_env"] > 32
                         else "kb_step_kernel<%d>" % out["lanes_per_env"])
        return out

    def get_state(self):
        out = np.zeros((self.E, self.state_bytes_per_env), np.uint8)
        _check(_fn["get_state"](self.h, _hptr(out)), "kb_get_state")
        return out

    def set_state(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.uint8).reshape(self.E, self.state_bytes_per_env)
        _check(_fn["set_state"](self.h, _hptr(blob)), "kb_set_state")
