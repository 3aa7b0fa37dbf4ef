"""KilobotsVecEnv -- the vectorised N-env wrapper around the batched CUDA step.

The reference steps one environment per Python call (gym_kilobots/envs/kilobots_env.py:161-215);
this class steps E of them with one kernel launch.  Semantics per environment are exactly those of
`KilobotsEnv.step` / `reset`; the observation keeps the reference's dict layout
({'kilobots': [N,3], 'objects': [M,3], 'light': [L]}, kilobots_env.py:115-118) with a leading env axis.
The envs of one batch may differ in their numbers of objects and kilobots: N and M are then the largest counts,
`kilobot_mask` / `object_mask` say which rows an env populates, and the rows it does not are NaN.
With `local_observation=scene.LocalObsSpec(...)` the observation also holds obs['local'] [E, N, D]: what each kilobot
senses in its own frame (neighbours, objects, light), computed on the device after every step and reset.
With `actuation=scene.ActuationSpec(...)` the kilobots' motors differ per robot and episode (gains, drift, failures) and
are noisy per sub-step, drawn on the device.
"""
import numpy as np

from .. import _abi as abi
from .. import _native


class KilobotsVecEnv:
    """E independent Kilobots environments on one GPU.

    scenario: a `gym_kilobots_b200.scenarios.Scenario` (scene templates + initial poses), or anything
    with the attributes scenes / env_scene / body_pose / light_state / max_contacts.
    """

    def __init__(self, scenario, device=0, action_mode=abi.KB_ACTION_LIGHT, task=None, targets=None,
                 flat_observation=False, allow_status_flags=False, local_observation=None, actuation=None):
        """task / targets: optional `scene.TaskSpec` and per-env target poses [E,3] -- on-device reward, done and
        episode statistics (an extension: the reference's hooks are abstract and its in-tree envs return constants).
        flat_observation: also emit obs['flat'], the vector YamlKilobotsEnv.observation_space describes.
        local_observation: a `scene.LocalObsSpec`; also emit obs['local'], each kilobot's local observation.
        actuation: a `scene.ActuationSpec`; the kilobots drive through that actuation model (`set_actuation`)."""
        self.scenario = scenario
        # KB_STATUS_* bits (contact / solver capacity overflow, non-finite pose) raise KbStatusError in step() and
        # check_status() unless explicitly allowed: a dropped pair is silently different physics
        self.allow_status_flags = allow_status_flags
        self.batch = _native.NativeBatch(scenario.scenes, scenario.body_pose.shape[0], scenario.env_scene,
                                         scenario.max_contacts, device=device)
        self.num_envs = self.batch.E
        self.num_kilobots = self.batch.N
        self.num_objects = self.batch.M
        self.action_mode = action_mode
        self.action_dim = 2 * self.batch.N if action_mode == abi.KB_ACTION_KILOBOTS else self.batch.A
        self._host = None
        self._sim_steps = 0
        self.obs_flat = self.batch.bind_flat_observation() if flat_observation else None
        self.local_spec = local_observation
        if local_observation is not None:
            self.local_dim = self.batch.local_observation_dim(local_observation)   # refuses a part the batch lacks
        self._init_masks()
        if task is not None:
            self.set_task(task, targets)
        if actuation is not None:
            self.set_actuation(actuation)

    def _init_masks(self):
        """kilobot_mask [E,N] / object_mask [E,M]: bool CUDA tensors, True where the env's current scene has that
        kilobot / object.  They follow every reset on the device: an env's counts change only when a reset rebuilds
        it after `set_env_scene`."""
        import torch
        dev = self.batch.device
        specs = self.scenario.scenes
        self._scene_objects = torch.tensor([sp.num_objects for sp in specs], dtype=torch.int64, device=dev)
        self._scene_kilobots = torch.tensor([sp.num_kilobots for sp in specs], dtype=torch.int64, device=dev)
        es = self.scenario.env_scene
        self._env_scene = torch.zeros(self.num_envs, dtype=torch.int64, device=dev) if es is None else \
            torch.as_tensor(np.asarray(es, np.int64), device=dev)
        self._scene_now = self._env_scene.clone()   # the scene each env was last reset with
        self.mixed_counts = len({(sp.num_objects, sp.num_kilobots) for sp in specs}) > 1
        self._update_masks()

    def _update_masks(self):
        import torch
        dev = self.batch.device
        self.kilobot_mask = torch.arange(self.num_kilobots, device=dev)[None, :] < self._scene_kilobots[self._scene_now][:, None]
        self.object_mask = torch.arange(self.num_objects, device=dev)[None, :] < self._scene_objects[self._scene_now][:, None]

    def _after_reset(self, mask):
        if not self.mixed_counts:
            return
        import torch
        if mask is None:
            self._scene_now = self._env_scene.clone()
        else:
            m = torch.as_tensor(mask, device=self.batch.device).reshape(self.num_envs).bool()
            self._scene_now = torch.where(m, self._env_scene, self._scene_now)
        self._update_masks()

    def _after_sampled_reset(self, mask):
        """A sampled reset of a mixed batch may move envs to scenes of other sizes: read the scenes on the device (no
        synchronisation) and let the masks follow; the reset envs' next scene is the one they were reset with."""
        if not self.mixed_counts:
            return
        import torch
        self._scene_now = self.batch.current_scenes().long()
        if mask is None:
            self._env_scene = self._scene_now.clone()
        else:
            m = torch.as_tensor(mask, device=self.batch.device).reshape(self.num_envs).bool()
            self._env_scene = torch.where(m, self._scene_now, self._env_scene)
        self._update_masks()

    def set_env_scene(self, env_scene):
        """Move envs to other scene templates of the batch (int [E]); an env changes at its next reset, which may change
        its numbers of objects and kilobots (the masks follow at that reset)."""
        import torch
        es = np.asarray(env_scene, np.int32).reshape(self.num_envs)
        self.batch.set_env_scene(es)
        self.scenario.env_scene = es
        self._env_scene = torch.as_tensor(es.astype(np.int64), device=self.batch.device)

    @classmethod
    def from_envs(cls, envs, device=0, **kwargs):
        """Vectorise reference-style envs (instances of KilobotsEnv subclasses, e.g. E YamlKilobotsEnv built from
        one configuration): their scenes are recorded by `scenarios.from_envs` and stepped as ONE batch.
        DirectControlKilobotsEnv instances select per-kilobot actions."""
        from .. import scenarios
        from .direct_control_kilobots_env import DirectControlKilobotsEnv
        envs = list(envs)
        sc = scenarios.from_envs(envs)
        mode = abi.KB_ACTION_KILOBOTS if isinstance(envs[0], DirectControlKilobotsEnv) else abi.KB_ACTION_LIGHT
        vec = cls(sc, device=device, action_mode=mode, **kwargs)
        vec.envs = envs
        return vec

    def resample(self, mask=None):
        """Re-run `_configure_environment` of the (masked) source envs -> fresh initial poses / light states, the
        way a reference `reset()` re-samples its scene.  Only for batches built by `from_envs`; scene templates
        must not change.  Returns (body_pose [E,B,3], light_state [E,L]) for `reset` / `reset_done`."""
        if getattr(self, "envs", None) is None:
            raise RuntimeError("resample() needs the source env objects: build the batch with KilobotsVecEnv.from_envs "
                               "(or use on-device sampling: KilobotsVecEnv.from_configuration)")
        from .. import scenarios
        sc = self.scenario
        for i, env in enumerate(self.envs):
            if mask is not None and not mask[i]:
                continue
            _, pose, light, _ = env._record_scene()
            sc.body_pose[i] = scenarios.stack_poses(sc.scenes, [0 if sc.env_scene is None else sc.env_scene[i]], [pose])[0]
            if light is not None:
                sc.light_state[i] = light
        return sc.body_pose, sc.light_state

    # -- task layer (extension) -----------------------------------------------------------------
    def set_task(self, task, targets=None):
        self.batch.set_task(task, targets)

    # -- actuation model (extension) --------------------------------------------------------------
    def set_actuation(self, spec):
        """Attach a `scene.ActuationSpec` (None detaches it).  Draws episode 0 of every env now; every reset then draws the
        reset envs' next episode on the device."""
        self.batch.set_actuation(spec)

    def actuation_draws(self):
        """float32 [E, N, 4] host array: every kilobot slot's (speed gain, turn-rate gain, turn-rate drift rad/s, alive)
        in the env's current episode -- for logging or a privileged critic."""
        return self.batch.actuation()[0]

    def episode_stats(self):
        """dict of [E] float64 arrays: return, length, position_error, orientation_error, success, done_count."""
        st = self.batch.episode_stats()
        return {n: st[:, i] for i, n in enumerate(abi.EPISODE_STAT_NAMES)}

    @classmethod
    def from_configuration(cls, configuration, num_envs, seed=0, env_id_base=0, device=0, max_contacts=0, **kwargs):
        """E YamlKilobotsEnv(configuration=...) as ONE batch whose scenes are drawn on the device: objects, light(s)
        and kilobots are re-sampled inside the reset kernel (counter-based, keyed by seed / global env id / episode),
        like every reference reset() re-draws them (yaml_kilobots_env.py:194-198,256-283,299,327-354).
        env_id_base: global id of this batch's env 0 (rank * num_envs), so that R ranks draw what one rank would."""
        from .. import scenarios
        from ..sampler import SceneSampler
        sampler = SceneSampler(configuration, seed=seed, env_id_base=env_id_base)
        specs = sampler.scene_specs()
        pose, light, scene = sampler.sample_numpy(np.arange(num_envs), 0)
        sc = scenarios.Scenario("yaml", specs, scene.astype(np.int32), pose, light, max_contacts=max_contacts)
        vec = cls(sc, device=device, **kwargs)
        vec.use_device_sampler(sampler)
        return vec

    @classmethod
    def from_configurations(cls, configurations, num_envs, weights=None, env_config=None, seed=0, env_id_base=0, device=0,
                            max_contacts=0, **kwargs):
        """E envs over several Yaml configurations as ONE batch whose scenes are drawn on the device (`sampler.SamplerMix`):
        a curriculum or domain randomisation over swarm size and object sets.  The configurations may differ in their
        numbers of objects and kilobots (`kilobot_mask` / `object_mask` follow every reset on the device).  Give exactly
        one of
          weights     [K]: every sampled reset draws the env's configuration with these weights (keyed by seed / global
                      env id / episode, like every other draw: 1 and 8 GPUs agree);
          env_config  [E]: the configuration of every env; it keeps it at every reset until `set_env_scene` moves it
                      (to `sampler.first_scene(c)` of another configuration c).
        env_id_base: global id of this batch's env 0 (rank * num_envs)."""
        from .. import scenarios
        from ..sampler import SamplerMix
        if (weights is None) == (env_config is None):
            raise ValueError("give exactly one of weights / env_config")
        mix = SamplerMix(configurations, weights=weights, seed=seed, env_id_base=env_id_base)
        env_scene = None
        if env_config is not None:
            cfg = np.asarray(env_config, np.int64).reshape(-1)
            if len(cfg) != num_envs or np.any(cfg < 0) or np.any(cfg >= len(mix.samplers)):
                raise ValueError("env_config must hold one configuration index per env")
            env_scene = mix.scene_offset[cfg]
        # the scenario at creation is the episode-0 draw, so that creation and the first reset() agree
        pose, light, scene, _ = mix.sample_numpy(np.arange(num_envs), 0, env_scene)
        sc = scenarios.Scenario("yaml-mix", mix.scene_specs(), scene.astype(np.int32), pose, light,
                                max_contacts=max_contacts)
        vec = cls(sc, device=device, **kwargs)
        vec.use_device_sampler(mix)
        return vec

    def use_device_sampler(self, sampler, seed=0, env_id_base=0):
        """Attach on-device scene sampling: `reset()` and `reset_done()` then draw fresh scenes inside the reset kernel
        (kb_reset_sampled, one launch, no host round trip).  sampler: a `sampler.SceneSampler`, a `sampler.SamplerMix`
        (several configurations: see `from_configurations`), or a Yaml configuration (then the batch's scenes must
        already be the sampler's: see `from_configuration`)."""
        from ..sampler import SamplerMix, SceneSampler
        if isinstance(sampler, SamplerMix):
            if (sampler.M, sampler.N, sampler.light_state_dim()) != (self.batch.M, self.batch.N, self.batch.L):
                raise ValueError("the configurations do not match the batch (objects / kilobots / light state)")
            if len(sampler.scene_config) > len(self.scenario.scenes):
                raise ValueError("the batch lacks scene templates of the mix (from_configurations)")
            self.batch.set_sampler_mix(sampler)
            self.sampler = sampler
            return sampler
        if self.mixed_counts:
            raise ValueError("on-device scene sampling draws one configuration: the batch's scenes differ in their "
                             "numbers of objects / kilobots")
        if not isinstance(sampler, SceneSampler):
            sampler = SceneSampler(sampler, seed=seed, env_id_base=env_id_base)
        if (sampler.M, sampler.N, sampler.light_state_dim()) != (self.batch.M, self.batch.N, self.batch.L):
            raise ValueError("configuration does not match the batch (objects / kilobots / light state)")
        if len(sampler.perms) > len(self.scenario.scenes):
            raise ValueError("a shuffled composite light needs one scene template per permutation (from_configuration)")
        self.batch.set_sampler(sampler)
        self.sampler = sampler
        return sampler

    def reset_done(self, done, body_pose=None, light_state=None):
        """Auto-reset: rebuild only the envs whose `done` flag is set (device or host array).  Poses come from the
        arguments, else from the attached device sampler (a fresh draw inside the reset kernel), else from the
        scenario's initial poses."""
        if body_pose is None and getattr(self, "sampler", None) is not None:
            self.batch.reset_sampled(done)
            self._after_sampled_reset(done)
        else:
            pose = self.scenario.body_pose if body_pose is None else body_pose
            light = self.scenario.light_state if light_state is None else light_state
            self.batch.reset(pose, light, None, done)
            self._after_reset(done)
        if self.local_spec is not None:
            self.batch.local_observation(self.local_spec, mask=done)   # the rebuilt envs' rows of obs['local']

    def local_observation(self, mask=None):
        """obs['local'] of the current state on demand: device float32 [E, N, D] (the buffer step_device returns);
        mask [E]: refresh only those envs' rows."""
        if self.local_spec is None:
            raise ValueError("the batch was built without local_observation=LocalObsSpec(...)")
        return self.batch.local_observation(self.local_spec, mask=mask)

    # -- gym-like surface ---------------------------------------------------------------------
    @property
    def action_space(self):
        from ..spaces import Box
        sc = self.scenario.scenes[0]
        lo = np.concatenate([np.asarray(l.action_bounds[0], float).ravel()[:l.action_dim] for l in sc.lights]) \
            if sc.lights else np.zeros(0)
        hi = np.concatenate([np.asarray(l.action_bounds[1], float).ravel()[:l.action_dim] for l in sc.lights]) \
            if sc.lights else np.zeros(0)
        return Box(lo, hi, dtype=np.float64)

    def reset(self, body_pose=None, light_state=None, kb_velocity=None, mask=None):
        """KilobotsEnv.reset for every (masked) env: rebuild bodies at the poses, one settle step."""
        if body_pose is None and getattr(self, "sampler", None) is not None:
            self.batch.reset_sampled(mask)    # a fresh scene per env, like every reference reset()
            self._after_sampled_reset(mask)
        else:
            pose = self.scenario.body_pose if body_pose is None else body_pose
            light = self.scenario.light_state if light_state is None else light_state
            if kb_velocity is None:
                kb_velocity = getattr(self.scenario, "kb_velocity", None)
            self.batch.reset(pose, light, kb_velocity, mask)
            self._after_reset(mask)
        self._sim_steps = 0
        obs = self.get_observation()
        if self.local_spec is not None:
            obs["local"] = self.batch.local_observation(self.local_spec, mask=mask).cpu().numpy()
        return obs

    def step_device(self, action):
        """Device tensors in, device tensors out, no synchronisation (training-loop path)."""
        k, o, l, r, d, s = self.batch.step_device(action, self.action_mode if action is not None else None)
        self._sim_steps += self.scenario.scenes[0].steps_per_action
        obs = {"kilobots": k, "objects": o, "light": l}
        if self.obs_flat is not None:
            obs["flat"] = self.obs_flat
        if self.local_spec is not None:
            obs["local"] = self.batch.local_observation(self.local_spec)
        return obs, r, d, {"status": s}

    def _host_buffers(self):
        if self._host is None:
            import torch
            b = self.batch
            pin = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()
            # one pinned block laid out like the library's staging area -> a single device->host copy per step
            off, total = b.host_layout()
            block = pin((max(total, 1),), torch.uint8)
            self._host_block = block

            def view(i, shape, dt):
                n = int(np.prod(shape)) * np.dtype(dt).itemsize
                return block[off[i]:off[i] + n].view(dt).reshape(shape)
            self._host = {
                "action": pin((b.E, max(self.action_dim, 1)), torch.float64),
                "kilobots": view(0, (b.E, b.N, 3), np.float32),
                "objects": view(1, (b.E, b.M, 3), np.float32),
                "light": view(2, (b.E, b.L), np.float64),
                "reward": view(3, (b.E,), np.float32),
                "status": view(4, (b.E,), np.int32),
                "done": view(5, (b.E,), np.uint8),
            }
        return self._host

    def step(self, action):
        """Host numpy in, host numpy out (pinned staging, copies inside the call): the drop-in path.

        Returns (observation dict, reward [E], done [E], info) like KilobotsEnv.step."""
        hb = self._host_buffers()
        if action is None:
            mode, act = abi.KB_ACTION_NONE, None
        else:
            mode = self.action_mode
            act = hb["action"]
            a = np.asarray(action)
            if a.dtype == np.float64 and a.flags.c_contiguous and a.size == act.size:
                act = a.reshape(act.shape)   # the caller's buffer goes to the device as it is (pin it for async copies)
            else:
                act[...] = np.asarray(action, dtype=np.float64).reshape(act.shape)
        self.batch.step_host(act, mode, hb)
        if not self.allow_status_flags and hb["status"].any():
            raise _native.KbStatusError(_native.describe_status(hb["status"]))
        self._sim_steps += self.scenario.scenes[0].steps_per_action
        obs = {"kilobots": hb["kilobots"], "objects": hb["objects"], "light": hb["light"]}
        if self.obs_flat is not None:
            obs["flat"] = self.obs_flat.cpu().numpy()
        if self.local_spec is not None:
            obs["local"] = self.batch.local_observation(self.local_spec).cpu().numpy()
        return obs, hb["reward"], hb["done"].astype(bool), {"status": hb["status"]}

    def check_status(self):
        """The device path (`step_device`, `reset`) never synchronises; call this at logging cadence.  Raises
        KbStatusError if any env carries a status bit (unless allow_status_flags), returns the int32 [E] words."""
        st = self.batch.get_status()
        if not self.allow_status_flags and st.any():
            raise _native.KbStatusError(_native.describe_status(st))
        return st

    def all_reduce_episode_stats(self, group=None):
        """Episode statistics of the WHOLE job: this rank's envs are summed on the device (kb_reduce_episode_stats,
        one launch) and the KB_REDUCED_STATS doubles are all-reduced over the ranks (NCCL when torch.distributed is
        initialised with the nccl backend -- the only collective of this path; environments never exchange physics).
        Returns a dict of Python floats: env count, sums and means of the per-env statistics, flagged envs."""
        import torch.distributed as dist
        t = self.batch.reduce_episode_stats()
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            if dist.get_backend(group) != "nccl":
                t = t.cpu()   # gloo (CPU test rigs) reduces host tensors
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        v = t.cpu().numpy()
        out = {"sum_" + n: float(x) for n, x in zip(abi.REDUCED_STAT_NAMES, v)}
        n = max(out["sum_envs"], 1.0)
        out.update({"envs": int(out.pop("sum_envs")), "envs_with_status": int(out.pop("sum_envs_with_status")),
                    "episodes_done": out["sum_done_count"]})
        for k in ("return", "length", "position_error", "orientation_error", "success"):
            out["mean_" + k] = out["sum_" + k] / n
        return out

    def host_io_bytes(self):
        """(bytes host->device, bytes device->host) moved by one `step` call."""
        hb = self._host_buffers()
        h2d = hb["action"].nbytes if self.action_dim > 0 else 0
        d2h = sum(hb[k].nbytes for k in ("kilobots", "objects", "light", "reward", "done", "status"))
        return h2d, d2h

    def render(self, env_ids=(0,), width=1200, height=900, mode="rgb_array"):
        """The frame(s) KilobotsEnv.render would draw (kilobots_env.py:221-275) for the given envs, rasterised on
        the GPU: uint8 [len(env_ids), height, width, 3] (numpy for 'rgb_array', CUDA tensor for 'tensor')."""
        img = self.batch.render(env_ids, width, height)
        return img if mode == "tensor" else img.cpu().numpy()

    def get_state(self):
        b = self.batch.bodies()
        _, light = self.batch.controllers()
        M = self.num_objects
        pose = np.stack([b[..., 8].astype(np.float64) / 25.0, b[..., 9].astype(np.float64) / 25.0,
                         b[..., 2].astype(np.float64)], axis=-1)
        kb, obj = pose[:, M:], pose[:, :M]
        if self.mixed_counts:   # rows of absent bodies are NaN, as in step()
            n_obj, n_kb = self.batch.body_counts()
            kb[np.arange(self.num_kilobots)[None, :] >= n_kb[:, None]] = np.nan
            obj[np.arange(M)[None, :] >= n_obj[:, None]] = np.nan
        return {"kilobots": kb, "objects": obj, "light": light}

    def get_observation(self):
        return self.get_state()

    def close(self):
        self.batch.close()
