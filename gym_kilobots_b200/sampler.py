"""SceneSampler -- the random scene initialisation of YamlKilobotsEnv as a counter-based function.

The reference re-draws its scene in every reset() (gym_kilobots/envs/yaml_kilobots_env.py:194-198 objects, :256-283
lights, :299 shuffle of a composite light's components, :327-354 kilobots) from numpy's global generator.  The batched
path draws the same quantities INSIDE the reset kernel (csrc/kb_sample.cuh) as a pure function of
(seed, global env id, episode count); this module holds the host description of that function (`to_abi`), the scene
templates it needs (one per permutation of a shuffled composite light: light constants are per scene), and a numpy
evaluation of the very same draws (`sample_numpy`) that the tests compare the device against and that CPU-side tools
can use without a GPU.
"""
import copy
import ctypes as C
import itertools
import math

import numpy as np

from . import _abi as abi
from . import philox as PX


def _leaves(lc):
    """Light components in configuration order; (components, shuffle) for a top-level composite light."""
    if lc is None:
        return [], False
    if isinstance(lc, dict):
        from types import SimpleNamespace
        lc = SimpleNamespace(type=lc.get("type", lc.get("obj_type")), init=lc.get("init"), radius=lc.get("radius"),
                             components=lc.get("components"))
    if lc.type == "composite":
        out = []
        for c in lc.components:
            out += _leaves(c)[0]
        return out, isinstance(lc.init, str) and lc.init == "random"
    return [lc], False


class SceneSampler:
    def __init__(self, conf, seed=0, env_id_base=0):
        self.conf = conf
        self.seed = int(seed)
        self.env_id_base = int(env_id_base)
        self.size = np.array([float(conf.width), float(conf.height)])
        self.objects = []
        for o in conf.objects:
            random = isinstance(o.init, str) and o.init == "random"
            pose = np.zeros(3) if random else np.asarray(o.init, dtype=np.float64)
            self.objects.append((abi.KB_SAMPLE_RANDOM if random else abi.KB_SAMPLE_FIXED, pose,
                                 max(float(o.width), float(o.height))))
        leaves, self.shuffle = _leaves(getattr(conf, "light", None))
        self.light_types = [{"circular": abi.KB_LIGHT_CIRCULAR, "momentum": abi.KB_LIGHT_MOMENTUM,
                             "linear": abi.KB_LIGHT_LINEAR}[l.type] for l in leaves]
        self.lights = []
        for l in leaves:
            if l.type == "linear":
                self.lights.append((abi.KB_SAMPLE_FIXED, np.array([float(l.init), 0.0])))
            elif isinstance(l.init, str) and l.init == "random":
                self.lights.append((abi.KB_SAMPLE_RANDOM, np.zeros(2)))
            elif isinstance(l.init, str) and l.init == "object":
                self.lights.append((abi.KB_SAMPLE_AT_OBJECT, np.zeros(2)))
            else:
                self.lights.append((abi.KB_SAMPLE_FIXED, np.asarray(l.init, dtype=np.float64)))
        self.shuffle = self.shuffle and len(self.lights) > 1
        mean = conf.kilobots.mean
        if isinstance(mean, str) and mean == "light":
            self.mean_mode, self.mean = abi.KB_SAMPLE_MEAN_LIGHT, np.zeros(2)
        elif isinstance(mean, str) and mean == "random":
            self.mean_mode, self.mean = abi.KB_SAMPLE_MEAN_RANDOM, np.zeros(2)
        else:
            self.mean_mode, self.mean = abi.KB_SAMPLE_FIXED, np.asarray(mean, dtype=np.float64)
        self.std = float(conf.kilobots.std)
        self.M, self.N = len(self.objects), int(conf.kilobots.num)
        # permutations of the components in lexicographic order: perms[rank][pos] = component at position pos
        self.perms = list(itertools.permutations(range(len(self.lights)))) if self.shuffle else [tuple(range(len(self.lights)))]
        self.perm_scene = list(range(len(self.perms)))

    # ------------------------------------------------------------------ scene templates
    def scene_specs(self):
        """One SceneSpec per permutation of the light components (just one without shuffle); index == perm_scene[rank]."""
        from .envs.yaml_kilobots_env import YamlKilobotsEnv
        conf = copy.deepcopy(self.conf)
        if self.shuffle:
            conf.light.init = None   # the canonical component order (the facade would shuffle it in place)
        state = np.random.get_state()
        try:
            spec = YamlKilobotsEnv(configuration=conf)._record_scene()[0]
        finally:
            np.random.set_state(state)
        out = []
        for perm in self.perms:
            s = copy.copy(spec)
            s.lights = [spec.lights[c] for c in perm]
            out.append(s)
        return out

    def light_state_dim(self):
        return sum({abi.KB_LIGHT_CIRCULAR: 2, abi.KB_LIGHT_MOMENTUM: 4, abi.KB_LIGHT_LINEAR: 1}[t] for t in self.light_types)

    # ------------------------------------------------------------------ C-ABI description
    def to_abi(self):
        objs = (abi.KbSampleObject * max(self.M, 1))()
        for i, (mode, pose, extent) in enumerate(self.objects):
            objs[i].mode = mode
            objs[i].pose[:] = list(pose)
            objs[i].extent = extent
        lights = (abi.KbSampleLight * max(len(self.lights), 1))()
        for i, (mode, init) in enumerate(self.lights):
            lights[i].mode = mode
            lights[i].init[:] = list(init)
        perm = (C.c_int32 * len(self.perm_scene))(*self.perm_scene)
        s = abi.KbSampleSpec()
        s.seed, s.env_id_base = self.seed, self.env_id_base
        s.world_width, s.world_height = float(self.size[0]), float(self.size[1])
        s.num_objects, s.num_lights = self.M, len(self.lights)
        s.objects = C.cast(objs, C.POINTER(abi.KbSampleObject))
        s.lights = C.cast(lights, C.POINTER(abi.KbSampleLight))
        s.shuffle_lights = 1 if self.shuffle else 0
        s.kilobot_mean_mode = self.mean_mode
        s.perm_scene = C.cast(perm, C.POINTER(C.c_int32))
        s.kilobot_mean[:] = list(self.mean)
        s.kilobot_std = self.std
        return s, (objs, lights, perm)

    # ------------------------------------------------------------------ the same draws in numpy
    def sample_numpy(self, env_ids, episodes=0):
        """(body_pose [E, M+N, 3], light_state [E, L], scene [E]) for the given LOCAL env ids and episode counts --
        draw for draw what kb_sample.cuh computes (differences: the last ulp of log / sin / cos)."""
        env = np.asarray(env_ids, dtype=np.int64)
        E = len(env)
        rng = PX.EnvRng(self.seed, env + self.env_id_base, episodes)
        lo = -self.size / 2
        M, N, NL = self.M, self.N, len(self.lights)
        pose = np.zeros((E, M + N, 3))
        # shuffle -> order[e][pos] = component
        order = np.tile(np.arange(max(NL, 1)), (E, 1))
        scene = np.zeros(E, np.int32)
        if self.shuffle:
            for j in range(NL - 1, 0, -1):
                u0, _ = rng.uniform2(PX.STREAM_SHUFFLE, j)
                r = np.minimum((u0 * (j + 1)).astype(np.int64), j)
                idx = np.arange(E)
                oj, orr = order[idx, j].copy(), order[idx, r].copy()
                order[idx, j], order[idx, r] = orr, oj
            rank_of = {p: i for i, p in enumerate(self.perms)}
            scene = np.array([self.perm_scene[rank_of[tuple(o[:NL])]] for o in order], np.int32)
        for i, (mode, fixed, _) in enumerate(self.objects):
            if mode == abi.KB_SAMPLE_RANDOM:
                u0, u1 = rng.uniform2(PX.STREAM_OBJECT, 2 * i)
                a0, _ = rng.uniform2(PX.STREAM_OBJECT, 2 * i + 1)
                pose[:, i, 0] = (u0 * self.size[0] + lo[0]) * 0.7
                pose[:, i, 1] = (u1 * self.size[1] + lo[1]) * 0.7
                pose[:, i, 2] = a0 * 2 * math.pi - math.pi
            else:
                pose[:, i] = fixed
        extent = np.array([o[2] for o in self.objects]) if M else np.zeros(1)
        L = self.light_state_dim()
        light = np.zeros((E, max(L, 1)))
        positional = [[] for _ in range(E)]     # state offsets of the positional lights per env
        types = np.array(self.light_types + [0])[order] if NL else np.zeros((E, 0), int)
        for e in range(E):
            off = 0
            for pos in range(NL):
                c, t = order[e, pos], types[e, pos]
                mode, init = self.lights[c]
                if t == abi.KB_LIGHT_LINEAR:
                    light[e, off] = init[0]
                    off += 1
                    continue
                sel = np.array([e])
                if mode == abi.KB_SAMPLE_RANDOM:
                    u0, u1 = rng.uniform2(PX.STREAM_LIGHT, 4 * pos, sel=sel)
                    p = np.array([u0[0] * self.size[0] + lo[0], u1[0] * self.size[1] + lo[1]])
                elif mode == abi.KB_SAMPLE_AT_OBJECT and M > 0:
                    u0, u1 = rng.uniform2(PX.STREAM_LIGHT, 4 * pos + 1, sel=sel)
                    which = min(int(u0[0] * M), M - 1)
                    radius = 1.2 * extent[which] / 2
                    angle = u1[0] * 2 * math.pi - math.pi
                    p = pose[e, which, :2] + np.array([math.cos(angle) * radius, math.sin(angle) * radius])
                else:
                    p = np.asarray(init, dtype=np.float64)
                light[e, off:off + 2] = p
                positional[e].append(off)
                if t == abi.KB_LIGHT_MOMENTUM:
                    u0, _ = rng.uniform2(PX.STREAM_LIGHT, 4 * pos + 2, sel=sel)
                    angle = u0[0] * 2 * math.pi - math.pi
                    light[e, off + 2:off + 4] = (math.sin(angle) * .01, math.cos(angle) * .01)
                    off += 4
                else:
                    off += 2
        npos = np.array([len(p) for p in positional])
        mean_mode = np.where((self.mean_mode == abi.KB_SAMPLE_MEAN_LIGHT) & (npos == 0), abi.KB_SAMPLE_MEAN_RANDOM, self.mean_mode)
        u0, u1 = rng.uniform2(PX.STREAM_SWARM, 0)
        rmean = np.stack([(u0 * self.size[0] + lo[0]) * 0.9, (u1 * self.size[1] + lo[1]) * 0.9], axis=-1)
        k = np.arange(N)[None, :]
        pick_u, _ = rng.uniform2(PX.STREAM_SWARM, 1 + k)
        z0, z1 = rng.normal2(PX.STREAM_KILOBOT_POS, k)
        mu = np.zeros((E, N, 2))
        for e in range(E):
            if mean_mode[e] == abi.KB_SAMPLE_MEAN_LIGHT:
                if npos[e] > 1:
                    pick = np.minimum((pick_u[e] * npos[e]).astype(np.int64), npos[e] - 1)
                else:
                    pick = np.zeros(N, np.int64)
                offs = np.array(positional[e])[pick]
                mu[e, :, 0], mu[e, :, 1] = light[e, offs], light[e, offs + 1]
            elif mean_mode[e] == abi.KB_SAMPLE_MEAN_RANDOM:
                mu[e] = rmean[e]
            else:
                mu[e] = self.mean
        xy = np.stack([z0, z1], axis=-1) * self.std + mu
        xy = np.minimum(np.maximum(xy, lo + 0.02), -lo - 0.02)
        pose[:, M:, :2] = xy
        return pose, light[:, :L], scene


class SamplerMix:
    """Several Yaml configurations over ONE batch (kb_set_sampler_mix): a curriculum or domain randomisation over swarm
    size and object sets.  Every configuration keeps its own `SceneSampler`; the batch's scene templates are theirs,
    concatenated (configuration c owns scenes scene_offset[c] ..).  Bodies use the batch's padded layout: with M / N the
    largest object / kilobot counts, an env's objects are rows 0..M_e-1 and its kilobots rows M + k.

    weights None: a sampled reset draws the configuration of the env's scene (`KilobotsVecEnv.set_env_scene` moves an env
    to another configuration).  weights [K] (finite, >= 0, positive sum): every sampled reset draws the configuration,
    c = first k with u < cdf[k], u a uniform of its own stream (philox.STREAM_CONFIG) keyed by (seed, global env id,
    episode) -- then the scene of c exactly as c's SceneSampler would.  So a size curriculum is a pure device loop whose
    draws do not depend on the batch size or the number of ranks."""

    def __init__(self, configurations, weights=None, seed=0, env_id_base=0):
        confs = list(configurations)
        K = len(confs)
        if not 1 <= K <= abi.KB_SAMPLE_MAX_CONFIGS:
            raise ValueError("a mix holds 1 to %d configurations, got %d" % (abi.KB_SAMPLE_MAX_CONFIGS, K))
        self.seed, self.env_id_base = int(seed), int(env_id_base)
        self.samplers = [SceneSampler(c, seed=seed, env_id_base=env_id_base) for c in confs]
        s0 = self.samplers[0]
        for c, s in enumerate(self.samplers):
            if s.M > abi.KB_SAMPLE_MAX_OBJECTS:
                raise ValueError("configuration %d has %d objects: on-device sampling draws at most %d"
                                 % (c, s.M, abi.KB_SAMPLE_MAX_OBJECTS))
            if s.light_types != s0.light_types or s.light_state_dim() != s0.light_state_dim():
                raise ValueError("configuration %d has other light components than configuration 0: the envs of a batch "
                                 "share their light state and action vectors" % c)
            if not np.array_equal(s.size, s0.size):
                raise ValueError("configuration %d has another table size than configuration 0" % c)
        counts = [len(s.perms) for s in self.samplers]
        self.scene_offset = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
        for s, off in zip(self.samplers, self.scene_offset):
            s.perm_scene = [int(off) + i for i in range(len(s.perms))]
        self.scene_config = np.concatenate([np.full(n, c, np.int32) for c, n in enumerate(counts)])
        self.M = max(s.M for s in self.samplers)
        self.N = max(s.N for s in self.samplers)
        self.weights = self.cdf = None
        if weights is not None:
            w = np.asarray(weights, dtype=np.float64).reshape(-1)
            if len(w) != K:
                raise ValueError("%d weights for %d configurations" % (len(w), K))
            if not np.all(np.isfinite(w)) or np.any(w < 0):
                raise ValueError("weights must be finite and non-negative")
            total = 0.0
            for x in w:
                total += float(x)
            if not (total > 0.0 and math.isfinite(total)):
                raise ValueError("weights must have a positive sum")
            # the cumulative weights exactly as kb_set_sampler_mix forms them: 1.0 from the last positive weight on
            last = int(np.flatnonzero(w > 0)[-1])
            cdf, acc = [], 0.0
            for k in range(K):
                acc += float(w[k])
                cdf.append(1.0 if k >= last else acc / total)
            self.weights, self.cdf = w, np.array(cdf)

    def scene_specs(self):
        """The batch's scene templates: every configuration's (SceneSampler.scene_specs), in configuration order."""
        return [sp for s in self.samplers for sp in s.scene_specs()]

    def first_scene(self, config):
        """The scene an env of configuration `config` starts from (set_env_scene moves it there)."""
        return int(self.scene_offset[config])

    def light_state_dim(self):
        return self.samplers[0].light_state_dim()

    def to_abi(self):
        """(KbSampleSpec[K], K, weights f64[K] or None, keep-alive): the arguments of kb_set_sampler_mix."""
        K = len(self.samplers)
        specs = (abi.KbSampleSpec * K)()
        keep = []
        for c, s in enumerate(self.samplers):
            specs[c], k = s.to_abi()
            keep.append(k)
        w = None if self.weights is None else (C.c_double * K)(*[float(x) for x in self.weights])
        return specs, K, w, (specs, keep, w)

    def sample_numpy(self, env_ids, episodes=0, env_scene=None):
        """(body_pose [E, M+N, 3], light_state [E, L], scene [E], config [E]) for the given LOCAL env ids and episode
        counts, in the padded layout with NaN rows for absent bodies.  env_scene [E]: the envs' scenes, which pick the
        configuration when the mix has no weights."""
        env = np.asarray(env_ids, dtype=np.int64).reshape(-1)
        E = len(env)
        ep = np.broadcast_to(np.asarray(episodes, dtype=np.int64), (E,))
        K = len(self.samplers)
        if self.cdf is not None:
            u, _ = PX.EnvRng(self.seed, env + self.env_id_base, ep).uniform2(PX.STREAM_CONFIG, 0)
            config = np.argmax(u[:, None] < self.cdf[None, :], axis=1).astype(np.int32)
        elif K == 1:
            config = np.zeros(E, np.int32)
        elif env_scene is None:
            raise ValueError("without weights an env's configuration is that of its scene: pass env_scene")
        else:
            config = self.scene_config[np.asarray(env_scene, np.int64).reshape(E)]
            if np.any(config < 0):
                raise ValueError("env_scene holds a scene of no configuration")
        pose = np.full((E, self.M + self.N, 3), np.nan)
        light = np.zeros((E, self.light_state_dim()))
        scene = np.zeros(E, np.int32)
        for c, s in enumerate(self.samplers):
            sel = np.flatnonzero(config == c)
            if len(sel) == 0:
                continue
            p, l, sc = s.sample_numpy(env[sel], ep[sel])
            pose[sel, :s.M] = p[:, :s.M]
            pose[sel, self.M:self.M + s.N] = p[:, s.M:]
            light[sel] = l
            scene[sel] = sc if s.shuffle else s.perm_scene[0]
        if K == 1 and not self.samplers[0].shuffle and env_scene is not None:
            scene = np.asarray(env_scene, np.int32).reshape(E).copy()   # one configuration: the env keeps its scene
        return pose, light, scene, config
