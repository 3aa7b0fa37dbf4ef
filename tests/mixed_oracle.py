"""The CPU reference for batches whose scenes differ in their numbers of objects and kilobots.

In the reference every env owns its own b2World, so the reference of a mixed batch is one compact oracle world per env,
built from that env's scene alone (an unchanged `oracle.kbo.OracleBatch` of one env).  `MixedOracle` drives them with the
padded-layout inputs of include/kb_b200.h (kb_create) and reports everything in that layout, with the library's values
for the rows of absent bodies: NaN observations, the canonical body state (all zero, xf.q.c = 1), zero mass data,
controllers and fat AABBs.  Its methods mirror OracleBatch / NativeBatch, so parity_util.assert_same_state applies.

A scene switch (set_env_scene) takes effect at the env's next reset, which rebuilds that env's world; its task
statistics then restart (the test that switches scenes does not use the task layer).
"""
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from gym_kilobots_b200 import _abi as abi


class MixedOracle:
    def __init__(self, kbo, scenes, num_envs, env_scene=None, max_contacts=0, threads=8):
        self.kbo = kbo
        self.scenes = list(scenes)
        self.E = num_envs
        self.next_scene = np.zeros(num_envs, np.int64) if env_scene is None else np.asarray(env_scene, np.int64).copy()
        self.scene = self.next_scene.copy()
        protos = [kbo.OracleBatch(sp, 1) for sp in self.scenes]
        self.M = max(sp.num_objects for sp in self.scenes)
        self.N = max(sp.num_kilobots for sp in self.scenes)
        self.B = self.M + self.N
        self.P = max(p.P for p in protos)
        self.L, self.A = protos[0].L, protos[0].A
        # contact capacity of the whole batch (kb_create's rule on the padded sizes), given to every env's world
        P = self.P
        if max_contacts > 0:
            C = max_contacts
        elif max_contacts < 0:
            C = max(P * (P - 1) // 2, 4)
        else:
            C = min(P * (P - 1) // 2, 8 * self.B + 32)
        self.C = min((C + 3) & ~3, 65532)
        self._mass = np.zeros((len(self.scenes), self.B, 4), np.float32)
        for s, p in enumerate(protos):
            self._mass[s] = self._pad_bodies(p.mass_data()[0], s, 0.0)
            p.close()
        self.task, self.targets, self.obs_flat = None, np.zeros((num_envs, 3)), None
        self.envs = [self._make(e) for e in range(num_envs)]
        self.pool = ThreadPoolExecutor(max(1, threads))   # ctypes releases the GIL: the env worlds step in parallel

    # ---- layout helpers
    def _counts(self, s):
        return self.scenes[s].num_objects, self.scenes[s].num_kilobots

    def _rows(self, s):
        M, N = self._counts(s)
        return np.r_[np.arange(M), self.M + np.arange(N)]

    def _pad_bodies(self, compact, s, fill):
        out = np.full((self.B,) + compact.shape[1:], fill, compact.dtype)
        out[self._rows(s)] = compact
        return out

    def _make(self, e):
        ob = self.kbo.OracleBatch(self.scenes[self.scene[e]], 1, None, self.C)
        if self.task is not None:
            ob.set_task(self.task, self.targets[e:e + 1])
        if self.obs_flat is not None:
            ob.bind_flat_observation()
        return ob

    def _map(self, f):
        return list(self.pool.map(f, range(self.E)))

    def close(self):
        for ob in self.envs:
            ob.close()
        self.pool.shutdown()

    # ---- the batched API in the padded layout
    def body_counts(self):
        c = np.array([self._counts(s) for s in self.scene], np.int32).reshape(self.E, 2)
        return c[:, 0].copy(), c[:, 1].copy()

    def set_env_scene(self, env_scene):
        self.next_scene = np.asarray(env_scene, np.int64).reshape(self.E).copy()

    def set_task(self, task, targets=None):
        if task.mode == abi.KB_TASK_OBJECT_TO_TARGET:
            assert 0 <= task.object < min(sp.num_objects for sp in self.scenes), "object index that some scene lacks"
        self.task = task
        if targets is not None:
            self.targets = np.asarray(targets, np.float64).reshape(self.E, 3).copy()
        for e, ob in enumerate(self.envs):
            ob.set_task(task, self.targets[e:e + 1])

    def bind_flat_observation(self, enable=True):
        self.obs_flat = np.full((self.E, 2 * self.N + self.L + 4 * self.M), np.nan, np.float32) if enable else None
        for ob in self.envs:
            ob.bind_flat_observation(enable)
        return self.obs_flat

    def reset(self, body_pose, light_state=None, kb_velocity=None, mask=None):
        pose = np.asarray(body_pose, np.float64).reshape(self.E, self.B, 3)
        light = None if light_state is None else np.asarray(light_state, np.float64).reshape(self.E, self.L)
        vel = None if kb_velocity is None else np.asarray(kb_velocity, np.float64).reshape(self.E, self.N, 2)

        def one(e):
            if mask is not None and not mask[e]:
                return
            if self.next_scene[e] != self.scene[e]:
                self.envs[e].close()
                self.scene[e] = self.next_scene[e]
                self.envs[e] = self._make(e)
            s = self.scene[e]
            self.envs[e].reset(pose[e, self._rows(s)][None], None if light is None else light[e:e + 1],
                               None if vel is None else vel[e, :self._counts(s)[1]][None])
        self._map(one)

    def step(self, action=None, mode=None):
        act = None if action is None else np.asarray(action, np.float64).reshape(self.E, -1)
        kilobot_mode = mode == abi.KB_ACTION_KILOBOTS

        def one(e):
            a = None
            if act is not None:
                a = act[e, :2 * self._counts(self.scene[e])[1]] if kilobot_mode else act[e]
                a = np.ascontiguousarray(a)[None]
            return self.envs[e].step(a, mode)
        outs = self._map(one)
        res = {"kilobots": np.full((self.E, self.N, 3), np.nan, np.float32),
               "objects": np.full((self.E, self.M, 3), np.nan, np.float32)}
        for k in ("light", "reward", "done", "status"):
            res[k] = np.concatenate([o[k] for o in outs])
        for e, o in enumerate(outs):
            M, N = self._counts(self.scene[e])
            res["kilobots"][e, :N] = o["kilobots"][0]
            res["objects"][e, :M] = o["objects"][0]
            if self.obs_flat is not None:
                f, L = self.envs[e].obs_flat[0], self.L
                row = self.obs_flat[e]
                row[:] = np.nan
                row[:2 * N] = f[:2 * N]
                row[2 * self.N:2 * self.N + L] = f[2 * N:2 * N + L]
                row[2 * self.N + L:2 * self.N + L + 4 * M] = f[2 * N + L:]
        return res

    def bodies(self):
        canon = np.zeros(abi.KB_BODY_STATE_FLOATS, np.float32)
        canon[11] = 1.0
        out = np.tile(canon, (self.E, self.B, 1))
        for e, ob in enumerate(self.envs):
            out[e, self._rows(self.scene[e])] = ob.bodies()[0]
        return out

    def set_poses(self, pose, body_mask=None):
        pose = np.asarray(pose, np.float64).reshape(self.E, self.B, 3)
        for e, ob in enumerate(self.envs):
            r = self._rows(self.scene[e])
            m = None if body_mask is None else np.asarray(body_mask, np.uint8).reshape(self.E, self.B)[e, r][None]
            ob.set_poses(pose[e, r][None], m)

    def get_status(self):
        return np.concatenate([ob.get_status() for ob in self.envs])

    def contacts(self):
        cs = [ob.contacts() for ob in self.envs]
        return np.concatenate([c[0] for c in cs]), np.concatenate([c[1] for c in cs])

    def impulses(self):
        return np.concatenate([ob.impulses() for ob in self.envs])

    def counters(self):
        return np.concatenate([ob.counters() for ob in self.envs])

    def proxies(self):
        out = np.zeros((self.E, self.P, 4), np.float32)
        for e, ob in enumerate(self.envs):
            out[e, :ob.P] = ob.proxies()[0]
        return out

    def controllers(self):
        ctrl = np.zeros((self.E, self.N, 4), np.float64)
        light = np.zeros((self.E, self.L), np.float64)
        for e, ob in enumerate(self.envs):
            c, l = ob.controllers()
            ctrl[e, :c.shape[1]] = c[0]
            light[e] = l[0]
        return ctrl, light

    def mass_data(self):
        return self._mass.copy()

    def episode_stats(self):
        return np.concatenate([ob.episode_stats() for ob in self.envs])

    def render(self, env_ids=(0,), width=1200, height=900):
        return np.concatenate([self.envs[int(e)].render((0,), width, height) for e in env_ids])
