"""Synthetic scene batches for the BASELINE.json configurations (SURVEY.md section 8d).

Each builder returns a `Scenario`: scene template(s), the env->scene map and seeded float64 initial
poses / light states for E environments.  Sampling mirrors the reference's scene builders
(gym_kilobots/envs/yaml_kilobots_env.py:194-198,256-265,327-354 and
envs/kilobots_test_envs.py:23-82) but is vectorised over E and uses a seeded numpy Generator keyed
by the global env id, so a slice of a batch (one rank of N) sees the same per-env draws.
"""
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import _abi as abi
from . import philox as PX
from . import scene as S


@dataclass
class Scenario:
    name: str
    scenes: List[S.SceneSpec]
    env_scene: Optional[np.ndarray]
    body_pose: np.ndarray          # [E, B, 3] float64 (m, m, rad)
    light_state: np.ndarray        # [E, L] float64
    max_contacts: int = 0

    @property
    def num_envs(self):
        return self.body_pose.shape[0]


def _rng_for(seed, env_ids):
    """Independent per-env streams: results do not depend on how envs are split across ranks."""
    return [np.random.Generator(np.random.Philox(key=seed, counter=[0, 0, 0, int(i)])) for i in env_ids]


def _separated_gaussian(rngs, mean, std, n, lo, hi, min_dist, max_tries=200):
    """[E, n, 2] positions ~ N(mean, std^2), clipped to [lo, hi], pairwise >= min_dist (rejection)."""
    E = len(rngs)
    out = np.zeros((E, n, 2))
    for e, rng in enumerate(rngs):
        pts = out[e]
        for k in range(n):
            for _ in range(max_tries):
                p = rng.normal(scale=std, size=2) + mean[e]
                p = np.minimum(np.maximum(p, lo), hi)
                if k == 0 or np.all(np.hypot(pts[:k, 0] - p[0], pts[:k, 1] - p[1]) >= min_dist):
                    break
            pts[k] = p
    return out


def _separated_gaussian_vec(rng, mean, std, n, lo, hi, min_dist, max_tries=200):
    """Same distribution as `_separated_gaussian`, vectorised over the envs with counter-based draws (`philox.EnvRng`):
    try t of kilobot k of env e is draw (stream KILOBOT_POS, index k * max_tries + t) of that env, whatever the batch."""
    E = len(mean)
    out = np.zeros((E, n, 2))
    for k in range(n):
        pending = np.arange(E)
        for t in range(max_tries):
            z0, z1 = rng.normal2(PX.STREAM_KILOBOT_POS, k * max_tries + t, sel=pending)
            p = np.stack([z0, z1], axis=-1) * std + mean[pending]
            p = np.minimum(np.maximum(p, lo), hi)
            if k == 0 or t == max_tries - 1:
                ok = np.ones(len(pending), bool)
            else:
                prev = out[pending, :k]
                ok = np.all(np.hypot(prev[..., 0] - p[:, None, 0], prev[..., 1] - p[:, None, 1]) >= min_dist, axis=1)
            out[pending[ok], k] = p[ok]
            pending = pending[~ok]
            if len(pending) == 0:
                break
    return out


def _circular_light(radius, world_size):
    w, h = world_size
    bounds = (np.array([-w / 2, -h / 2]) * 1.1, np.array([w / 2, h / 2]) * 1.1)   # yaml_kilobots_env.py:270
    return S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=radius, bounds=bounds,
                       action_bounds=(np.array([-1, -1]) * .01, np.array([1, 1]) * .01))  # :280


def c1_single_env(num_envs=1, seed=0, env_offset=0, kilobot_kind=abi.KB_KILOBOT_PHOTOTAXIS, **scene_kw):
    """C1: 10 phototaxis kilobots + 1 square object + circular gradient light (YamlKilobotsEnv-style)."""
    world = (2.0, 1.5)
    sc = S.SceneSpec(bodies=[S.quad_body(.15, .15)] + [S.kilobot_body(kilobot_kind) for _ in range(10)],
                     num_objects=1, lights=[_circular_light(.2, world)], world_size=world, **scene_kw)
    rngs = _rng_for(seed, range(env_offset, env_offset + num_envs))
    wb = np.array([world[0] / 2, world[1] / 2])
    light = np.stack([(r.random(2) * 2 * wb - wb) * 0.9 for r in rngs])
    kb = _separated_gaussian(rngs, light, 0.03, 10, -wb + 0.02, wb - 0.02, 2 * S.KILOBOT_RADIUS + 1e-3)
    pose = np.zeros((num_envs, 11, 3))
    pose[:, 1:, :2] = kb
    return Scenario("C1", [sc], None, pose, light, max_contacts=128)


def c2_quad_assembly(num_envs=4096, seed=0, env_offset=0, degenerate=True, **scene_kw):
    """C2: QuadAssemblyKilobotsEnv (kilobots_test_envs.py:23-82): 15 PhototaxisKilobots + 4 CornerQuads.

    degenerate=True reproduces the reference spawn (3 coincident copies of a 5-point cross);
    degenerate=False is C2' (same scene, kilobots ~ N(S, 0.03^2) rejection-separated)."""
    world = (2.0, 1.5)
    sc = S.SceneSpec(bodies=[S.quad_body(.15, .15) for _ in range(4)] +
                     [S.kilobot_body(abi.KB_KILOBOT_PHOTOTAXIS) for _ in range(15)],
                     num_objects=4, lights=[S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=.2)], world_size=world,
                     reward_const=1.0, **scene_kw)
    rngs = _rng_for(seed, range(env_offset, env_offset + num_envs))
    swarm = np.stack([np.array([-.95, -.7]) + r.random(2) * np.array([.9, 1.4]) for r in rngs])
    obj = np.stack([np.array([.05, -.7]) + r.random(2) * np.array([.9, .65]) for r in rngs])
    pose = np.zeros((num_envs, 19, 3))
    pose[:, 0] = (.45, .605, 0.0)
    pose[:, 1] = (.605, .605, -np.pi / 2)
    pose[:, 2] = (.605, .45, -np.pi)
    pose[:, 3, :2] = obj
    pose[:, 3, 2] = -np.pi / 2
    if degenerate:
        offs = np.array([(.0, .0), (.03, .0), (.0, .03), (-.03, .0), (.0, -.03)] * 3)
        pose[:, 4:, :2] = swarm[:, None, :] + offs[None]
    else:
        wb = np.array([world[0] / 2, world[1] / 2])
        pose[:, 4:, :2] = _separated_gaussian(rngs, swarm, 0.03, 15, -wb + 0.02, wb - 0.02,
                                              2 * S.KILOBOT_RADIUS + 1e-3)
    return Scenario("C2" if degenerate else "C2'", [sc], None, pose, swarm.copy(), max_contacts=160)


def c3_shapes(num_envs=8192, seed=0, env_offset=0, num_kilobots=50, **scene_kw):
    """C3: 50 kilobots + 1 object of shape [LForm, Triangle, Circle][env_id % 3]."""
    world = (2.0, 1.5)
    kb = [S.kilobot_body(abi.KB_KILOBOT_PHOTOTAXIS) for _ in range(num_kilobots)]
    objs = [S.polygon_body(S.LFORM_TEMPLATE, .15, .15), S.polygon_body(S.TRIANGLE_TEMPLATE, .15, .15), S.circle_body(.075)]
    scenes = [S.SceneSpec(bodies=[o] + kb, num_objects=1, lights=[_circular_light(.2, world)], world_size=world,
                          **scene_kw) for o in objs]
    ids = np.arange(env_offset, env_offset + num_envs)
    rng = PX.EnvRng(seed, ids)
    wb = np.array([world[0] / 2, world[1] / 2])
    u0, u1 = rng.uniform2(PX.STREAM_LIGHT, 0)
    light = (np.stack([u0, u1], axis=-1) * 2 * wb - wb) * 0.9
    pose = np.zeros((num_envs, 1 + num_kilobots, 3))
    u0, u1 = rng.uniform2(PX.STREAM_OBJECT, 0)
    pose[:, 0, :2] = (np.stack([u0, u1], axis=-1) * 2 * wb - wb) * 0.7       # yaml_kilobots_env.py:194-198
    pose[:, 0, 2] = rng.uniform2(PX.STREAM_OBJECT, 1)[0] * 2 * np.pi - np.pi
    pose[:, 1:, :2] = _separated_gaussian_vec(rng, light, 0.06, num_kilobots, -wb + 0.02, wb - 0.02,
                                              2 * S.KILOBOT_RADIUS + 1e-3)
    pose[:, 1:, 2] = rng.uniform2(PX.STREAM_KILOBOT_ANGLE, np.arange(num_kilobots)[None, :])[0] * 2 * np.pi - np.pi
    return Scenario("C3", scenes, (ids % 3).astype(np.int32), pose, light, max_contacts=320)


def c5_small(num_envs=1 << 20, seed=0, env_offset=0, **scene_kw):
    """C5: 4 kilobots + 1 Quad(0.15, 0.15); throughput sweep.  Vectorised counter-based sampling (E is large):
    a rank's slice of the 2^20 envs draws exactly what the same global env ids draw in a single-GPU batch."""
    world = (2.0, 1.5)
    sc = S.SceneSpec(bodies=[S.quad_body(.15, .15)] + [S.kilobot_body(abi.KB_KILOBOT_PHOTOTAXIS) for _ in range(4)],
                     num_objects=1, lights=[_circular_light(.2, world)], world_size=world, **scene_kw)
    rng = PX.EnvRng(seed, np.arange(env_offset, env_offset + num_envs))
    wb = np.array([world[0] / 2, world[1] / 2])
    u0, u1 = rng.uniform2(PX.STREAM_LIGHT, 0)
    light = (np.stack([u0, u1], axis=-1) * 2 * wb - wb) * 0.9
    pose = np.zeros((num_envs, 5, 3))
    u0, u1 = rng.uniform2(PX.STREAM_OBJECT, 0)
    pose[:, 0, :2] = (np.stack([u0, u1], axis=-1) * 2 * wb - wb) * 0.7
    pose[:, 0, 2] = rng.uniform2(PX.STREAM_OBJECT, 1)[0] * 2 * np.pi - np.pi
    # SURVEY 8(d): kilobots ~ N(L0, 0.03^2), clipped, rejection-separated (yaml_kilobots_env.py:346-352)
    pose[:, 1:, :2] = _separated_gaussian_vec(rng, light, 0.03, 4, -wb + 0.02, wb - 0.02, 2 * S.KILOBOT_RADIUS + 1e-3)
    pose[:, 1:, 2] = rng.uniform2(PX.STREAM_KILOBOT_ANGLE, np.arange(4)[None, :])[0] * 2 * np.pi - np.pi
    return Scenario("C5", [sc], None, pose, light, max_contacts=32)


def c4_swarm(num_envs=256, seed=0, env_offset=0, side=32, **scene_kw):
    """C4 (SURVEY 8d): side^2 PhototaxisKilobots on a side x side lattice of pitch 0.036 m centred at the origin,
    U(+-0.001 m) jitter, headings U(-pi, pi); one CircularGradientLight of radius 0.8 m at the origin and the zero
    action, so the whole swarm pushes inward: dense persistent contacts (large-swarm tier, grid broadphase)."""
    world = (2.0, 1.5)
    n = side * side
    sc = S.SceneSpec(bodies=[S.kilobot_body(abi.KB_KILOBOT_PHOTOTAXIS) for _ in range(n)], num_objects=0,
                     lights=[_circular_light(.8, world)], world_size=world, **scene_kw)
    rng = PX.EnvRng(seed, np.arange(env_offset, env_offset + num_envs))
    g = (np.arange(side) - (side - 1) / 2.0) * 0.036
    lattice = np.stack(np.meshgrid(g, g, indexing="xy"), axis=-1).reshape(n, 2)
    idx = np.arange(n)[None, :]
    j0, j1 = rng.uniform2(PX.STREAM_KILOBOT_POS, idx)
    pose = np.zeros((num_envs, n, 3))
    pose[:, :, :2] = lattice[None] + (np.stack([j0, j1], axis=-1) * 2.0 - 1.0) * 0.001
    pose[:, :, 2] = rng.uniform2(PX.STREAM_KILOBOT_ANGLE, idx)[0] * 2 * np.pi - np.pi
    light = np.zeros((num_envs, 2))
    return Scenario("C4", [sc], None, pose, light, max_contacts=0)


def swarm_corner(num_envs=8, n=48, seed=0, env_offset=0, kilobot_kind=abi.KB_KILOBOT_PHOTOTAXIS, light_radius=.4,
                 spread=.05, world=(1.0, 0.5), corner=True, **scene_kw):
    """Kilobots only (no pushable object): a swarm next to the bottom-left corner of a small table with the light
    beyond the corner, so that it jams against two table edges (wall contacts, continuous collision, dense
    kilobot-kilobot contacts); corner=False spreads it over the table under a small light instead (most kilobots
    see no gradient: sleeping islands that the moving light wakes again).  Used to cross-check the large-swarm
    tier against the lane-group kernels and the oracle."""
    wb = np.array([world[0] / 2, world[1] / 2])
    bounds = (-wb * 1.1, wb * 1.1)
    act = (np.array([-1, -1]) * .01, np.array([1, 1]) * .01)
    sc = S.SceneSpec(bodies=[S.kilobot_body(kilobot_kind) for _ in range(n)], num_objects=0,
                     lights=[S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=light_radius, bounds=bounds, action_bounds=act)],
                     world_size=world, **scene_kw)
    rng = PX.EnvRng(seed, np.arange(env_offset, env_offset + num_envs))
    u0, u1 = rng.uniform2(PX.STREAM_SWARM, 0)
    jit = (np.stack([u0, u1], axis=-1) - 0.5) * 0.04
    if corner:
        centre = -wb + np.array([0.09, 0.09]) + jit
        light = np.tile(-wb * 1.05, (num_envs, 1)) + jit
    else:
        centre = jit * 5.0
        light = centre + np.array([0.1, 0.05])
    pose = np.zeros((num_envs, n, 3))
    pose[:, :, :2] = _separated_gaussian_vec(rng, centre, spread, n, -wb + 0.02, wb - 0.02, 2 * S.KILOBOT_RADIUS + 1e-3)
    pose[:, :, 2] = rng.uniform2(PX.STREAM_KILOBOT_ANGLE, np.arange(n)[None, :])[0] * 2 * np.pi - np.pi
    return Scenario("swarm-corner" if corner else "swarm-spread", [sc], None, pose, light, max_contacts=0)


def stack_poses(specs, env_scene, poses):
    """Stack per-env body poses into the padded body layout of a batch over `specs` (include/kb_b200.h kb_create).

    poses[e] is [B_e, 3] for the scene specs[env_scene[e]]: its objects, then its kilobots.  The result is float64
    [E, Mmax + Nmax, 3], Mmax / Nmax the largest object / kilobot counts of `specs`: object j of env e at row j, kilobot
    k at row Mmax + k, zeros at the rows the env's scene does not populate (absent bodies).  A batch whose scenes all
    have the same counts is stacked unchanged."""
    Mmax = max(sp.num_objects for sp in specs)
    Nmax = max(sp.num_kilobots for sp in specs)
    out = np.zeros((len(poses), Mmax + Nmax, 3))
    for e, (s, p) in enumerate(zip(env_scene, poses)):
        sp = specs[int(s)]
        p = np.asarray(p, dtype=np.float64).reshape(sp.num_bodies, 3)
        out[e, :sp.num_objects] = p[:sp.num_objects]
        out[e, Mmax:Mmax + sp.num_kilobots] = p[sp.num_objects:]
    return out


def from_envs(envs, name="from_envs"):
    """Vectorise reference-style environments: every element of `envs` is a KilobotsEnv subclass instance
    (YamlKilobotsEnv(configuration=...), QuadAssemblyKilobotsEnv(), a user's own subclass ...).  Each one's
    `_configure_environment` is run once, exactly as `reset()` would (kilobots_env.py:150-156), including its
    random initialisation; the recorded scenes are de-duplicated into templates and the poses stacked.
    All envs must have the same light layout; their numbers of objects and kilobots may differ (the poses and
    kb_velocity are stacked in the padded body layout, see `stack_poses`)."""
    from .envs.kilobots_env import KilobotsEnv
    specs, keys, env_scene, poses, lights, vels = [], {}, [], [], [], []
    for env in envs:
        spec, pose, light, vel = env._record_scene()
        k = KilobotsEnv._spec_key(spec)
        if k not in keys:
            keys[k] = len(specs)
            specs.append(spec)
        env_scene.append(keys[k])
        poses.append(pose)
        lights.append(np.zeros(0) if light is None else np.asarray(light, float))
        vels.append(vel)
    for sp in specs:
        if sp.light_state_dim != specs[0].light_state_dim:
            raise ValueError("from_envs: all environments must agree in their light layout")
    sc = Scenario(name, specs, np.asarray(env_scene, np.int32), stack_poses(specs, env_scene, poses), np.stack(lights))
    Nmax = max(sp.num_kilobots for sp in specs)
    sc.kb_velocity = None
    if any(v is not None for v in vels):
        sc.kb_velocity = np.zeros((len(vels), Nmax, 2))
        for e, v in enumerate(vels):
            if v is not None:
                sc.kb_velocity[e, :len(v)] = v
    return sc


def random_actions(scenario_or_dim, num_envs, steps, seed=1):
    """i.i.d. U([-0.01, 0.01]^A) per env-step: mirrors env.action_space.sample() (gym_kilobots/test.py:25)."""
    A = scenario_or_dim if isinstance(scenario_or_dim, int) else scenario_or_dim.scenes[0].action_dim
    rng = np.random.Generator(np.random.Philox(key=seed))
    return rng.uniform(-0.01, 0.01, size=(steps, num_envs, A))


# ----------------------------------------------------------------------------------------------
# Extra parity scenes: they exercise the rest of the reference's hot-path surface (every object shape of
# lib/body.py:288-334, object-object and object-table contacts, the other controllers and lights).
def pushing_yard(num_envs=16, seed=0, env_offset=0, kilobot_kind=abi.KB_KILOBOT_SIMPLE_PHOTOTAXIS, num_kilobots=12,
                 light="momentum", **scene_kw):
    """A small 1.0 x 0.5 m arena (QuadPushingEnv's size, kilobots_test_envs.py:12) crowded with one object of
    every shape and a swarm that follows a moving light: objects are pushed into each other and into the table."""
    world = (1.0, 0.5)
    objs = [S.quad_body(.1, .1), S.polygon_body(S.TFORM_TEMPLATE, .12, .12), S.polygon_body(S.CFORM_TEMPLATE, .12, .12),
            S.polygon_body(S.LFORM_TEMPLATE, .12, .12), S.polygon_body(S.TRIANGLE_TEMPLATE, .12, .12), S.circle_body(.04)]
    wb = np.array([world[0] / 2, world[1] / 2])
    bounds = (-wb * 1.1, wb * 1.1)
    act = (np.array([-1, -1]) * .01, np.array([1, 1]) * .01)
    if light == "momentum":
        lights = [S.LightSpec(abi.KB_LIGHT_MOMENTUM, radius=.3, bounds=bounds, action_bounds=act, max_velocity=.01)]
    elif light == "composite":
        lights = [S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=.25, bounds=bounds, action_bounds=act),
                  S.LightSpec(abi.KB_LIGHT_MOMENTUM, radius=.2, bounds=bounds, action_bounds=act, max_velocity=.01)]
    elif light == "linear":
        lights = [S.LightSpec(abi.KB_LIGHT_LINEAR, action_bounds=(np.array([-2 * np.pi, 0.]), np.array([2 * np.pi, 0.])))]
    else:
        lights = [S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=.3, bounds=bounds, action_bounds=act)]
    sc = S.SceneSpec(bodies=objs + [S.kilobot_body(kilobot_kind) for _ in range(num_kilobots)], num_objects=len(objs),
                     lights=lights, world_size=world, **scene_kw)
    rngs = _rng_for(seed, range(env_offset, env_offset + num_envs))
    M = len(objs)
    pose = np.zeros((num_envs, M + num_kilobots, 3))
    slots = np.array([(-.36, .13), (-.2, -.1), (-.03, .12), (.13, -.1), (.28, .1), (.4, -.12)])
    for e, r in enumerate(rngs):
        pose[e, :M, :2] = slots + r.uniform(-.015, .015, size=(M, 2))
        pose[e, :M, 2] = r.uniform(-np.pi, np.pi, size=M)
    centre = np.stack([r.uniform(-.3, .3, size=2) * np.array([1.0, .4]) for r in rngs])
    pose[:, M:, :2] = _separated_gaussian(rngs, centre, 0.08, num_kilobots, -wb + 0.02, wb - 0.02,
                                          2 * S.KILOBOT_RADIUS + 1e-3)
    for e, r in enumerate(rngs):
        pose[e, M:, 2] = r.uniform(-np.pi, np.pi, size=num_kilobots)
    ls = []
    for e, r in enumerate(rngs):
        row = []
        for l in lights:
            if l.type == abi.KB_LIGHT_MOMENTUM:
                row += list(centre[e]) + [0.0, 0.0]
            elif l.type == abi.KB_LIGHT_LINEAR:
                row += [float(r.uniform(-np.pi, np.pi))]
            else:
                row += list(centre[e] + r.uniform(-.05, .05, size=2))
        ls.append(row)
    return Scenario("yard-%s" % light, [sc], None, pose, np.asarray(ls, dtype=np.float64), max_contacts=176)


def direct_control(num_envs=16, seed=0, env_offset=0, **scene_kw):
    """DirectControlKilobotsEnv-style batch (envs/direct_control_kilobots_env.py): velocity- and
    acceleration-controlled kilobots around a quad, actions [E, N, 2] routed to Kilobot.set_action."""
    world = (1.0, 0.5)
    kinds = [abi.KB_KILOBOT_VELOCITY, abi.KB_KILOBOT_ACCELERATION] * 4
    sc = S.SceneSpec(bodies=[S.quad_body(.1, .1), S.circle_body(.05)] + [S.kilobot_body(k) for k in kinds], num_objects=2,
                     lights=[], world_size=world, **scene_kw)
    rngs = _rng_for(seed, range(env_offset, env_offset + num_envs))
    wb = np.array([world[0] / 2, world[1] / 2])
    pose = np.zeros((num_envs, 2 + len(kinds), 3))
    pose[:, 0, :2] = (-.12, 0.0)
    pose[:, 1, :2] = (.12, 0.0)
    ring = np.array([(np.cos(a), np.sin(a)) for a in np.linspace(0, 2 * np.pi, len(kinds), endpoint=False)]) * .2
    ring[:, 1] *= .6
    for e, r in enumerate(rngs):
        pose[e, 2:, :2] = np.minimum(np.maximum(ring + r.uniform(-.01, .01, size=ring.shape), -wb + 0.02), wb - 0.02)
        pose[e, 2:, 2] = r.uniform(-np.pi, np.pi, size=len(kinds))
    return Scenario("direct", [sc], None, pose, np.zeros((num_envs, 0)), max_contacts=64)


def random_kilobot_actions(scenario, num_envs, steps, seed=2):
    """[steps, E, N, 2]: (v, omega) or (dv, domega) samples wide enough to hit the clips of
    lib/kilobot.py:216-218,269."""
    N = scenario.scenes[0].num_kilobots
    rng = np.random.Generator(np.random.Philox(key=seed))
    a = np.zeros((steps, num_envs, N, 2))
    a[..., 0] = rng.uniform(-0.004, 0.014, size=(steps, num_envs, N))
    a[..., 1] = rng.uniform(-2.0, 2.0, size=(steps, num_envs, N))
    return a.reshape(steps, num_envs, 2 * N)
