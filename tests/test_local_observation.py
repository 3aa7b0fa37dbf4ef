"""Per-kilobot local observations (include/kb_b200.h kb_local_observation, csrc/kb_local.cuh): the numpy mirror
(gym_kilobots_b200/local_obs.py) against a float64 k-d tree and hand-built lattices on the CPU, then both kernels (a warp
per env, and the uniform grid of large swarms) against the mirror on the GPU, bit for bit except the light part
(float64 rounded to float32; within 1 ulp)."""
import itertools

import numpy as np
import pytest

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import scenarios as SC
from gym_kilobots_b200 import scene as S
from gym_kilobots_b200.local_obs import local_observation_numpy
from gym_kilobots_b200.scene import LocalObsSpec

ALL_PARTS = [dict(neighbours=a, objects=b, light=c) for a, b, c in itertools.product([True, False], repeat=3) if a or b or c]


# ------------------------------------------------------------------------------------------------------------ CPU
def _synthetic(pos, angle, obj_pos=None, obj_angle=None, kind=abi.KB_KILOBOT_PHOTOTAXIS, lights=None):
    """One env: bodies [1, B, 12] / obs arrays built the way kb_get_bodies and kb_step report a state."""
    n = len(pos)
    m = 0 if obj_pos is None else len(obj_pos)
    scene = S.SceneSpec(bodies=[S.quad_body(.1, .1)] * m + [S.kilobot_body(kind)] * n, num_objects=m,
                        lights=lights or [])
    xy = np.concatenate([np.zeros((0, 2)) if obj_pos is None else obj_pos, pos]) * 25.0
    ang = np.concatenate([np.zeros(0) if obj_angle is None else obj_angle, angle])
    bodies = np.zeros((1, m + n, 12), np.float32)
    bodies[0, :, 8:10] = xy.astype(np.float32)
    bodies[0, :, 10] = np.sin(ang).astype(np.float32)
    bodies[0, :, 11] = np.cos(ang).astype(np.float32)
    obs = (bodies[..., 8:10].astype(np.float64) / 25.0).astype(np.float32)
    return scene, bodies, obs[:, m:], obs[:, :m]


def test_mirror_neighbours_match_a_float64_kdtree():
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(0)
    n, r, K = 600, 0.1, 8
    pos = rng.uniform(-1, 1, (n, 2)) * np.array([1.0, 0.75])
    scene, bodies, kb, ob = _synthetic(pos, rng.uniform(-np.pi, np.pi, n))
    spec = LocalObsSpec(r, max_neighbours=K, objects=False)
    out = local_observation_numpy(spec, bodies, kb, ob, np.zeros((1, 0)), [scene])[0]
    p = kb[0].astype(np.float64)
    tree = cKDTree(p)
    eps = 8 * np.spacing(np.float32(r))
    checked = 0
    for i in range(n):
        d = np.hypot(*(p - p[i]).T)
        d[i] = np.inf
        if np.any(np.abs(d - r) < eps):
            continue   # a pair within a few ulp of the radius: float32 and float64 may disagree
        near = sorted(j for j in tree.query_ball_point(p[i], r) if j != i)
        assert out[i, 0] == len(near)
        want = np.sort(d[near])[:K]
        got = out[i, 1:].reshape(K, 4)
        assert np.allclose(got[:len(want), 2], want, rtol=1e-6, atol=0)
        assert np.allclose(np.hypot(got[:len(want), 0], got[:len(want), 1]), want, rtol=1e-5)
        assert np.all(got[:len(want), 3] == 1) and np.all(got[len(want):] == 0)
        checked += 1
    assert checked > 0.95 * n


def test_mirror_orders_ties_by_padded_index():
    """An exact lattice (pitch 1/16 m: every d2 is exact) with many equidistant neighbours, heading 0: slot order is
    ascending (d2, j), ties going to the lower padded index."""
    g = np.arange(-3, 4) / 16.0
    pos = np.stack(np.meshgrid(g, g, indexing="xy"), -1).reshape(-1, 2)
    perm = np.random.default_rng(2).permutation(len(pos))
    pos = pos[perm]                               # padded indices unrelated to geometry
    scene, bodies, kb, ob = _synthetic(pos, np.zeros(len(pos)))
    K = 24
    out = local_observation_numpy(LocalObsSpec(0.2, max_neighbours=K, objects=False), bodies, kb, ob, np.zeros((1, 0)),
                                  [scene])[0]
    centre = int(np.flatnonzero((pos == 0).all(1))[0])
    slots = out[centre, 1:].reshape(K, 4)
    lookup = {(round(x * 16), round(y * 16)): j for j, (x, y) in enumerate(pos)}
    js = [lookup[(round(float(x) * 16), round(float(y) * 16))] for x, y in slots[:, :2]]
    d2 = [(pos[j] ** 2).sum() for j in js]
    assert js == sorted(js, key=lambda j: ((pos[j] ** 2).sum(), j))
    expect = sorted((((pos[j] ** 2).sum(), j) for j in range(len(pos)) if j != centre and (pos[j] ** 2).sum() <= 0.04))
    assert out[centre, 0] == len(expect) and [j for _, j in expect[:K]] == js and len(set(d2)) < K


@pytest.mark.parametrize("parts", ALL_PARTS, ids=lambda p: "-".join(k for k, v in p.items() if v))
def test_layout_and_dim_of_every_combination(parts):
    rng = np.random.default_rng(3)
    light = [S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=.3)]
    scene, bodies, kb, ob = _synthetic(rng.uniform(-.2, .2, (12, 2)), rng.uniform(-3, 3, 12), rng.uniform(-.2, .2, (3, 2)),
                                       rng.uniform(-3, 3, 3), lights=light)
    full = LocalObsSpec(0.15, max_neighbours=5, neighbours=True, objects=True, light=True)
    spec = LocalObsSpec(0.15, max_neighbours=5, **parts)
    ls = np.array([[0.05, -0.02]])
    a = local_observation_numpy(full, bodies, kb, ob, ls, [scene])
    b = local_observation_numpy(spec, bodies, kb, ob, ls, [scene])
    widths = {"neighbours": 1 + 4 * 5, "objects": 5 * 3, "light": 3}
    assert spec.dim(3) == sum(widths[k] for k, v in parts.items() if v) == b.shape[-1]
    sl, fsl = spec.slices(3), full.slices(3)
    assert sorted(sl) == sorted(k for k, v in parts.items() if v)
    c = 0
    for name in ("neighbours", "objects", "light"):
        if name in sl:
            assert sl[name] == slice(c, c + widths[name])
            c += widths[name]
            assert np.array_equal(b[..., sl[name]], a[..., fsl[name]])
    assert np.isfinite(a).all()


def test_padded_batch_absent_kilobots_and_objects():
    rng = np.random.default_rng(4)
    small = S.SceneSpec(bodies=[S.quad_body(.1, .1)] + [S.kilobot_body(abi.KB_KILOBOT_PHOTOTAXIS)] * 3, num_objects=1)
    big = S.SceneSpec(bodies=[S.quad_body(.1, .1)] * 2 + [S.kilobot_body(abi.KB_KILOBOT_PHOTOTAXIS)] * 5, num_objects=2)
    M, N = 2, 5
    bodies = np.zeros((2, M + N, 12), np.float32)
    bodies[..., 8:10] = rng.uniform(-1, 1, (2, M + N, 2)).astype(np.float32)   # within 0.1 m of each other (b2 units)
    bodies[..., 11] = 1
    obs = (bodies[..., 8:10].astype(np.float64) / 25.0).astype(np.float32)
    kb, ob = obs[:, M:].copy(), obs[:, :M].copy()
    kb[0, 3:] = np.nan
    ob[0, 1:] = np.nan
    spec = LocalObsSpec(0.5, max_neighbours=6)
    out = local_observation_numpy(spec, bodies, kb, ob, np.zeros((2, 0)), [small, big], env_scene=[0, 1])
    assert np.isnan(out[0, 3:]).all() and np.isfinite(out[0, :3]).all() and np.isfinite(out[1]).all()
    assert np.all(out[0, :3, 0] == 2) and np.all(out[1, :, 0] == 4)      # absent kilobots are never neighbours
    o = spec.slices(M)["objects"]
    assert np.all(out[0, :3, o][:, 5:] == 0) and np.all(out[0, :3, o][:, 4] == 1)


@pytest.mark.parametrize("kw", [dict(neighbours=False, objects=False, light=False), dict(max_neighbours=0),
                                dict(max_neighbours=33), dict(radius=0.0), dict(radius=-1.0), dict(radius=np.nan),
                                dict(radius=np.inf), dict(radius=1e39)])
def test_spec_refusals(kw):
    args = dict(radius=0.1)
    args.update(kw)
    with pytest.raises(ValueError):
        LocalObsSpec(**args)


def test_mirror_refuses_parts_the_batch_lacks():
    scene, bodies, kb, ob = _synthetic(np.zeros((2, 2)), np.zeros(2))
    with pytest.raises(ValueError, match="objects"):
        local_observation_numpy(LocalObsSpec(0.1), bodies, kb, ob, np.zeros((1, 0)), [scene])
    with pytest.raises(ValueError, match="light"):
        local_observation_numpy(LocalObsSpec(0.1, objects=False, light=True), bodies, kb, ob, np.zeros((1, 0)), [scene])


# ------------------------------------------------------------------------------------------------------------ GPU
def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _state_obs(nb):
    """obs_kilobots / obs_objects / light state of the state the batch holds (what the next gather would report)."""
    b = nb.bodies()
    pos = (b[..., 8:10].astype(np.float64) / 25.0).astype(np.float32)
    return {"kilobots": pos[:, nb.M:], "objects": pos[:, :nb.M], "light": nb.controllers()[1]}


def _assert_matches(nb, spec, obs, got=None, where=""):
    if got is None:
        got = nb.local_observation(spec).cpu().numpy()
    scenes = nb.current_scenes().cpu().numpy()
    want = local_observation_numpy(spec, nb.bodies(), obs["kilobots"], obs["objects"], obs["light"], nb.scenes, scenes)
    assert got.shape == want.shape, where
    exact = np.ones(got.shape[-1], bool)
    if spec.light:
        exact[spec.slices(nb.M)["light"]] = False
        g, w = got[..., ~exact], want[..., ~exact]
        assert np.array_equal(np.isnan(g), np.isnan(w)), where
        ok = ~np.isnan(w)
        assert np.all(np.abs(g[ok] - w[ok]) <= np.spacing(np.abs(w[ok]).astype(np.float32))), where + ": light part"
    assert np.array_equal(_bits(got[..., exact]), _bits(want[..., exact])), where
    return got


def _run(nb, sc, spec, steps=4, actions=None, mode=None):
    nb.reset(sc.body_pose, sc.light_state)
    _assert_matches(nb, spec, _state_obs(nb), where="after reset")
    for t in range(steps):
        a = None if actions is None else actions[t]
        obs = nb.step(a, mode)
        _assert_matches(nb, spec, obs, where="after step %d" % t)


def _batch(native, sc):
    return native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c2", "c3", "yard-momentum", "yard-composite", "yard-linear", "direct"])
@pytest.mark.parametrize("K", [8, 20])
def test_lane_group_batches(native, case, K, monkeypatch):
    mode, acts = None, None
    if case == "c2":
        sc = SC.c2_quad_assembly(64, seed=1)
    elif case == "c3":
        sc = SC.c3_shapes(60, seed=2)
    elif case == "direct":
        sc = SC.direct_control(16)
        mode, acts = abi.KB_ACTION_KILOBOTS, SC.random_kilobot_actions(sc, 16, 4)
    else:
        sc = SC.pushing_yard(16, light=case.split("-")[1],
                             kilobot_kind=abi.KB_KILOBOT_PHOTOTAXIS if case.endswith("linear") else abi.KB_KILOBOT_SIMPLE_PHOTOTAXIS)
    if acts is None:
        acts = SC.random_actions(sc, sc.num_envs, 4)
    spec = LocalObsSpec(0.1, max_neighbours=K, light=bool(sc.scenes[0].lights))
    nb = _batch(native, sc)
    assert nb.launch_config()["lanes_per_env"] <= 32
    _run(nb, sc, spec, actions=acts, mode=mode)
    a = nb.local_observation(spec).cpu().numpy()
    monkeypatch.setenv("KB_LOCAL_FORCE_GRID", "1")
    b = nb.local_observation(spec).cpu().numpy()
    assert np.array_equal(_bits(a), _bits(b)), "grid and brute-force kernels differ"


def _heap(E=2, n=90):
    sc = SC.swarm_corner(E, n=n, spread=.07, corner=False)
    rng = np.random.default_rng(5)
    sc.body_pose[:, :, :2] = np.clip(rng.normal(0.0, 0.01, (E, n, 2)), -0.03, 0.03)
    sc.body_pose[0, 1, :2] = sc.body_pose[0, 0, :2]          # two exactly coincident kilobots: a d2 = 0 tie
    sc.body_pose[0, 2, :2] = sc.body_pose[0, 0, :2]
    sc.max_contacts = n * (n - 1) // 2 + 4 * n
    return sc


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c4-256", "c4-1024", "c4-1681", "heap"])
def test_swarm_tier(native, case):
    if case == "heap":
        sc = _heap()
    else:
        side = {"c4-256": 16, "c4-1024": 32, "c4-1681": 41}[case]
        sc = SC.c4_swarm(2 if side < 41 else 1, side=side)
    nb = _batch(native, sc)
    assert nb.launch_config()["lanes_per_env"] > 32
    for K in (8, 32):
        spec = LocalObsSpec(0.1, max_neighbours=K, objects=False, light=True)
        _run(nb, sc, spec, steps=2, actions=np.zeros((2, sc.num_envs, 2)))


@pytest.mark.gpu
def test_heap_coincident_ties_right_after_reset(native):
    sc = _heap()
    nb = _batch(native, sc)
    nb.reset(sc.body_pose, sc.light_state)
    nb.set_poses(sc.body_pose)   # no settle step after it: the coincident centres stay coincident
    spec = LocalObsSpec(0.05, max_neighbours=4, objects=False)
    got = _assert_matches(nb, spec, _state_obs(nb), where="coincident")
    slots = got[0, 0, 1:].reshape(4, 4)
    assert np.all(slots[:2, 2] == 0.0) and np.all(slots[:2, 3] == 1.0)   # kilobots 1 and 2 at distance 0, in index order


def _mixed_swarm():
    sizes = (10, 40, 100)
    homs = [SC.swarm_corner(3, n=n, spread=.05, corner=False, seed=i) for i, n in enumerate(sizes)]
    specs = [h.scenes[0] for h in homs]
    env_scene = np.array([e % 3 for e in range(9)], np.int32)
    poses = [homs[e % 3].body_pose[e // 3] for e in range(9)]
    light = np.stack([homs[e % 3].light_state[e // 3] for e in range(9)])
    return SC.Scenario("mixed", specs, env_scene, SC.stack_poses(specs, env_scene, poses), light)


@pytest.mark.gpu
def test_mixed_batch(native, monkeypatch):
    sc = _mixed_swarm()
    nb = _batch(native, sc)
    spec = LocalObsSpec(0.5, max_neighbours=32, objects=False, light=True)
    _run(nb, sc, spec, steps=3, actions=np.zeros((3, sc.num_envs, 2)))
    got = nb.local_observation(spec).cpu().numpy()
    n = np.array([10, 40, 100] * 3)
    present = np.arange(nb.N)[None, :] < n[:, None]
    assert np.isnan(got[~present]).all() and np.isfinite(got[present]).all()
    assert np.all(got[present][:, 0] <= np.repeat(n, n) - 1)     # absent kilobots are never neighbours


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [5.0, 1e-4, 0.03])
def test_radius_extremes_and_both_kernels(native, radius, monkeypatch):
    """A radius wider than the table (one grid cell), a tiny one (no neighbours), and K larger than every count; the
    grid kernel forced on a batch the warp kernel runs gives the same bits."""
    for sc in (SC.c3_shapes(12, seed=4, num_kilobots=40), SC.swarm_corner(3, n=100, spread=.07)):
        nb = _batch(native, sc)
        nb.reset(sc.body_pose, sc.light_state)
        obs = nb.step(SC.random_actions(sc, sc.num_envs, 1)[0])
        spec = LocalObsSpec(radius, max_neighbours=32, objects=nb.M > 0, light=True)
        monkeypatch.delenv("KB_LOCAL_FORCE_GRID", raising=False)
        a = _assert_matches(nb, spec, obs, where="radius %g" % radius)
        if radius == 5.0:
            assert np.all(a[..., 0][~np.isnan(a[..., 0])] == np.array([40, 100])[int(nb.N == 100)] - 1)
        if radius == 1e-4:
            assert np.all(a[..., 0] == 0)
        monkeypatch.setenv("KB_LOCAL_FORCE_GRID", "1")
        b = nb.local_observation(spec).cpu().numpy()
        assert np.array_equal(_bits(a), _bits(b))


@pytest.mark.gpu
def test_mask_keeps_unmasked_rows(native):
    import torch
    sc = SC.c2_quad_assembly(16, seed=3)
    nb = _batch(native, sc)
    nb.reset(sc.body_pose, sc.light_state)
    obs = nb.step(SC.random_actions(sc, 16, 1)[0])
    spec = LocalObsSpec(0.1)
    out = torch.full((nb.E, nb.N, nb.local_observation_dim(spec)), -7.0, dtype=torch.float32, device=nb.device)
    mask = (np.arange(16) % 3 == 0)
    nb.local_observation(spec, mask=torch.as_tensor(mask, device=nb.device), out=out)
    got = out.cpu().numpy()
    assert np.all(got[~mask] == -7.0)
    ref = _assert_matches(nb, spec, obs)
    assert np.array_equal(_bits(got[mask]), _bits(ref[mask]))


@pytest.mark.gpu
def test_side_stream_after_step_device(native):
    import torch
    sc = SC.c4_swarm(4, side=16)
    nb = _batch(native, sc)
    nb.reset(sc.body_pose, sc.light_state)
    spec = LocalObsSpec(0.1, objects=False, light=True)
    nb.step_device(torch.zeros((4, 2), dtype=torch.float64, device=nb.device))
    side = torch.cuda.Stream(device=nb.device)
    side.wait_stream(torch.cuda.current_stream(nb.device))
    with torch.cuda.stream(side):
        out = nb.local_observation(spec)
    side.synchronize()
    got = out.cpu().numpy()
    obs = {"kilobots": nb.obs_kilobots.cpu().numpy(), "objects": nb.obs_objects.cpu().numpy(),
           "light": nb.obs_light.cpu().numpy()}
    _assert_matches(nb, spec, obs, got=got)


@pytest.mark.gpu
def test_c_abi_refusals(native):
    sc = SC.direct_control(2)
    nb = _batch(native, sc)
    fn = native._fn
    import ctypes as C
    import torch
    out = torch.zeros((2, nb.N, 64), dtype=torch.float32, device=nb.device)
    p = C.c_void_p(out.data_ptr())

    def refuse(d, match, ptr=p):
        assert fn["local_observation"](nb.h, d, None, ptr, None) == -1     # KB_ERR_INVALID
        assert match in fn["last_error"]().decode()

    ok = abi.KbLocalObsDef(0.1, 8, abi.KB_LOCAL_NEIGHBOURS, 0)
    refuse(None, "null def")
    refuse(C.byref(ok), "null out", ptr=None)
    for parts in (0, 8, 9):
        refuse(C.byref(abi.KbLocalObsDef(0.1, 8, parts, 0)), "parts")
    for k in (0, 33):
        refuse(C.byref(abi.KbLocalObsDef(0.1, k, 1, 0)), "max_neighbours")
    for r in (0.0, -0.1, float("nan"), float("inf")):
        refuse(C.byref(abi.KbLocalObsDef(r, 8, 1, 0)), "radius")
    refuse(C.byref(abi.KbLocalObsDef(0.1, 8, abi.KB_LOCAL_LIGHT, 0)), "without lights")
    sw = SC.c4_swarm(1, side=8)
    nb2 = _batch(native, sw)
    assert fn["local_observation"](nb2.h, C.byref(abi.KbLocalObsDef(0.1, 8, abi.KB_LOCAL_OBJECTS, 0)), None, p, None) == -1
    assert "without objects" in fn["last_error"]().decode()
    assert fn["local_observation_dim"](nb.h, C.byref(ok)) == 33
    with pytest.raises(RuntimeError, match="without lights"):
        nb.local_observation_dim(LocalObsSpec(0.1, light=True))


@pytest.mark.gpu
def test_vec_env_step_and_step_device(native):
    import torch
    from gym_kilobots_b200.envs.vec_env import KilobotsVecEnv
    sc = SC.pushing_yard(8, light="composite")
    spec = LocalObsSpec(0.12, max_neighbours=6, light=True)
    vec = KilobotsVecEnv(sc, local_observation=spec)
    obs = vec.reset()
    nb = vec.batch
    assert obs["local"].shape == (8, nb.N, spec.dim(nb.M))
    _assert_matches(nb, spec, _state_obs(nb), got=obs["local"], where="reset")
    acts = SC.random_actions(sc, 8, 3)
    obs, _, _, _ = vec.step(acts[0])
    _assert_matches(nb, spec, obs, got=obs["local"], where="step")
    obs, _, _, _ = vec.step_device(torch.as_tensor(acts[1], device=nb.device))
    assert obs["local"].is_cuda
    host = {k: obs[k].cpu().numpy() for k in ("kilobots", "objects", "light")}
    _assert_matches(nb, spec, host, got=obs["local"].cpu().numpy(), where="step_device")
    assert vec.local_observation().data_ptr() == obs["local"].data_ptr()
    plain = KilobotsVecEnv(sc)
    plain.reset()
    assert "local" not in plain.step(acts[0])[0] and "local" not in plain.step_device(None)[0]


@pytest.mark.gpu
def test_vec_env_reset_done_with_device_sampler(native):
    import torch
    import yaml
    from gym_kilobots_b200.envs import KilobotsVecEnv, YamlKilobotsEnv  # noqa: F401  (YamlKilobotsEnv: the Yaml tags)
    conf = yaml.load("""
!EvalEnv
width: 1.2
height: 0.8
resolution: 600
objects:
  - !ObjectConf {idx: 0, color: null, shape: square, width: .15, height: .10, init: random, symmetry: null}
  - !ObjectConf {idx: 1, color: null, shape: triangle, width: .1, height: .1, init: [.2, -.1, .5], symmetry: null}
light: !LightConf {type: composite, init: random, components: [!LightConf {type: circular, init: random, radius: .2}, !LightConf {type: momentum, init: [.1, .1], radius: .1}]}
kilobots: !KilobotsConf {num: 12, mean: light, std: .05}
""", Loader=yaml.Loader)
    E = 24
    spec = LocalObsSpec(0.08, max_neighbours=4, light=True)
    vec = KilobotsVecEnv.from_configuration(conf, E, seed=3, local_observation=spec)
    vec.reset()
    nb = vec.batch
    acts = SC.random_actions(vec.action_dim, E, 3)
    for t in range(3):
        obs, _, _, _ = vec.step_device(torch.as_tensor(acts[t], device=nb.device))
    before = obs["local"].cpu().numpy()
    done = torch.as_tensor(np.arange(E) % 4 == 1, device=nb.device)
    vec.reset_done(done)
    after = vec.local_observation(mask=torch.zeros(E, dtype=torch.bool, device=nb.device)).cpu().numpy()
    d = done.cpu().numpy()
    assert np.array_equal(_bits(after[~d]), _bits(before[~d]))       # the other envs' rows are untouched
    ref = _assert_matches(nb, spec, _state_obs(nb), got=vec.local_observation().cpu().numpy(), where="reset_done")
    assert np.array_equal(_bits(after[d]), _bits(ref[d])) and not np.array_equal(_bits(after[d]), _bits(before[d]))
