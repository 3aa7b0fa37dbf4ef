"""Batches whose scenes differ in their numbers of objects and kilobots (include/kb_b200.h kb_create, padded body
layout): object j of an env at body index j, kilobot k at Mmax + k, the other indices absent.  Every env of a mixed
batch must compute exactly what the same env computes in a batch of its own size -- on the CPU oracle, on both
kernel tiers, and through the task layer, the lifecycle calls, direct control, the renderer and the host surface --
and the rows of absent bodies must be NaN (observations) or canonical (body state)."""
import numpy as np
import pytest

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import scenarios as SC
from gym_kilobots_b200.scene import TaskSpec

from mixed_oracle import MixedOracle
from parity_util import assert_same_state

MAXC = 320
# the counters that do not depend on the kernel's lane width (as in parity_util.run_parity): substeps, contacts, points,
# position iterations, TOI events, islands
PARITY_COUNTERS = [0, 1, 2, 4, 5, 7]
TASKS = {
    "const": None,
    "object": TaskSpec(mode=abi.KB_TASK_OBJECT_TO_TARGET, object=0, w_position=1.0, w_orientation=0.25,
                       step_penalty=0.001, success_bonus=2.0, position_tolerance=0.5, orientation_tolerance=1.0,
                       max_episode_steps=7),
    "swarm": TaskSpec(mode=abi.KB_TASK_SWARM_TO_TARGET, w_position=3.0, step_penalty=0.01, success_bonus=1.0,
                      position_tolerance=0.3, max_episode_steps=5),
}


def _sizes(per):
    """Three homogeneous scenarios of `per` envs each: QuadAssembly-like (4 quads, 15 kilobots), C1-like (1 quad,
    10 kilobots), one L-form with 30 kilobots."""
    c2 = SC.c2_quad_assembly(per, seed=1, degenerate=False)
    c1 = SC.c1_single_env(per, seed=2)
    c3 = SC.c3_shapes(per, seed=3, num_kilobots=30)
    c3 = SC.Scenario("L30", c3.scenes[:1], None, c3.body_pose, c3.light_state)
    return [c2, c1, c3]


def _mixed(homs):
    """Interleave the homogeneous scenarios env by env into one batch: env e is env e // 3 of homs[e % 3]."""
    per = homs[0].num_envs
    specs = [h.scenes[0] for h in homs]
    env_scene = np.array([e % 3 for e in range(3 * per)], np.int32)
    src = [(e % 3, e // 3) for e in range(3 * per)]
    poses = [homs[s].body_pose[i] for s, i in src]
    light = np.stack([homs[s].light_state[i] for s, i in src])
    return SC.Scenario("mixed", specs, env_scene, SC.stack_poses(specs, env_scene, poses), light, MAXC), src


def _targets(E, seed=3):
    rng = np.random.default_rng(seed)
    t = np.zeros((E, 3))
    t[:, 0] = rng.uniform(-0.8, 0.8, E)
    t[:, 1] = rng.uniform(-0.6, 0.6, E)
    t[:, 2] = rng.uniform(-7.0, 7.0, E)
    return t


def _compact(arr, M, Mmax, N):
    """rows of one env's padded body axis -> its compact (objects, kilobots) rows"""
    return np.concatenate([arr[:M], arr[Mmax:Mmax + N]])


def _check_env(mb, hb, e, i, spec, where):
    """env e of the mixed batch against env i of the homogeneous batch of its size, bit for bit"""
    M, N = spec.num_objects, spec.num_kilobots
    bm, bh = mb.bodies(), hb.bodies()
    assert np.array_equal(_compact(bm[e], M, mb.M, N), bh[i]), where + ": body state"
    absent = np.ones(mb.B, bool)
    absent[:M] = absent[mb.M:mb.M + N] = False
    canon = np.zeros(abi.KB_BODY_STATE_FLOATS, np.float32)
    canon[11] = 1.0
    assert np.all(bm[e, absent] == canon), where + ": absent bodies not canonical"
    (pm, nm), (ph, nh) = mb.contacts(), hb.contacts()
    assert nm[e] == nh[i] and np.array_equal(pm[e], ph[i]), where + ": contacts"
    assert np.array_equal(mb.impulses()[e], hb.impulses()[i]), where + ": impulses"
    assert np.array_equal(mb.counters()[e, PARITY_COUNTERS], hb.counters()[i, PARITY_COUNTERS]), where + ": counters"
    fm, fh = mb.proxies()[e], hb.proxies()[i]
    assert np.array_equal(fm[:hb.P], fh) and not fm[hb.P:].any(), where + ": proxies"
    (cm, lm), (ch, lh) = mb.controllers(), hb.controllers()
    assert np.array_equal(cm[e, :N], ch[i]) and not cm[e, N:].any(), where + ": controllers"
    assert np.array_equal(lm[e], lh[i]), where + ": light"
    assert np.array_equal(mb.episode_stats()[e], hb.episode_stats()[i]), where + ": episode statistics"
    assert mb.get_status()[e] == hb.get_status()[i], where + ": status"


def _check_obs(om, oh, e, i, spec, Mmax, Nmax, where, flat_m=None, flat_h=None):
    M, N = spec.num_objects, spec.num_kilobots
    assert np.array_equal(om["kilobots"][e, :N], oh["kilobots"][i]), where + ": kilobots"
    assert np.all(np.isnan(om["kilobots"][e, N:])), where + ": absent kilobot rows"
    assert np.array_equal(om["objects"][e, :M], oh["objects"][i]), where + ": objects"
    assert np.all(np.isnan(om["objects"][e, M:])), where + ": absent object rows"
    for k in ("light", "reward", "done", "status"):
        assert np.array_equal(om[k][e], oh[k][i]), where + ": " + k
    if flat_m is not None:
        L = oh["light"].shape[1]
        fm, fh = flat_m[e], flat_h[i]
        assert np.array_equal(fm[:2 * N], fh[:2 * N]) and np.all(np.isnan(fm[2 * N:2 * Nmax])), where + ": flat kilobots"
        assert np.array_equal(fm[2 * Nmax:2 * Nmax + L], fh[2 * N:2 * N + L]), where + ": flat light"
        o0 = 2 * Nmax + L
        assert np.array_equal(fm[o0:o0 + 4 * M], fh[2 * N + L:]) and np.all(np.isnan(fm[o0 + 4 * M:])), where + ": flat objects"


def _run_mixed_vs_homogeneous(make_mixed, make, homs, steps, task=None, flat=False):
    """Step a mixed batch and one homogeneous batch per size with the same inputs; compare every env."""
    mixed, src = _mixed(homs)
    E = mixed.num_envs
    mb = make_mixed(mixed.scenes, E, mixed.env_scene, MAXC)
    hbs = [make(h.scenes, h.num_envs, None, MAXC) for h in homs]
    assert (mb.M, mb.N, mb.B) == (4, 30, 34)
    obj, kb = mb.body_counts()
    assert np.array_equal(obj, [homs[s].scenes[0].num_objects for s, _ in src])
    assert np.array_equal(kb, [homs[s].scenes[0].num_kilobots for s, _ in src])
    tg = _targets(E)
    if task is not None:
        mb.set_task(task, tg)
        for s, hb in enumerate(hbs):
            hb.set_task(task, tg[s::3])
    fm = mb.bind_flat_observation() if flat else None
    fh = [hb.bind_flat_observation() if flat else None for hb in hbs]
    mb.reset(mixed.body_pose, mixed.light_state)
    for s, (h, hb) in enumerate(zip(homs, hbs)):
        hb.reset(h.body_pose, h.light_state)
    for e, (s, i) in enumerate(src):
        _check_env(mb, hbs[s], e, i, homs[s].scenes[0], "env %d after reset" % e)
    acts = SC.random_actions(2, E, steps, seed=7)
    for t in range(steps):
        om = mb.step(acts[t])
        oh = [hb.step(acts[t][s::3]) for s, hb in enumerate(hbs)]
        flm = None if fm is None else (fm.cpu().numpy() if hasattr(fm, "cpu") else fm.copy())
        for e, (s, i) in enumerate(src):
            flh = None if fh[s] is None else (fh[s].cpu().numpy() if hasattr(fh[s], "cpu") else fh[s])
            _check_obs(om, oh[s], e, i, homs[s].scenes[0], mb.M, mb.N, "step %d env %d" % (t, e), flm, flh)
    for e, (s, i) in enumerate(src):
        _check_env(mb, hbs[s], e, i, homs[s].scenes[0], "env %d after %d steps" % (e, steps))
    return mb, hbs, mixed, src


# ----------------------------------------------------------------------------------------------------- CPU oracle
@pytest.mark.parametrize("task", list(TASKS), ids=list(TASKS))
def test_oracle_mixed_batch_equals_homogeneous_batches(oracle, task):
    """the reference of a mixed batch (one compact oracle world per env, reported in the padded layout) against
    homogeneous oracle batches of each size"""
    make_mixed = lambda scenes, E, es, mc: MixedOracle(oracle, scenes, E, es, mc)
    make = lambda scenes, E, es, mc: oracle.OracleBatch(scenes, E, es, mc, threads=4)
    _run_mixed_vs_homogeneous(make_mixed, make, _sizes(2), 20, TASKS[task], flat=task != "const")


def test_stack_poses_layout():
    homs = _sizes(1)
    specs = [h.scenes[0] for h in homs]
    poses = [h.body_pose[0] for h in homs]
    out = SC.stack_poses(specs, [0, 1, 2], poses)
    assert out.shape == (3, 34, 3)
    assert np.array_equal(out[1, :1], poses[1][:1]) and not out[1, 1:4].any()
    assert np.array_equal(out[1, 4:14], poses[1][1:]) and not out[1, 14:].any()
    assert np.array_equal(out[2, 4:], poses[2][1:])
    # a homogeneous batch is stacked unchanged
    assert np.array_equal(SC.stack_poses(specs[:1], [0, 0], [poses[0], poses[0]]), np.stack([poses[0]] * 2))


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("task", list(TASKS), ids=list(TASKS))
def test_native_mixed_batch_equals_oracle_and_homogeneous(oracle, native, task):
    """lane-group tier (Bmax = 34: 16-lane groups): native mixed == native homogeneous per size, and == oracle mixed"""
    homs = _sizes(6)
    make = lambda scenes, E, es, mc: native.NativeBatch(scenes, E, es, mc)
    mb, _, mixed, _ = _run_mixed_vs_homogeneous(make, make, homs, 20, TASKS[task], flat=task != "const")
    assert mb.launch_config()["lanes_per_env"] == 16
    ob = MixedOracle(oracle, mixed.scenes, mixed.num_envs, mixed.env_scene, MAXC)
    nb = native.NativeBatch(mixed.scenes, mixed.num_envs, mixed.env_scene, MAXC)
    assert np.array_equal(ob.mass_data(), nb.mass_data())
    if TASKS[task] is not None:
        tg = _targets(mixed.num_envs)
        ob.set_task(TASKS[task], tg)
        nb.set_task(TASKS[task], tg)
    ob.reset(mixed.body_pose, mixed.light_state)
    nb.reset(mixed.body_pose, mixed.light_state)
    assert_same_state(ob, nb, "mixed after reset")
    acts = SC.random_actions(2, mixed.num_envs, 20, seed=7)
    for t in range(20):
        oo, on = ob.step(acts[t]), nb.step(acts[t])
        for k in oo:
            assert np.array_equal(oo[k], on[k], equal_nan=k in ("kilobots", "objects")), (t, k)
        assert_same_state(ob, nb, "mixed step %d" % t)
    assert np.array_equal(ob.counters()[:, PARITY_COUNTERS], nb.counters()[:, PARITY_COUNTERS])
    assert np.array_equal(ob.episode_stats(), nb.episode_stats())
    with pytest.raises(RuntimeError):
        nb.set_task(TaskSpec(mode=abi.KB_TASK_OBJECT_TO_TARGET, object=1))


# (spread, corner): swarms jammed into the table's corner where the spawn leaves the default contact capacity enough room;
# the 300-kilobot swarm spreads over the table instead (in the corner its clipped spawn piles kilobots on top of each
# other beyond any capacity)
SWARM_SPAWN = {10: (.05, True), 40: (.05, True), 100: (.07, True), 300: (.14, False)}


def _swarm_mix(sizes, per=2):
    scs = [SC.swarm_corner(per, n=n, seed=10 + n, spread=SWARM_SPAWN[n][0], corner=SWARM_SPAWN[n][1]) for n in sizes]
    specs = [s.scenes[0] for s in scs]
    src = [(e % len(sizes), e // len(sizes)) for e in range(per * len(sizes))]
    es = np.array([s for s, _ in src], np.int32)
    pose = SC.stack_poses(specs, es, [scs[s].body_pose[i] for s, i in src])
    light = np.stack([scs[s].light_state[i] for s, i in src])
    return SC.Scenario("swarm-mix", specs, es, pose, light, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("sizes,force", [((40, 100, 300), "0"), ((10, 40), "1")], ids=["40-100-300", "10-40-forced"])
def test_native_swarm_tier_mixed_batch_equals_oracle(oracle, native, sizes, force, monkeypatch):
    """large-swarm tier (Bmax > 62, or KB_FORCE_SWARM=1): swarms of several sizes, jammed against the table, continuous
    collision on"""
    monkeypatch.setenv("KB_FORCE_SWARM", force)
    sc = _swarm_mix(sizes)
    assert sc.scenes[0].enable_toi
    ob = MixedOracle(oracle, sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    nb = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    assert nb.launch_config()["lanes_per_env"] >= 128
    ob.reset(sc.body_pose, sc.light_state)
    nb.reset(sc.body_pose, sc.light_state)
    assert_same_state(ob, nb, "swarm mix after reset")
    acts = SC.random_actions(2, sc.num_envs, 12, seed=9)
    for t in range(12):
        oo, on = ob.step(acts[t]), nb.step(acts[t])
        for k in oo:
            assert np.array_equal(oo[k], on[k], equal_nan=k == "kilobots"), (t, k)
        assert_same_state(ob, nb, "swarm mix step %d" % t)
    assert np.array_equal(ob.counters()[:, PARITY_COUNTERS], nb.counters()[:, PARITY_COUNTERS])
    assert ob.counters()[:, 5].sum() > 0 and not nb.get_status().any()
    assert np.array_equal(nb.body_counts()[1], [sizes[s] for s in sc.env_scene])


@pytest.mark.gpu
def test_native_lifecycle_scene_switch_setpose_and_state_resume(oracle, native):
    homs = _sizes(2)
    mixed, src = _mixed(homs)
    E = mixed.num_envs
    ob = MixedOracle(oracle, mixed.scenes, E, mixed.env_scene, MAXC)
    nb = native.NativeBatch(mixed.scenes, E, mixed.env_scene, MAXC)
    for b in (ob, nb):
        b.reset(mixed.body_pose, mixed.light_state)
    acts = SC.random_actions(2, E, 6, seed=4)
    for b in (ob, nb):
        b.step(acts[0])
    # set_poses on absent bodies changes nothing (rows of absent bodies hold NaN here)
    pose = mixed.body_pose + 0.003
    obj, kb = nb.body_counts()
    for e in range(E):
        pose[e, obj[e]:nb.M] = np.nan
        pose[e, nb.M + kb[e]:] = np.nan
    for b in (ob, nb):
        b.set_poses(pose)
    assert_same_state(ob, nb, "after set_poses")
    # scene switch: envs 0 (QuadAssembly-like) and 1 (C1-like) swap sizes at a masked reset
    es = mixed.env_scene.copy()
    es[0], es[1] = 1, 0
    m = np.zeros(E, np.uint8)
    m[:2] = 1
    for b in (ob, nb):
        b.set_env_scene(es)
    assert np.array_equal(nb.body_counts()[1], kb)   # not before the reset
    swapped = mixed.body_pose.copy()
    swapped[0], swapped[1] = mixed.body_pose[1], mixed.body_pose[0]
    for b in (ob, nb):
        b.reset(swapped, mixed.light_state, mask=m)
    assert np.array_equal(nb.body_counts()[1][:2], [10, 15]) and np.array_equal(nb.body_counts()[1][2:], kb[2:])
    assert np.array_equal(nb.body_counts()[0][:2], [1, 4])
    assert_same_state(ob, nb, "after the scene switch")
    # get_state / set_state: bit-identical resume
    blob = nb.get_state()
    ref = [nb.step(acts[t]) for t in range(1, 4)]
    ref_bodies = nb.bodies()
    nb.set_state(blob)
    again = [nb.step(acts[t]) for t in range(1, 4)]
    for r, a in zip(ref, again):
        for k in r:
            assert np.array_equal(r[k], a[k], equal_nan=True), k
    assert np.array_equal(ref_bodies, nb.bodies())
    for t in range(1, 4):
        oo = ob.step(acts[t])
        for k in oo:
            assert np.array_equal(oo[k], again[t - 1][k], equal_nan=True), k
    assert_same_state(ob, nb, "after the resume")


@pytest.mark.gpu
def test_native_direct_control_ignores_absent_action_rows(oracle, native):
    small = SC.direct_control(4, seed=5)
    big = SC.direct_control(4, seed=6)
    sp_small = SC.S.SceneSpec(bodies=small.scenes[0].bodies[:6], num_objects=2, lights=[],
                              world_size=small.scenes[0].world_size)
    specs = [big.scenes[0], sp_small]
    es = np.array([0, 1, 0, 1, 0, 1, 0, 1], np.int32)
    poses = [big.body_pose[e // 2] if s == 0 else small.body_pose[e // 2][:6] for e, s in enumerate(es)]
    sc = SC.Scenario("direct-mix", specs, es, SC.stack_poses(specs, es, poses), np.zeros((8, 0)), 64)
    nb = native.NativeBatch(sc.scenes, 8, es, 64)
    ob = MixedOracle(oracle, sc.scenes, 8, es, 64)
    acts = SC.random_kilobot_actions(big, 8, 8, seed=3).reshape(8, 8, nb.N, 2)
    nan_acts = acts.copy()
    nan_acts[:, 1::2, 4:] = np.nan   # the small scene has 4 kilobots: rows 4..7 are absent
    for b in (ob, nb):
        b.reset(sc.body_pose, None)
    for t in range(8):
        on = nb.step(nan_acts[t].reshape(8, -1), abi.KB_ACTION_KILOBOTS)
        oo = ob.step(acts[t].reshape(8, -1), abi.KB_ACTION_KILOBOTS)
        assert not on["status"].any()
        for k in oo:
            assert np.array_equal(oo[k], on[k], equal_nan=True), (t, k)
        assert_same_state(ob, nb, "direct control step %d" % t)


@pytest.mark.gpu
def test_native_render_of_mixed_batch(oracle, native):
    homs = _sizes(1)
    mixed, src = _mixed(homs)
    nb = native.NativeBatch(mixed.scenes, mixed.num_envs, mixed.env_scene, MAXC)
    ob = MixedOracle(oracle, mixed.scenes, mixed.num_envs, mixed.env_scene, MAXC)
    nb.reset(mixed.body_pose, mixed.light_state)
    ob.reset(mixed.body_pose, mixed.light_state)
    img = nb.render(range(3), 320, 240).cpu().numpy()
    assert np.array_equal(img, ob.render(range(3), 320, 240))
    for s, h in enumerate(homs):
        hb = native.NativeBatch(h.scenes, 1, None, MAXC)
        hb.reset(h.body_pose, h.light_state)
        assert np.array_equal(img[s], hb.render((0,), 320, 240).cpu().numpy()[0]), "env %d" % s


@pytest.mark.gpu
def test_vec_env_from_envs_with_different_counts(native):
    import torch
    from gym_kilobots_b200.envs import QuadAssemblyKilobotsEnv, YamlKilobotsEnv
    from gym_kilobots_b200.envs.vec_env import KilobotsVecEnv
    import yaml
    text = """
!EvalEnv
width: 1.0
height: 1.0
resolution: 600
objects:
  - !ObjectConf {idx: 0, color: null, shape: square, width: .1, height: .1, init: random, symmetry: null}
light: !LightConf {type: circular, init: object, radius: .2}
kilobots: !KilobotsConf {num: %d, mean: light, std: .03, type: PhototaxisKilobot}
"""
    cfg8, cfg12 = (yaml.load(text % n, Loader=yaml.Loader) for n in (8, 12))
    np.random.seed(4)
    envs = [YamlKilobotsEnv(configuration=cfg8), YamlKilobotsEnv(configuration=cfg12), QuadAssemblyKilobotsEnv(),
            YamlKilobotsEnv(configuration=cfg8)]
    vec = KilobotsVecEnv.from_envs(envs, flat_observation=True, allow_status_flags=True)
    n = np.array([8, 12, 15, 8])
    m = np.array([1, 1, 4, 1])
    assert vec.num_kilobots == 15 and vec.num_objects == 4
    assert vec.kilobot_mask.is_cuda and vec.kilobot_mask.dtype == torch.bool
    assert np.array_equal(vec.kilobot_mask.cpu().numpy(), np.arange(15)[None] < n[:, None])
    assert np.array_equal(vec.object_mask.cpu().numpy(), np.arange(vec.num_objects)[None] < m[:, None])
    vec.reset()
    a = np.zeros((4, vec.action_dim))
    obs, r, d, info = vec.step(a)
    km = vec.kilobot_mask.cpu().numpy()
    om = vec.object_mask.cpu().numpy()
    assert np.all(np.isnan(obs["kilobots"][~km])) and np.all(np.isfinite(obs["kilobots"][km]))
    assert np.all(np.isnan(obs["objects"][~om])) and np.all(np.isfinite(obs["objects"][om]))
    flat = obs["flat"]
    assert np.all(np.isnan(flat[:, :30].reshape(4, 15, 2)[~km]))
    obs_d, _, _, _ = vec.step_device(a)
    assert torch.isnan(obs_d["kilobots"][~vec.kilobot_mask]).all()
    st = vec.get_state()
    assert np.all(np.isnan(st["kilobots"][~km])) and np.all(np.isfinite(st["kilobots"][km]))
    with pytest.raises(ValueError):
        vec.use_device_sampler(cfg8)
    # a scene switch moves the masks at the env's next reset
    es = vec._env_scene.cpu().numpy().copy()
    es[0], es[1] = es[1], es[0]
    vec.set_env_scene(es)
    assert np.array_equal(vec.kilobot_mask.cpu().numpy(), km)
    done = torch.zeros(4, dtype=torch.uint8, device=vec.batch.device)
    done[0] = 1
    pose = vec.scenario.body_pose.copy()
    pose[0] = pose[1]
    vec.reset_done(done, pose, vec.scenario.light_state)
    assert vec.kilobot_mask[0].sum().item() == 12
    assert np.array_equal(vec.batch.body_counts()[1], [12, 12, 15, 8])
