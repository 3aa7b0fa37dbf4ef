"""The environment layer around the physics (csrc/kb_env.cuh: lights, kilobot controllers, the task layer) on BOTH
kernel tiers -- the lane-group kernels (KB_FORCE_SWARM=0) and the large-swarm tier (KB_FORCE_SWARM=1) -- against the
CPU oracle, bit for bit, on kilobot-only scenes: momentum, linear and composite lights, direct control from a non-zero
reset velocity, and reward / done / episode statistics / flat observation with masked resets."""
import numpy as np
import pytest

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import scenarios as SC
from gym_kilobots_b200 import scene as S
from gym_kilobots_b200.scene import TaskSpec

from parity_util import assert_same_obs, assert_same_state, run_parity

pytestmark = pytest.mark.gpu

BOTH_TIERS = pytest.mark.parametrize("force", ["0", "1"])
SWARM_BLOCKS = (128, 256, 512)   # the lane-group kernels of these scenes run blocks of 64 threads
MIXED = [abi.KB_KILOBOT_PHOTOTAXIS, abi.KB_KILOBOT_SIMPLE_PHOTOTAXIS] * 15
WB = np.array([0.5, 0.25])       # half extents of swarm_corner's 1.0 x 0.5 m table
BOUNDS = (-WB * 1.1, WB * 1.1)
STEP = (np.array([-1, -1]) * .01, np.array([1, 1]) * .01)


def _check_tier(nb, force):
    assert (nb.launch_config()["block_threads"] in SWARM_BLOCKS) == (force == "1")


def _swarm(kinds, lights, light_state, num_envs, seed=0):
    """Kilobots of the given kinds spread over the middle of the table, no objects."""
    sc = SC.swarm_corner(num_envs, n=len(kinds), seed=seed, spread=.08, corner=False)
    sc.scenes[0].bodies = [S.kilobot_body(k) for k in kinds]
    sc.scenes[0].lights = lights
    sc.light_state = np.asarray(light_state, np.float64).reshape(num_envs, -1)
    return sc


def _momentum_light():
    return S.LightSpec(abi.KB_LIGHT_MOMENTUM, radius=.25, bounds=BOUNDS, action_bounds=STEP, max_velocity=.01)


def _light_case(light, E, T, rng):
    """(lights, initial light state [E, L], light actions [T, E, A]); actions reach past their bounds."""
    centre = rng.uniform(-.15, .15, (E, 2))
    if light == "momentum":
        state = np.concatenate([centre, rng.uniform(-.01, .01, (E, 2))], 1)   # some start above max_velocity
        return [_momentum_light()], state, rng.uniform(-.02, .02, (T, E, 2))
    if light == "linear":
        lights = [S.LightSpec(abi.KB_LIGHT_LINEAR, action_bounds=(np.array([-2 * np.pi, 0.]), np.array([2 * np.pi, 0.])))]
        return lights, rng.uniform(-np.pi, np.pi, (E, 1)), rng.uniform(-8.0, 8.0, (T, E, 1))   # clipped, then wrapped
    # composite: an absolutely positioned circular light (relative_actions=False) and a momentum light
    lights = [S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=.2, bounds=(np.array([-.3, -.15]), np.array([.3, .15])),
                          action_bounds=(np.array([-.4, -.2]), np.array([.4, .2])), relative_actions=False),
              _momentum_light()]
    state = np.concatenate([centre, -centre, np.zeros((E, 2))], 1)
    acts = np.concatenate([rng.uniform(-.5, .5, (T, E, 2)), rng.uniform(-.02, .02, (T, E, 2))], 2)
    return lights, state, acts


@BOTH_TIERS
@pytest.mark.parametrize("light", ["momentum", "linear", "composite"])
def test_lights_and_phototaxis_both_tiers(oracle, native, force, light, monkeypatch):
    """Phototaxis and simple-phototaxis kilobots following momentum, linear and composite lights."""
    monkeypatch.setenv("KB_FORCE_SWARM", force)
    E, T = 4, 20
    lights, state, acts = _light_case(light, E, T, np.random.default_rng(7))
    sc = _swarm(MIXED, lights, state, E)
    ob, nb = run_parity(oracle, native, sc, steps=T, actions=acts)
    _check_tier(nb, force)


@BOTH_TIERS
def test_direct_control_from_reset_velocity_both_tiers(oracle, native, force, monkeypatch):
    """Velocity and acceleration kilobots reset with a non-zero kb_velocity, then driven with KB_ACTION_KILOBOTS."""
    monkeypatch.setenv("KB_FORCE_SWARM", force)
    E, T = 4, 20
    kinds = [abi.KB_KILOBOT_VELOCITY, abi.KB_KILOBOT_ACCELERATION] * 12
    sc = _swarm(kinds, [], np.zeros((E, 0)), E)
    rng = np.random.default_rng(3)
    vel = np.stack([rng.uniform(0.0, 0.01, (E, len(kinds))), rng.uniform(-1.0, 1.0, (E, len(kinds)))], -1)
    ob = oracle.OracleBatch(sc.scenes, E, sc.env_scene, sc.max_contacts, threads=8)
    nb = native.NativeBatch(sc.scenes, E, sc.env_scene, sc.max_contacts)
    _check_tier(nb, force)
    ob.reset(sc.body_pose, sc.light_state, kb_velocity=vel)
    nb.reset(sc.body_pose, sc.light_state, kb_velocity=vel)
    assert_same_state(ob, nb, "direct control after reset")
    assert np.array_equal(nb.controllers()[0][..., :2], vel)
    acts = SC.random_kilobot_actions(sc, E, T)
    for t in range(T):
        oo = ob.step(acts[t], abi.KB_ACTION_KILOBOTS)
        on = nb.step(acts[t], abi.KB_ACTION_KILOBOTS)
        assert_same_obs(oo, on, "direct control step %d" % t)
        assert_same_state(ob, nb, "direct control step %d" % t)


@BOTH_TIERS
def test_swarm_task_layer_both_tiers(oracle, native, force, monkeypatch):
    """KB_TASK_SWARM_TO_TARGET: reward, done, status, flat observation and episode statistics every env-step, with a
    masked reset of the finished envs."""
    monkeypatch.setenv("KB_FORCE_SWARM", force)
    E, T = 6, 20
    rng = np.random.default_rng(11)
    light = S.LightSpec(abi.KB_LIGHT_CIRCULAR, radius=.25, bounds=BOUNDS, action_bounds=STEP)
    sc = _swarm(MIXED, [light], rng.uniform(-.1, .1, (E, 2)), E)
    task = TaskSpec(mode=abi.KB_TASK_SWARM_TO_TARGET, w_position=3.0, step_penalty=0.01, success_bonus=1.0,
                    position_tolerance=0.02, max_episode_steps=7)
    tg = np.zeros((E, 3))
    tg[:, :2] = sc.body_pose[:, :, :2].mean(1) + rng.uniform(-.03, .03, (E, 2))   # near the swarm: some envs succeed
    ob = oracle.OracleBatch(sc.scenes, E, sc.env_scene, sc.max_contacts, threads=8)
    nb = native.NativeBatch(sc.scenes, E, sc.env_scene, sc.max_contacts)
    _check_tier(nb, force)
    ob.set_task(task, tg)
    nb.set_task(task, tg)
    fo, fn = ob.bind_flat_observation(), nb.bind_flat_observation()
    ob.reset(sc.body_pose, sc.light_state)
    nb.reset(sc.body_pose, sc.light_state)
    acts = SC.random_actions(sc, E, T, seed=5)
    dones = 0
    for t in range(T):
        oo, on = ob.step(acts[t]), nb.step(acts[t])
        assert_same_obs(oo, on, "task step %d" % t)
        assert np.array_equal(fo, fn.cpu().numpy()), "step %d: flat observation differs" % t
        assert np.array_equal(ob.episode_stats(), nb.episode_stats()), "step %d: episode statistics differ" % t
        d = oo["done"]
        dones += int(d.sum())
        if d.any():
            ob.reset(sc.body_pose, sc.light_state, mask=d)
            nb.reset(sc.body_pose, sc.light_state, mask=d)
            assert_same_state(ob, nb, "task masked reset after step %d" % t)
    assert dones > 0
    assert_same_state(ob, nb, "task end")
