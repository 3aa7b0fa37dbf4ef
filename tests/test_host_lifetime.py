"""Lifetime of a batch's device resources (kb_create / kb_destroy): a rejected kb_create leaves nothing behind, batches
that use every resource a handle owns can be created and destroyed over and over without changing what a fresh batch
computes, and a batch is destroyed on its own device whichever device is current."""
import ctypes

import numpy as np
import pytest
import yaml

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import scenarios as SC
from gym_kilobots_b200.envs import KilobotsVecEnv
from gym_kilobots_b200.scene import LocalObsSpec

pytestmark = pytest.mark.gpu

KB_ERR_INVALID = -1   # include/kb_b200.h


@pytest.fixture
def native():
    from gym_kilobots_b200 import _native
    _native.load()
    return _native


def _conf(num_objects, num_kilobots):
    objects = ["!ObjectConf {idx: 0, color: null, shape: square, width: .15, height: .10, init: random, symmetry: null}",
               "!ObjectConf {idx: 1, color: null, shape: circle, width: .08, height: .08, init: random, symmetry: null}"]
    text = """
!EvalEnv
width: 1.2
height: 0.8
resolution: 600
objects: [%s]
light: !LightConf {type: circular, init: random, radius: .2}
kilobots: !KilobotsConf {num: %d, mean: random, std: .05}
""" % (", ".join(objects[:num_objects]), num_kilobots)
    return yaml.load(text, Loader=yaml.Loader)


def test_out_of_range_env_scene_is_rejected(native):
    sc = SC.c2_quad_assembly(8)
    descs = (abi.KbSceneDesc * 1)()
    descs[0], keep = sc.scenes[0].to_desc()
    h = ctypes.c_void_p()
    for bad in (1, -1):
        env_scene = np.zeros(8, np.int32)
        env_scene[5] = bad
        rc = native._fn["create"](descs, 1, env_scene.ctypes.data_as(ctypes.c_void_p), 8, sc.max_contacts, 0,
                                  ctypes.byref(h))
        assert rc == KB_ERR_INVALID and b"env_scene out of range" in native._fn["last_error"]()
    nb = native.NativeBatch(sc.scenes, 8, np.zeros(8, np.int32), sc.max_contacts)
    nb.reset(sc.body_pose, sc.light_state)
    out = nb.step(SC.random_actions(sc, 8, 1)[0])
    assert np.isfinite(out["kilobots"]).all() and not out["status"].any()
    nb.close()


def _run(force_swarm, monkeypatch):
    """A mixed-configuration batch through everything its handle allocates: the sampler buffers, sampled resets (all
    envs and masked), local observations, the render id buffer and host steps pipelined over three chunks."""
    monkeypatch.setenv("KB_FORCE_SWARM", force_swarm)
    monkeypatch.setenv("KB_HOST_CHUNKS", "3")
    confs = [_conf(0, 6), _conf(0, 9)] if force_swarm == "1" else [_conf(1, 6), _conf(2, 9)]
    E = 40
    spec = LocalObsSpec(0.2, max_neighbours=4, objects=force_swarm == "0", light=True)
    vec = KilobotsVecEnv.from_configurations(confs, E, weights=[1.0, 2.0], seed=3, local_observation=spec)
    assert (vec.batch.launch_config()["block_threads"] >= 128) == (force_swarm == "1")
    out = [vec.reset()["local"]]
    acts = SC.random_actions(vec.scenario, E, 3, seed=5)
    for t in range(3):
        obs, reward, done, info = vec.step(acts[t])
        out += [obs["kilobots"].copy(), obs["objects"].copy(), obs["light"].copy(), reward.copy(), info["status"].copy(),
                obs["local"]]
    out.append(vec.render(env_ids=[0, 7, 39], width=64, height=48))
    vec.reset_done(np.arange(E) % 3 == 0)
    out += [vec.batch.bodies(), vec.local_observation().cpu().numpy()]
    vec.close()
    return out


@pytest.mark.parametrize("force_swarm", ["0", "1"])
def test_repeated_create_and_destroy(native, force_swarm, monkeypatch):
    before = _run(force_swarm, monkeypatch)
    for _ in range(4):
        _run(force_swarm, monkeypatch)
    after = _run(force_swarm, monkeypatch)
    assert len(after) == len(before)
    for i, (a, b) in enumerate(zip(before, after)):
        assert a.dtype == b.dtype and np.array_equal(a, b, equal_nan=True), i


def test_destroy_on_another_device(native):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    sc = SC.c5_small(1 << 18)
    nb = native.NativeBatch(sc.scenes, sc.num_envs, None, sc.max_contacts, device=1)
    nb.reset(sc.body_pose, sc.light_state)
    nb.step(SC.random_actions(sc, sc.num_envs, 1)[0])
    blob_bytes = nb.state_bytes_per_env * nb.E
    torch.cuda.synchronize(1)
    free_before, _ = torch.cuda.mem_get_info(1)
    torch.cuda.set_device(0)
    nb.close()
    free_after, _ = torch.cuda.mem_get_info(1)
    assert free_after - free_before >= blob_bytes // 2
    # both devices still take new batches
    for dev in (0, 1):
        b = native.NativeBatch(sc.scenes[:1], 64, None, sc.max_contacts, device=dev)
        b.reset(sc.body_pose[:64], sc.light_state[:64])
        assert np.isfinite(b.step(SC.random_actions(sc, 64, 1)[0])["kilobots"]).all()
        b.close()
