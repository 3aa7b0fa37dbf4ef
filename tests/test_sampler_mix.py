"""On-device scene sampling for batches that mix several Yaml configurations (kb_set_sampler_mix, sampler.SamplerMix,
KilobotsVecEnv.from_configurations).  Each configuration is drawn exactly as its own SceneSampler draws it, placed in the
padded body layout (objects at rows 0..M_e-1, kilobots at Mmax + k, NaN rows for absent bodies); with weights, the
configuration itself is drawn first from its own Philox stream, keyed by (seed, global env id, episode).  On the GPU, both
kernel tiers are compared with the numpy mirror (1e-12: libm vs CUDA log / sin / cos) and, after the reset, with the CPU
reference of a mixed batch (tests/mixed_oracle.py) bit for bit."""
import numpy as np
import pytest
import yaml

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import philox as PX
from gym_kilobots_b200 import scenarios as SC
from gym_kilobots_b200.envs import KilobotsVecEnv  # noqa: F401  (also registers the Yaml configuration tags)
from gym_kilobots_b200.sampler import SamplerMix, SceneSampler
from gym_kilobots_b200.scene import TaskSpec

OBJECTS = ["!ObjectConf {idx: 0, color: null, shape: square, width: .15, height: .10, init: random, symmetry: null}",
           "!ObjectConf {idx: 1, color: null, shape: triangle, width: .1, height: .1, init: [.2, -.1, .5], symmetry: null}",
           "!ObjectConf {idx: 2, color: null, shape: circle, width: .08, height: .08, init: random, symmetry: null}"]
COMPOSITE = ("!LightConf {type: composite, init: %s, components: [!LightConf {type: circular, init: random, radius: .2}, "
             "!LightConf {type: momentum, init: [.1, .1], radius: .1}]}")
SHUFFLED, FIXED_ORDER = COMPOSITE % "random", COMPOSITE % "null"
MOMENTUM_AT_OBJECT = "!LightConf {type: momentum, init: object, radius: .2}"
MOMENTUM_RANDOM = "!LightConf {type: momentum, init: random, radius: .2}"


def _conf(num_objects, num_kilobots, light, mean="light", std=.03, width=1.2, height=.8, objects=None):
    objs = (objects if objects is not None else OBJECTS)[:num_objects]
    text = """
!EvalEnv
width: %s
height: %s
resolution: 600
objects: [%s]
light: %s
kilobots: !KilobotsConf {num: %d, mean: %s, std: %s}
""" % (width, height, ", ".join(objs), light, num_kilobots, mean, std)
    return yaml.load(text, Loader=yaml.Loader)


def _composite_confs():
    """three configurations with one light structure: a shuffled composite (two scenes each) and a fixed-order one"""
    return [_conf(2, 6, SHUFFLED), _conf(1, 10, FIXED_ORDER), _conf(0, 14, SHUFFLED, mean="random")]


def _assert_padded_equal(mix, confs, pose, light, scene, config, env_ids, episodes, seed, base):
    """every env's draws == its configuration's own SceneSampler, placed in the padded layout"""
    for c, conf in enumerate(confs):
        sel = np.flatnonzero(config == c)
        if len(sel) == 0:
            continue
        ref = SceneSampler(conf, seed=seed, env_id_base=base)
        p, l, s = ref.sample_numpy(np.asarray(env_ids)[sel], np.broadcast_to(episodes, (len(env_ids),))[sel])
        M, N = ref.M, ref.N
        assert np.array_equal(pose[sel, :M], p[:, :M]), c
        assert np.array_equal(pose[sel, mix.M:mix.M + N], p[:, M:]), c
        assert np.all(np.isnan(pose[sel, M:mix.M])) and np.all(np.isnan(pose[sel, mix.M + N:])), c
        assert np.array_equal(light[sel], l), c
        assert np.array_equal(scene[sel], mix.scene_offset[c] + s), c


# --------------------------------------------------------------------------------------------------------------- CPU
def test_env_config_mode_draws_each_configuration_like_its_own_sampler():
    confs = _composite_confs()
    mix = SamplerMix(confs, seed=5, env_id_base=100)
    assert list(mix.scene_offset) == [0, 2, 3] and list(mix.scene_config) == [0, 0, 1, 2, 2]
    assert (mix.M, mix.N) == (2, 14) and len(mix.scene_specs()) == 5
    assert [s.perm_scene for s in mix.samplers] == [[0, 1], [2], [3, 4]]
    E = 30
    cfg = np.arange(E) % 3
    eps = np.arange(E) % 4
    pose, light, scene, config = mix.sample_numpy(np.arange(E), eps, mix.scene_offset[cfg])
    assert pose.shape == (E, 16, 3) and light.shape == (E, 6)
    assert np.array_equal(config, cfg)
    _assert_padded_equal(mix, confs, pose, light, scene, config, np.arange(E), eps, 5, 100)
    assert set(scene[cfg == 0]) == {0, 1} and set(scene[cfg == 2]) == {3, 4} and set(scene[cfg == 1]) == {2}


def test_weighted_mode_frequencies_keys_and_streams():
    confs = _composite_confs()
    w = np.array([1.0, 2.0, 1.0])
    mix = SamplerMix(confs, weights=w, seed=9, env_id_base=40)
    assert mix.cdf[-1] == 1.0 and np.allclose(mix.cdf, [.25, .75, 1.0])
    n = 20000
    whole = mix.sample_numpy(np.arange(n), 3)
    p = w / w.sum()
    freq = np.bincount(whole[3], minlength=3) / n
    assert np.all(np.abs(freq - p) <= 6 * np.sqrt(p * (1 - p) / n)), freq
    # a pure function of (seed, global env id, episode): "rank 5 of 20" draws what the whole job draws for its envs
    part = SamplerMix(confs, weights=w, seed=9, env_id_base=40 + 5000).sample_numpy(np.arange(1000), 3)
    for a, b in zip(part, whole):
        assert np.array_equal(a, b[5000:6000], equal_nan=True)
    # the configuration is the first k with u < cdf[k], u from its own stream
    u, _ = PX.EnvRng(9, np.arange(n) + 40, 3).uniform2(PX.STREAM_CONFIG, 0)
    assert np.array_equal(whole[3], np.searchsorted(mix.cdf, u, side="right"))
    # a new episode, new configurations
    again = mix.sample_numpy(np.arange(n), 4)[3]
    assert 0.5 < np.mean(again != whole[3]) < 0.75
    # given its configuration, every other draw of an env is the single-configuration sampler's: the new stream shifts
    # nothing
    k = 600
    _assert_padded_equal(mix, confs, whole[0][:k], whole[1][:k], whole[2][:k], whole[3][:k], np.arange(k), 3, 9, 40)


def test_zero_weights_are_never_drawn():
    confs = _composite_confs()
    mix = SamplerMix(confs, weights=[0.0, 3.0, 0.0], seed=2)
    assert list(mix.cdf) == [0.0, 1.0, 1.0]
    assert np.all(mix.sample_numpy(np.arange(500), 0)[3] == 1)


def test_refusals():
    confs = _composite_confs()
    with pytest.raises(ValueError, match="light components"):
        SamplerMix([confs[0], _conf(1, 8, MOMENTUM_RANDOM)])
    with pytest.raises(ValueError, match="light components"):   # the same state dimension, other types
        SamplerMix([_conf(1, 8, "!LightConf {type: circular, init: random, radius: .2}"),
                    _conf(1, 8, "!LightConf {type: linear, init: .5, radius: .2}"),
                    _conf(1, 8, "!LightConf {type: linear, init: .5, radius: .2}")])
    with pytest.raises(ValueError, match="table size"):
        SamplerMix([confs[0], _conf(1, 8, SHUFFLED, width=1.0)])
    many = ["!ObjectConf {idx: %d, color: null, shape: square, width: .05, height: .05, init: random, symmetry: null}" % i
            for i in range(17)]
    with pytest.raises(ValueError, match="17 objects"):
        SamplerMix([confs[0], _conf(17, 4, SHUFFLED, objects=many)])
    with pytest.raises(ValueError, match="1 to 16"):
        SamplerMix([confs[1]] * 17)
    with pytest.raises(ValueError, match="1 to 16"):
        SamplerMix([])
    for bad in ([1.0, -1.0, 1.0], [0.0, 0.0, 0.0], [1.0, np.nan, 1.0], [1.0, np.inf, 1.0], [1.0, 1.0]):
        with pytest.raises(ValueError, match="weights"):
            SamplerMix(confs, weights=bad)
    with pytest.raises(ValueError, match="env_scene"):
        SamplerMix(confs).sample_numpy(np.arange(3), 0)
    with pytest.raises(ValueError, match="exactly one"):
        KilobotsVecEnv.from_configurations(confs, 6)
    with pytest.raises(ValueError, match="exactly one"):
        KilobotsVecEnv.from_configurations(confs, 6, weights=[1, 1, 1], env_config=[0] * 6)
    with pytest.raises(ValueError, match="one configuration index per env"):
        KilobotsVecEnv.from_configurations(confs, 6, env_config=[0, 1, 2, 3, 0, 1])


# --------------------------------------------------------------------------------------------------------------- GPU
def _check_sampled_reset(vec, ref, mask=None):
    """the device's draws == the numpy mirror (1e-12), scenes exactly, NaN rows where the mirror has them; the body
    counts and both masks follow the drawn configurations.  Returns the device's (pose, light, scene, episodes)."""
    pose, light, scene, ep = vec.batch.get_sampled()
    m = np.ones(vec.num_envs, bool) if mask is None else mask
    assert np.array_equal(np.isnan(pose[m]), np.isnan(ref[0][m]))
    assert np.nanmax(np.abs(pose[m] - ref[0][m])) <= 1e-12 and np.abs(light[m] - ref[1][m]).max() <= 1e-12
    assert np.array_equal(scene[m], ref[2][m])
    mix = vec.sampler
    obj, kb = vec.batch.body_counts()
    assert np.array_equal(obj, [mix.samplers[c].M for c in mix.scene_config[scene]])
    assert np.array_equal(kb, [mix.samplers[c].N for c in mix.scene_config[scene]])
    assert np.array_equal(vec.kilobot_mask.cpu().numpy(), np.arange(vec.num_kilobots)[None] < kb[:, None])
    assert np.array_equal(vec.object_mask.cpu().numpy(), np.arange(vec.num_objects)[None] < obj[:, None])
    assert np.array_equal(vec.batch.current_scenes().cpu().numpy(), scene)
    return pose, light, scene, ep


def _step_both(vec, ob, acts, ts, flat=False):
    for t in ts:
        o1, r1, d1, _ = vec.step(acts[t])
        o2 = ob.step(acts[t])
        for k in ("kilobots", "objects", "light"):
            assert np.array_equal(o1[k], o2[k], equal_nan=True), (t, k)
        assert np.array_equal(r1, o2["reward"]) and np.array_equal(d1, o2["done"].astype(bool)), t
        if flat:
            assert np.array_equal(o1["flat"], ob.obs_flat, equal_nan=True), t
    assert np.array_equal(vec.batch.bodies(), ob.bodies())


@pytest.mark.gpu
def test_lane_group_tier_weighted_mix(oracle, native):
    import torch
    from mixed_oracle import MixedOracle
    confs = [_conf(2, 6, MOMENTUM_AT_OBJECT), _conf(1, 12, MOMENTUM_RANDOM), _conf(0, 20, MOMENTUM_RANDOM, mean="random")]
    E, w, seed, base = 60, [1.0, 2.0, 1.0], 21, 500
    task = TaskSpec(mode=abi.KB_TASK_SWARM_TO_TARGET, w_position=3.0, step_penalty=0.01, success_bonus=1.0,
                    position_tolerance=0.3, max_episode_steps=50)
    tg = np.zeros((E, 3))
    tg[:, 0] = np.linspace(-.4, .4, E)
    vec = KilobotsVecEnv.from_configurations(confs, E, weights=w, seed=seed, env_id_base=base, task=task, targets=tg,
                                             flat_observation=True)
    assert vec.batch.launch_config()["lanes_per_env"] <= 32 and (vec.num_objects, vec.num_kilobots) == (2, 20)
    mix, sc = vec.sampler, vec.scenario
    vec.reset()
    ref = mix.sample_numpy(np.arange(E), 0)
    assert set(ref[3]) == {0, 1, 2}
    pose, light, scene, ep = _check_sampled_reset(vec, ref)
    assert np.all(ep == 1) and np.array_equal(scene, sc.env_scene)   # creation drew what the first reset draws
    ob = MixedOracle(oracle, sc.scenes, E, sc.env_scene, sc.max_contacts)
    ob.set_task(task, tg)
    ob.bind_flat_observation()
    ob.set_env_scene(scene)
    ob.reset(pose, light)
    assert np.array_equal(vec.batch.bodies(), ob.bodies())
    acts = SC.random_actions(sc, E, 6, seed=3)
    _step_both(vec, ob, acts, range(3), flat=True)
    # masked auto-reset: exactly the done envs re-draw, with their episode-1 configurations and scenes
    done = torch.zeros(E, dtype=torch.uint8, device="cuda")
    done[::3] = 1
    m = done.cpu().numpy().astype(bool)
    vec.reset_done(done)
    ref2 = mix.sample_numpy(np.arange(E), 1)
    pose2, light2, scene2, ep2 = _check_sampled_reset(vec, ref2, m)
    assert np.array_equal(ep2, 1 + m.astype(np.uint32))
    assert np.array_equal(pose2[~m], pose[~m], equal_nan=True) and np.array_equal(scene2[~m], scene[~m])
    assert np.any(ref2[3][m] != ref[3][m])              # some envs changed their configuration (and sizes)
    ob.set_env_scene(scene2)
    ob.reset(pose2, light2, mask=m.astype(np.uint8))
    assert np.array_equal(vec.batch.bodies(), ob.bodies())
    _step_both(vec, ob, acts, range(3, 6), flat=True)
    assert not vec.check_status().any()
    # the second half of the global env ids, as a batch of its own, draws the same scenes
    half = KilobotsVecEnv.from_configurations(confs, E // 2, weights=w, seed=seed, env_id_base=base + E // 2)
    half.reset()
    ph, lh, sh, _ = half.batch.get_sampled()
    assert np.array_equal(ph, pose[E // 2:], equal_nan=True) and np.array_equal(lh, light[E // 2:])
    assert np.array_equal(sh, scene[E // 2:])
    half.close()
    vec.close()
    ob.close()


@pytest.mark.gpu
def test_swarm_tier_weighted_mix(oracle, native):
    import torch
    from mixed_oracle import MixedOracle
    light = "!LightConf {type: circular, init: random, radius: .3}"
    # a fixed mean ('mean: light' with a light at the table's edge stacks kilobots on the clip line beyond any contact
    # capacity), spreads that keep the peak density of the Gaussian spawn near a third of the table's area in kilobots
    confs = [_conf(0, 40, light, mean="[0.1, -0.05]", std=.12, width=2.0, height=2.0),
             _conf(0, 100, light, mean="[-0.1, 0.05]", std=.19, width=2.0, height=2.0),
             _conf(0, 300, light, mean="[0.0, 0.0]", std=.33, width=2.0, height=2.0)]
    E = 9
    vec = KilobotsVecEnv.from_configurations(confs, E, weights=[1.0, 1.0, 1.0], seed=4, env_id_base=70)
    assert vec.batch.launch_config()["block_threads"] in (128, 256, 512)   # the swarm tier
    mix, sc = vec.sampler, vec.scenario
    vec.reset()
    ref = mix.sample_numpy(np.arange(E), 0)
    assert len(set(ref[3])) >= 2
    pose, light_s, scene, ep = _check_sampled_reset(vec, ref)
    ob = MixedOracle(oracle, sc.scenes, E, sc.env_scene, sc.max_contacts)
    ob.set_env_scene(scene)
    ob.reset(pose, light_s)
    assert np.array_equal(vec.batch.bodies(), ob.bodies())
    acts = SC.random_actions(sc, E, 4, seed=8)
    _step_both(vec, ob, acts, range(2))
    done = torch.zeros(E, dtype=torch.uint8, device="cuda")
    done[1::2] = 1
    m = done.cpu().numpy().astype(bool)
    vec.reset_done(done)
    ref2 = mix.sample_numpy(np.arange(E), 1)
    pose2, light2, scene2, ep2 = _check_sampled_reset(vec, ref2, m)
    assert np.array_equal(ep2, 1 + m.astype(np.uint32)) and np.array_equal(pose2[~m], pose[~m], equal_nan=True)
    ob.set_env_scene(scene2)
    ob.reset(pose2, light2, mask=m.astype(np.uint8))
    assert np.array_equal(vec.batch.bodies(), ob.bodies())
    _step_both(vec, ob, acts, range(2, 4))
    assert not vec.check_status().any()
    half = KilobotsVecEnv.from_configurations(confs, 4, weights=[1.0, 1.0, 1.0], seed=4, env_id_base=75)
    half.reset()
    ph, _, sh, _ = half.batch.get_sampled()
    assert np.array_equal(ph, pose[5:], equal_nan=True) and np.array_equal(sh, scene[5:])
    half.close()
    vec.close()
    ob.close()


@pytest.mark.gpu
def test_env_config_mode_set_env_scene_moves_an_env_at_its_next_reset(native):
    import torch
    confs = _composite_confs()
    E = 8
    cfg = np.array([0, 1, 2, 0, 1, 2, 0, 1])
    vec = KilobotsVecEnv.from_configurations(confs, E, env_config=cfg, seed=6, env_id_base=30)
    mix = vec.sampler
    vec.reset()
    ref = mix.sample_numpy(np.arange(E), 0, mix.scene_offset[cfg])
    assert np.array_equal(ref[3], cfg)
    _, _, scene, _ = _check_sampled_reset(vec, ref)
    # move env 0 to configuration 2 and env 1 to configuration 0: nothing changes before their next sampled reset
    es = scene.copy()
    es[0], es[1] = mix.first_scene(2), mix.first_scene(0)
    vec.set_env_scene(es)
    counts = vec.batch.body_counts()
    done = torch.zeros(E, dtype=torch.uint8, device="cuda")
    done[2] = 1
    vec.reset_done(done)
    assert np.array_equal(vec.batch.body_counts()[1], counts[1])
    done[:] = 0
    done[:2] = 1
    vec.reset_done(done)
    m = done.cpu().numpy().astype(bool)
    _, _, _, ep = vec.batch.get_sampled()
    ref2 = mix.sample_numpy(np.arange(E), ep.astype(np.int64) - 1, es)
    assert list(ref2[3][:3]) == [2, 0, 2]
    _check_sampled_reset(vec, ref2, m)
    assert list(vec.batch.body_counts()[1][:3]) == [14, 6, 14]
    # a scene of no configuration is refused while the mix is attached
    bad = es.copy()
    bad[0] = 99
    with pytest.raises(RuntimeError):
        vec.set_env_scene(bad)
    vec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("light", ["plain", "shuffled"])
def test_one_spec_mix_equals_set_sampler(native, light):
    """kb_set_sampler_mix with one spec on a homogeneous batch is kb_set_sampler, bit for bit"""
    import torch
    conf = _conf(2, 6, MOMENTUM_AT_OBJECT if light == "plain" else SHUFFLED)
    single = SceneSampler(conf, seed=13, env_id_base=7)
    mix = SamplerMix([conf], seed=13, env_id_base=7)
    E = 40
    pose, lt, scene = single.sample_numpy(np.arange(E), 0)
    specs = single.scene_specs()
    batches = [native.NativeBatch(specs, E, scene, 0) for _ in range(2)]
    batches[0].set_sampler(single)
    batches[1].set_sampler_mix(mix)
    done = torch.zeros(E, dtype=torch.uint8, device="cuda")
    done[::2] = 1
    for mask in (None, done, None):
        outs = []
        for b in batches:
            b.reset_sampled(mask)
            outs.append(b.get_sampled() + (b.bodies(),))
        for x, y in zip(*outs):
            assert np.array_equal(x, y)
    assert np.array_equal(outs[0][3], [3 if e % 2 == 0 else 2 for e in range(E)])
    if light == "shuffled":
        assert set(outs[0][2]) == {0, 1}


@pytest.mark.gpu
def test_set_sampler_mix_refusals(native):
    import ctypes as C
    confs = _composite_confs()
    mix = SamplerMix(confs, weights=[1, 1, 1], seed=1)
    E = 6
    _, _, scene, _ = mix.sample_numpy(np.arange(E), 0)
    scene[:3] = [0, 2, 3]      # every configuration present
    nb = native.NativeBatch(mix.scene_specs(), E, scene, 0)

    def call(specs, k, weights):
        w = None if weights is None else (C.c_double * len(weights))(*weights)
        rc = native._fn["set_sampler_mix"](nb.h, specs, k, w)
        return rc, native._fn["last_error"]().decode()

    specs, K, w, keep = mix.to_abi()
    assert call(specs, K, [1, 1, 1])[0] == 0
    # a scene claimed by two specs: configuration 1 also claims configuration 0's first scene (same counts needed first)
    twin = SamplerMix([confs[0], confs[0]], seed=1)
    nb2 = native.NativeBatch(twin.scene_specs(), E, np.zeros(E, np.int32), 0)
    s2, k2, _, keep2 = twin.to_abi()
    s2[1].perm_scene = s2[0].perm_scene
    rc = native._fn["set_sampler_mix"](nb2.h, s2, k2, None)
    assert rc != 0 and "two specs" in native._fn["last_error"]().decode()
    nb2.close()
    # an env on a scene no spec claims: only the first two configurations
    rc, msg = call(specs, 2, [1, 1])
    assert rc != 0 and "no spec" in msg
    # a spec whose object count does not match its scenes
    specs[1].num_objects = 2
    rc, msg = call(specs, K, None)
    assert rc != 0 and "num_objects" in msg
    specs[1].num_objects = 1
    rc, msg = call(specs, 0, None)
    assert rc != 0 and "1..16" in msg
    many = (abi.KbSampleSpec * 17)(*([specs[1]] * 17))
    rc, msg = call(many, 17, None)
    assert rc != 0 and "1..16" in msg
    rc, msg = call(specs, K, [1, -1, 1])
    assert rc != 0 and "non-negative" in msg
    rc, msg = call(specs, K, [0, 0, 0])
    assert rc != 0 and "positive" in msg
    assert call(specs, K, None)[0] == 0
    nb.close()
