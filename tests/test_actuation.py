"""Actuation model (include/kb_b200.h kb_set_actuation): per-episode motor gains, turn-rate drift and dead kilobots, and
per-sub-step noise, drawn on the device in both kernel tiers.  Checked bit for bit against the CPU oracle with the model
(tests/kbo_actuation.cpp: the unchanged oracle/ sources with the model around their controllers), against the
numpy mirror (gym_kilobots_b200/actuation.py) draw for draw, and -- without a model -- against the step kernels' own
code before the model existed (their SASS)."""
import ctypes
import hashlib
import json
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import yaml

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import actuation as ACT
from gym_kilobots_b200 import scenarios as SC
from gym_kilobots_b200.scene import ActuationSpec

from mixed_oracle import MixedOracle
from parity_util import assert_same_obs, assert_same_state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gym_kilobots_b200", "csrc")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")

FULL = ActuationSpec(seed=11, gain_v_lo=0.6, gain_v_hi=1.4, gain_w_lo=0.5, gain_w_hi=1.5, drift_w=0.3, noise_v=0.2,
                     noise_w=0.3, p_dead=0.1)
IDENTITY = ActuationSpec(seed=5)
PARITY_COUNTERS = [0, 1, 2, 4, 5, 7]   # as parity_util.run_parity: the counters that do not depend on the lane width

CONF = """
!EvalEnv
width: 1.2
height: 0.8
resolution: 600
objects:
  - !ObjectConf {idx: 0, color: null, shape: square, width: .15, height: .10, init: random, symmetry: null}
light: !LightConf {type: circular, init: random, radius: .2}
kilobots: !KilobotsConf {num: 6, mean: light, std: .03}
"""


@pytest.fixture(scope="session")
def act_oracle(oracle, tmp_path_factory):
    """The CPU oracle with the actuation model (tests/kbo_actuation.cpp around the unchanged oracle/ sources), compiled
    with the oracle's own flags (oracle/Makefile); .OracleBatch drives it like oracle.kbo.OracleBatch."""
    import types
    odir = os.path.join(ROOT, "oracle")
    srcs = [os.path.join(odir, f) for f in ("kbo_shapes.cpp", "kbo_collide.cpp", "kbo_solver.cpp", "kbo_toi.cpp",
                                            "kbo_world.cpp")] + [os.path.join(ROOT, "tests", "kbo_actuation.cpp")]
    lib_path = str(tmp_path_factory.mktemp("kbo_actuation") / "libkbo_actuation.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-o",
                           lib_path] + srcs + ["-lpthread"])
    lib = ctypes.CDLL(lib_path)
    fn = abi.bind(lib, "kbo_")
    for name in ("set_actuation", "get_actuation"):
        f = getattr(lib, "kbo_" + name)
        f.restype, f.argtypes = abi.PRODUCT_ONLY[name]
        fn[name] = f
    lib.kbo_set_threads.restype = ctypes.c_int
    lib.kbo_set_threads.argtypes = [ctypes.c_void_p, ctypes.c_int32]

    class OracleBatch(oracle.OracleBatch):
        def __init__(self, scenes, num_envs, env_scene=None, max_contacts=0, threads=1):
            self.lib, self.fn = lib, fn
            scenes = list(scenes) if isinstance(scenes, (list, tuple)) else [scenes]
            self.scenes = scenes
            descs = (abi.KbSceneDesc * len(scenes))()
            self._keep = []
            for i, sp in enumerate(scenes):
                descs[i], keep = sp.to_desc()
                self._keep.append(keep)
            es = None if env_scene is None else np.ascontiguousarray(env_scene, dtype=np.int32)
            h = ctypes.c_void_p()
            rc = fn["create"](descs, len(scenes), None if es is None else es.ctypes.data_as(ctypes.c_void_p), num_envs,
                              max_contacts, 0, ctypes.byref(h))
            assert rc == 0, fn["last_error"]()
            self.h = h
            dims = abi.KbDims()
            fn["get_dims"](h, ctypes.byref(dims))
            self.E, self.B, self.M, self.N = dims.num_envs, dims.num_bodies, dims.num_objects, dims.num_kilobots
            self.P, self.C, self.L, self.A = dims.num_proxies, dims.max_contacts, dims.light_state_dim, dims.action_dim
            self.set_threads(threads)

        def set_actuation(self, spec):
            d = None if spec is None else spec.to_def()
            if fn["set_actuation"](self.h, None if d is None else ctypes.byref(d)) != 0:
                raise ValueError(fn["last_error"]().decode())

        def actuation(self):
            draws = np.zeros((self.E, self.N, 4), np.float32)
            ep = np.zeros(self.E, np.uint32)
            step = ctypes.c_uint64()
            rc = fn["get_actuation"](self.h, draws.ctypes.data_as(ctypes.c_void_p), ep.ctypes.data_as(ctypes.c_void_p),
                                     ctypes.byref(step))
            assert rc == 0, fn["last_error"]()
            return draws, ep, int(step.value)

    return types.SimpleNamespace(OracleBatch=OracleBatch)


def _with(spec, **kw):
    d = dict(spec.__dict__)
    d.update(kw)
    return ActuationSpec(**d)


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_actuation_def_layout_matches_the_header(tmp_path):
    """KbActuationDef as gcc lays it out (sizeof and every field's offset) against the ctypes mirror"""
    fields = [n for n, _ in abi.KbActuationDef._fields_]
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "kb_b200.h"', "int main(void) {",
             'printf("%zu", sizeof(KbActuationDef));']
    lines += ['printf(" %%zu", offsetof(KbActuationDef, %s));' % f for f in fields]
    lines += ['printf("\\n");', "return 0; }"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines))
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got[0] == ctypes.sizeof(abi.KbActuationDef)
    assert got[1:] == [getattr(abi.KbActuationDef, f).offset for f in fields]


def _sass_functions(path):
    """{mangled name: SASS body} of every function in a cubin or shared library"""
    out = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", path], capture_output=True, text=True,
                         check=True).stdout
    res, name, buf = {}, None, []
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m or (name is not None and line.strip().startswith(".....")):
            if name is not None:
                res[name] = "\n".join(buf)
            name, buf = (m.group(1) if m else None), []
        elif name is not None:
            buf.append(line.strip())
    if name is not None:
        res[name] = "\n".join(buf)
    return res


# the headers and options kb_create compiles the specialised step kernel with (csrc/Makefile JIT_HDRS, csrc/kb_jit.h)
JIT_HDRS = ["kb_types.cuh", "kb_narrow.cuh", "kb_sample.cuh", "kb_solver.cuh", "kb_env.cuh", "kb_step.cuh", "kb_toi.cuh",
            "kb_step_kernel.cuh", "../../include/kb_b200.h"]
JIT_OPTIONS = ["-arch=sm_100a", "-fmad=false", "-std=c++17", "-lineinfo", "-default-device", "--ptxas-options=-v"]


def _nvrtc():
    try:
        return ctypes.CDLL(os.path.join(CUDA, "lib64", "libnvrtc.so.12"))
    except OSError:
        return None


def _nvrtc_sass(lib, source, kernel):
    names = [h.encode() for h in JIT_HDRS]
    texts = [open(os.path.join(CSRC, h), "rb").read() for h in JIT_HDRS]
    prog, n = ctypes.c_void_p(), len(names)
    assert lib.nvrtcCreateProgram(ctypes.byref(prog), source.encode(), b"kb_step_jit.cu", n,
                                  (ctypes.c_char_p * n)(*texts), (ctypes.c_char_p * n)(*names)) == 0
    opts = [o.encode() for o in JIT_OPTIONS]
    assert lib.nvrtcCompileProgram(prog, len(opts), (ctypes.c_char_p * len(opts))(*opts)) == 0
    size = ctypes.c_size_t()
    lib.nvrtcGetCUBINSize(prog, ctypes.byref(size))
    cubin = ctypes.create_string_buffer(size.value)
    lib.nvrtcGetCUBIN(prog, cubin)
    lib.nvrtcDestroyProgram(ctypes.byref(prog))
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "step.cubin")
        with open(p, "wb") as f:
            f.write(cubin.raw)
        return _sass_functions(p)[kernel]


def test_step_kernels_without_a_model_are_the_code_they_were(native):
    """Every step kernel that runs without an actuation model -- kb_step_kernel at 4/8/16/32 lanes, kb_swarm_step_kernel
    at every CTA size, and the specialised kernel kb_create compiles for the C2 and C5 layouts -- has the SASS it had
    before the model existed (tests/golden/step_kernels_sass_off.json, recorded with CUDA 12.9)."""
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "step_kernels_sass_off.json")))
    lib = _nvrtc()
    if lib is None or not os.path.exists(os.path.join(CUDA, "bin", "cuobjdump")):
        pytest.skip("needs cuobjdump and NVRTC")
    major, minor = ctypes.c_int(), ctypes.c_int()
    lib.nvrtcVersion(ctypes.byref(major), ctypes.byref(minor))
    if "%d.%d" % (major.value, minor.value) != golden["nvrtc"]:
        pytest.skip("the fingerprints were recorded with CUDA %s" % golden["nvrtc"])
    digest = lambda body: hashlib.sha256(body.encode()).hexdigest()
    got = {}
    for name, body in _sass_functions(os.path.join(CSRC, "libkb_b200.so")).items():
        m = re.match(r"_ZN2kb(?:14|20)(kb_step_kernel|kb_swarm_step_kernel)ILi(\d+)EEEvNS_10KernelArgsE$", name)
        if m:
            got["%s<%s>" % m.groups()] = digest(body)
    for name, sc in (("C2", SC.c2_quad_assembly(64)), ("C5", SC.c5_small(256))):
        src, _, _ = native.jit_step_source(sc.scenes, sc.max_contacts)
        got["kb_step_kernel_jit " + name] = digest(_nvrtc_sass(lib, src, "kb_step_kernel_jit"))
    assert got == golden["kernels"]


def test_mirror_draws_and_noise_ranges():
    spec = _with(FULL, p_dead=0.3)
    d = ACT.episode_draws(spec, np.arange(64), 0, 50)
    assert d.dtype == np.float32 and d.shape == (64, 50, 4)
    assert (d[..., 0] >= 0.6).all() and (d[..., 0] <= 1.4).all() and (d[..., 1] >= 0.5).all() and (d[..., 1] <= 1.5).all()
    assert (np.abs(d[..., 2]) <= 0.3).all() and set(np.unique(d[..., 3])) == {0.0, 1.0}
    assert 0.2 < 1.0 - d[..., 3].mean() < 0.4
    assert not np.array_equal(d, ACT.episode_draws(spec, np.arange(64), 1, 50))
    assert np.array_equal(d[10:20], ACT.episode_draws(spec, np.arange(10, 20), 0, 50))   # a slice draws what the whole does
    fv, fw = ACT.substep_factors(spec, np.arange(64), 3, 7, 50)
    assert (np.abs(fv - 1) <= 0.2).all() and (np.abs(fw - 1) <= 0.3).all()
    ident = ACT.episode_draws(IDENTITY, np.arange(8), 0, 10)
    assert (ident == np.array([1, 1, 0, 1], np.float32)).all()


def test_oracle_draws_match_the_mirror_and_resets_advance_them(act_oracle):
    sc = SC.c2_quad_assembly(8)
    spec = _with(FULL, env_id_base=100)
    ob = act_oracle.OracleBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    ob.set_actuation(spec)
    d, ep, step = ob.actuation()
    assert step == 0 and not ep.any() and np.array_equal(d, ACT.episode_draws(spec, 100 + np.arange(8), 0, ob.N))
    mask = np.array([1, 0, 0, 1, 1, 0, 0, 0], np.uint8)
    ob.reset(sc.body_pose, sc.light_state)
    ob.reset(sc.body_pose, sc.light_state, mask=mask)
    d, ep, _ = ob.actuation()
    assert np.array_equal(ep, 1 + mask) and np.array_equal(d, ACT.episode_draws(spec, 100 + np.arange(8), ep, ob.N))
    ob.step(SC.random_actions(sc, 8, 1)[0])
    assert ob.actuation()[2] == 1


def test_oracle_identity_model_is_the_physics_without_a_model(oracle, act_oracle):
    """the plain oracle against the actuation oracle with the identity model"""
    sc = SC.pushing_yard(3, kilobot_kind=abi.KB_KILOBOT_PHOTOTAXIS, light="circular")
    a = oracle.OracleBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    b = act_oracle.OracleBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    b.set_actuation(IDENTITY)
    for x in (a, b):
        x.reset(sc.body_pose, sc.light_state)
    for act in SC.random_actions(sc, sc.num_envs, 12):
        assert_same_obs(a.step(act), b.step(act), "identity")
    assert_same_state(a, b, "identity")
    b.set_actuation(FULL)   # and a real model changes the physics
    for act in SC.random_actions(sc, sc.num_envs, 3):
        a.step(act), b.step(act)
    assert not np.array_equal(a.bodies(), b.bodies())


@pytest.mark.parametrize("field,value", [("gain_v_lo", np.nan), ("gain_w_hi", np.inf), ("drift_w", -0.1),
                                         ("noise_v", -1e-3), ("noise_w", np.nan), ("gain_v_lo", -0.5),
                                         ("p_dead", 1.5), ("p_dead", -0.1), ("gain_v_lo", 1.5), ("gain_w_lo", 2.0)])
def test_oracle_refuses_invalid_specs(act_oracle, field, value):
    sc = SC.c1_single_env(1)
    ob = act_oracle.OracleBatch(sc.scenes, 1)
    with pytest.raises(ValueError, match=field):
        ob.set_actuation(_with(IDENTITY, **{field: value}))


# ---------------------------------------------------------------------------------------------------------------- GPU
def _twin_run(a, b, sc, steps, actions, mode, where):
    for x in (a, b):
        x.reset(sc.body_pose, sc.light_state)
    assert_same_state(a, b, where + " after reset")
    for t in range(steps):
        assert_same_obs(a.step(actions[t], mode), b.step(actions[t], mode), "%s step %d" % (where, t))
        assert_same_state(a, b, "%s step %d" % (where, t))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c2-jit", "c2-generic", "lanes4", "swarm"])
def test_identity_model_is_bit_identical_to_no_model(native, case, monkeypatch):
    if case == "c2-generic":
        monkeypatch.setenv("KB_JIT", "0")
    if case == "lanes4":
        monkeypatch.setenv("KB_LANES_PER_ENV", "4")
    sc = SC.c4_swarm(2, side=8) if case == "swarm" else SC.c2_quad_assembly(40, degenerate=False)
    a = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    b = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    b.set_actuation(IDENTITY)
    cfg = b.launch_config()
    assert cfg["actuation"] and not a.launch_config()["actuation"]
    assert cfg["specialised"] == a.launch_config()["specialised"], cfg["jit_reason"]
    if case.startswith("c2"):
        assert cfg["specialised"] == (case == "c2-jit"), cfg["jit_reason"]
    if case == "lanes4":
        assert cfg["lanes_per_env"] == 4
    acts = SC.random_actions(sc, sc.num_envs, 20)
    _twin_run(a, b, sc, 20, acts, abi.KB_ACTION_LIGHT, case)
    b.set_actuation(None)   # detached: the off kernel again
    assert not b.launch_config()["actuation"] and b.launch_config()["specialised"] == a.launch_config()["specialised"]


def _on_parity(ob, nb, sc, spec, steps, actions, mode, where):
    ob.set_actuation(spec)
    nb.set_actuation(spec)
    assert np.array_equal(ob.actuation()[0], nb.actuation()[0]), where + ": draws differ"
    _twin_run(ob, nb, sc, steps, actions, mode, where)
    do, eo, so = ob.actuation()
    dn, en, sn = nb.actuation()
    assert np.array_equal(do, dn) and np.array_equal(eo, en) and so == sn == steps
    assert np.array_equal(ob.counters()[:, PARITY_COUNTERS], nb.counters()[:, PARITY_COUNTERS])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["phototaxis", "simple-phototaxis", "direct", "direct-dead", "swarm"])
def test_device_matches_oracle_with_the_model(act_oracle, native, case):
    spec = _with(FULL, env_id_base=7)
    mode = abi.KB_ACTION_LIGHT
    if case == "phototaxis":
        sc = SC.pushing_yard(6, kilobot_kind=abi.KB_KILOBOT_PHOTOTAXIS, light="circular")
    elif case == "simple-phototaxis":
        sc = SC.pushing_yard(6, light="momentum")
    elif case == "swarm":
        sc = SC.c4_swarm(2, side=8)
    else:
        sc = SC.direct_control(12)
        mode = abi.KB_ACTION_KILOBOTS
        if case == "direct-dead":
            spec = _with(spec, p_dead=0.3)
    steps = 12
    acts = SC.random_kilobot_actions(sc, sc.num_envs, steps) if mode == abi.KB_ACTION_KILOBOTS else \
        SC.random_actions(sc, sc.num_envs, steps)
    ob = act_oracle.OracleBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts, threads=8)
    nb = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    _on_parity(ob, nb, sc, spec, steps, acts, mode, case)
    if case == "direct-dead":
        assert (nb.actuation()[0][..., 3] == 0).any()


@pytest.mark.gpu
def test_device_matches_oracle_with_the_model_in_a_mixed_count_batch(act_oracle, native):
    """one compact oracle world per env (MixedOracle), each with the env's global id as its env_id_base"""
    homs = [SC.c2_quad_assembly(3, seed=1, degenerate=False), SC.c1_single_env(3, seed=2)]
    specs = [h.scenes[0] for h in homs]
    es = np.array([e % 2 for e in range(6)], np.int32)
    pose = SC.stack_poses(specs, es, [homs[e % 2].body_pose[e // 2] for e in range(6)])
    light = np.stack([homs[e % 2].light_state[e // 2] for e in range(6)])
    sc = SC.Scenario("mixed", specs, es, pose, light, 320)
    ob = MixedOracle(act_oracle, sc.scenes, sc.num_envs, sc.env_scene, 320)
    nb = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, 320)
    for e, o in enumerate(ob.envs):
        o.set_actuation(_with(FULL, env_id_base=e))
    nb.set_actuation(FULL)
    n = nb.body_counts()[1]
    draws = nb.actuation()[0]
    for e, o in enumerate(ob.envs):
        assert np.array_equal(o.actuation()[0][0], draws[e, :n[e]])
    ob.reset(sc.body_pose, sc.light_state)
    nb.reset(sc.body_pose, sc.light_state)
    acts = SC.random_actions(2, sc.num_envs, 12, seed=7)
    for t in range(12):
        oo, on = ob.step(acts[t]), nb.step(acts[t])
        for k in oo:
            assert np.array_equal(oo[k], on[k], equal_nan=k in ("kilobots", "objects")), (t, k)
        assert_same_state(ob, nb, "mixed step %d" % t)
    ob.close()


@pytest.mark.gpu
def test_device_draws_match_the_mirror_through_resets(native):
    from gym_kilobots_b200.envs.vec_env import KilobotsVecEnv
    conf = yaml.load(CONF, Loader=yaml.Loader)
    E = 24
    spec = _with(FULL, env_id_base=1000)
    vec = KilobotsVecEnv.from_configuration(conf, E, seed=3, env_id_base=1000, actuation=spec)
    nb, ids = vec.batch, 1000 + np.arange(E)
    d, ep, step = nb.actuation()
    assert step == 0 and not ep.any() and np.array_equal(d, ACT.episode_draws(spec, ids, 0, nb.N))
    assert np.array_equal(vec.actuation_draws(), d)
    mask = (np.arange(E) % 3 == 0).astype(np.uint8)
    nb.reset(vec.scenario.body_pose, vec.scenario.light_state, None, mask)       # kb_reset, masked
    d, ep, _ = nb.actuation()
    assert np.array_equal(ep, mask) and np.array_equal(d, ACT.episode_draws(spec, ids, ep, nb.N))
    vec.reset()                                                                  # kb_reset_sampled, all envs
    vec.step(SC.random_actions(vec.scenario, E, 1)[0])
    vec.reset_done(1 - mask)                                                     # kb_reset_sampled, masked
    d, ep, step = nb.actuation()
    assert np.array_equal(ep, mask + 1 + (1 - mask)) and step == 1
    assert np.array_equal(d, ACT.episode_draws(spec, ids, ep, nb.N))
    vec.close()


@pytest.mark.gpu
def test_two_half_batches_equal_one_batch(native):
    """One handle of 2E envs and two handles of E envs with env_id_base 0 and E draw the same and step the same"""
    E = 10
    whole = SC.c2_quad_assembly(2 * E, degenerate=False)
    halves = [SC.c2_quad_assembly(E, env_offset=h * E, degenerate=False) for h in (0, 1)]
    assert np.array_equal(np.concatenate([h.body_pose for h in halves]), whole.body_pose)
    nw = native.NativeBatch(whole.scenes, 2 * E, whole.env_scene, whole.max_contacts)
    nw.set_actuation(FULL)
    nh = [native.NativeBatch(h.scenes, E, h.env_scene, h.max_contacts) for h in halves]
    for i, b in enumerate(nh):
        b.set_actuation(_with(FULL, env_id_base=i * E))
    nw.reset(whole.body_pose, whole.light_state)
    for b, h in zip(nh, halves):
        b.reset(h.body_pose, h.light_state)
    acts = SC.random_actions(whole, 2 * E, 10)
    for t in range(10):
        ow = nw.step(acts[t])
        oh = [b.step(acts[t][i * E:(i + 1) * E]) for i, b in enumerate(nh)]
        for k in ow:
            assert np.array_equal(ow[k], np.concatenate([o[k] for o in oh])), (t, k)
    assert np.array_equal(nw.actuation()[0], np.concatenate([b.actuation()[0] for b in nh]))
    assert np.array_equal(nw.bodies(), np.concatenate([b.bodies() for b in nh]))


def _one_velocity_kilobot(E, steps_per_action):
    """E envs of one velocity-controlled kilobot alone in a large table: every motion is its own"""
    from gym_kilobots_b200 import scene as S
    spec = S.SceneSpec(bodies=[S.kilobot_body(abi.KB_KILOBOT_VELOCITY)], num_objects=0, lights=[], world_size=(2.0, 2.0),
                       steps_per_action=steps_per_action)
    pose = np.zeros((E, 1, 3))
    return SC.Scenario("one-kilobot", [spec], None, pose, np.zeros((E, 0)), max_contacts=0)


@pytest.mark.gpu
def test_dead_kilobots_do_not_drive(native):
    sc = _one_velocity_kilobot(4, 10)
    nb = native.NativeBatch(sc.scenes, 4, None, 0)
    nb.set_actuation(ActuationSpec(p_dead=1.0))
    nb.reset(sc.body_pose, None)
    fwd = np.tile([0.01, 0.0], (4, 1))
    for _ in range(5):
        out = nb.step(fwd, abi.KB_ACTION_KILOBOTS)
    assert (nb.actuation()[0][..., 3] == 0).all()
    assert np.array_equal(out["kilobots"][:, 0, :2], np.zeros((4, 2), np.float32))
    nb.set_actuation(None)   # the same command moves a live kilobot
    out = nb.step(fwd, abi.KB_ACTION_KILOBOTS)
    assert (out["kilobots"][:, 0, 0] > 0.005).all()


@pytest.mark.gpu
def test_speed_noise_factors_seen_on_the_device(native):
    """One sub-step per env-step: a free kilobot's speed after the step, over its speed without noise, is f_v"""
    E, T = 16, 8
    sc = _one_velocity_kilobot(E, 1)
    spec = ActuationSpec(seed=9, noise_v=0.2)
    a = native.NativeBatch(sc.scenes, E, None, 0)
    b = native.NativeBatch(sc.scenes, E, None, 0)
    b.set_actuation(spec)
    for x in (a, b):
        x.reset(sc.body_pose, None)
    fwd = np.tile([0.01, 0.0], (E, 1))
    ratios = []
    for t in range(T):
        a.step(fwd, abi.KB_ACTION_KILOBOTS)
        b.step(fwd, abi.KB_ACTION_KILOBOTS)
        va, vb = a.bodies()[:, 0, 3], b.bodies()[:, 0, 3]
        ratios.append(vb.astype(np.float64) / va)
        fv, _ = ACT.substep_factors(spec, np.arange(E), t, 0, 1)
        assert np.allclose(ratios[-1], fv[:, 0], rtol=1e-6, atol=0)
    r = np.array(ratios)
    assert (r >= 0.8 - 1e-6).all() and (r <= 1.2 + 1e-6).all()
    assert len(np.unique(np.round(r[:, 0], 6))) == T   # a new factor every sub-step


@pytest.mark.gpu
def test_device_refuses_invalid_specs_naming_the_field(native):
    sc = SC.c1_single_env(1)
    nb = native.NativeBatch(sc.scenes, 1)
    for field, value in (("gain_v_hi", np.nan), ("noise_w", -0.5), ("p_dead", 2.0), ("gain_w_lo", 3.0)):
        with pytest.raises(RuntimeError, match=field):
            nb.set_actuation(_with(IDENTITY, **{field: value}))
    with pytest.raises(RuntimeError, match="no actuation model"):
        nb.actuation()
