"""The step kernel compiled at kb_create for the batch's layout (csrc/kb_jit.h): its generated source compiles with NVRTC
for every lane width without spilling (no GPU needed), and on the GPU it computes bit for bit what the generic
kb_step_kernel<LPE> computes, through the kernel cache (memory and disk) and its fallbacks."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import _native as native
from gym_kilobots_b200 import scenarios as SC
from gym_kilobots_b200.scene import TaskSpec

STEPS = 20


def _mixed(per=6):
    """Envs of three sizes in one batch (C2', 1 quad + 10 kilobots, an L-form + 40 kilobots): the layout is the padded
    maxima, 4 objects + 40 kilobots, on 32-lane groups."""
    homs = [SC.c2_quad_assembly(per, seed=1, degenerate=False), SC.c1_single_env(per, seed=2),
            SC.c3_shapes(per, seed=3, num_kilobots=40)]
    specs = [h.scenes[0] for h in homs]
    env_scene = np.array([e % 3 for e in range(3 * per)], np.int32)
    poses = [homs[e % 3].body_pose[e // 3] for e in range(3 * per)]
    light = np.stack([homs[e % 3].light_state[e // 3] for e in range(3 * per)])
    return SC.Scenario("mixed", specs, env_scene, SC.stack_poses(specs, env_scene, poses), light, 320)


SCENARIOS = {
    "C2": lambda: SC.c2_quad_assembly(24),
    "C2p": lambda: SC.c2_quad_assembly(24, degenerate=False),
    "C3": lambda: SC.c3_shapes(12),
    "C3_30": lambda: SC.c3_shapes(12, num_kilobots=30),   # 31 bodies: 16-lane groups
    "C5": lambda: SC.c5_small(256),
    "mixed": _mixed,
    "direct": lambda: SC.direct_control(16),
}
LANES = {"C2": 8, "C2p": 8, "C3": 32, "C3_30": 16, "C5": 4, "mixed": 32, "direct": 8}


def _generic_resources(lpe):
    """(registers, stack bytes) of the generic kb_step_kernel<lpe> in the built library, from cuobjdump."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "-res-usage", native._LIB_PATH], capture_output=True, text=True, check=True).stdout
    name = "_ZN2kb14kb_step_kernelILi%dEEEvNS_10KernelArgsE" % lpe
    m = re.search(re.escape(name) + r":?\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    assert m, "kb_step_kernel<%d> not found in the library" % lpe
    return int(m.group(1)), int(m.group(2))


@pytest.mark.parametrize("name", ["C2", "C2p", "C3", "C3_30", "C5", "mixed"])
def test_specialised_source_compiles_without_spills(name):
    sc = SCENARIOS[name]()
    src, log, ms = native.jit_step_source(sc.scenes, sc.max_contacts, compile=True)
    lpe = LANES[name]
    assert "struct JitLayout" in src and "stepKernelBody<%d>" % lpe in src
    m = re.search(r"Function properties for kb_step_kernel_jit\s*\n.*?(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads", log)
    assert m, log[-2000:]
    stack, spill_st, spill_ld = (int(x) for x in m.groups())
    # the generic 32-lane kernel spills too (152 / 196 bytes at its 128-register bound); the narrower ones do not
    assert lpe == 32 or (spill_st == 0 and spill_ld == 0)
    assert stack <= _generic_resources(lpe)[1]
    assert ms > 0.0


def test_specialised_source_is_exact_layout():
    """Floats are written as hex literals, so the compile-time layout carries the runtime Layout's bits."""
    sc = SC.c2_quad_assembly(4)
    src, _, _ = native.jit_step_source(sc.scenes, sc.max_contacts)
    dt = float.fromhex(re.search(r"float dt = (\S+)f;", src).group(1))
    assert np.float32(dt) == np.float32(sc.scenes[0].dt) and dt == float(np.float32(dt))
    assert re.search(r"int32_t B = 19;", src) and re.search(r"int32_t lanesPerEnv = 8;", src)


def _batch(sc, jit, monkeypatch):
    monkeypatch.setenv("KB_JIT", jit)
    try:
        nb = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts)
    finally:
        monkeypatch.delenv("KB_JIT")
    nb.reset(sc.body_pose, sc.light_state)
    return nb


def _run_pair(sc, monkeypatch, actions, mode=None, task=None, masked_reset=False):
    """The same seeded batch through a generic and a specialised handle: every output and the whole state blob equal."""
    pair = [_batch(sc, "0", monkeypatch), _batch(sc, "1", monkeypatch)]
    assert [nb.launch_config()["specialised"] for nb in pair] == [False, True]
    assert pair[0].launch_config()["jit_reason"] == "KB_JIT=0" and pair[1].launch_config()["jit_reason"] == ""
    if task is not None:
        rng = np.random.default_rng(7)
        targets = np.stack([rng.uniform(-.5, .5, sc.num_envs), rng.uniform(-.5, .5, sc.num_envs),
                            rng.uniform(-3, 3, sc.num_envs)], axis=-1)
        for nb in pair:
            nb.set_task(task, targets)
    rng = np.random.default_rng(11)
    for t in range(STEPS):
        if masked_reset and t == STEPS // 2:
            mask = (rng.random(sc.num_envs) < 0.5).astype(np.uint8)
            for nb in pair:
                nb.reset(sc.body_pose, sc.light_state, mask=mask)
        a = None if actions is None else actions[t % len(actions)]
        out = [nb.step(a, mode) for nb in pair]
        for k in out[0]:
            assert np.array_equal(out[0][k], out[1][k], equal_nan=True), "env-step %d: %s differs" % (t, k)
    assert np.array_equal(pair[0].get_state(), pair[1].get_state())
    assert np.array_equal(pair[0].get_status(), pair[1].get_status())
    return pair


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C2p", "C3", "C3_30", "C5", "mixed"])
def test_specialised_matches_generic(name, monkeypatch, tmp_path):
    monkeypatch.setenv("KB_JIT_CACHE", str(tmp_path))
    sc = SCENARIOS[name]()
    acts = SC.random_actions(sc, sc.num_envs, 8)
    task = TaskSpec(mode=abi.KB_TASK_OBJECT_TO_TARGET, object=0, w_position=1.0, w_orientation=0.25,
                    step_penalty=0.001, success_bonus=2.0, position_tolerance=0.5, orientation_tolerance=1.0,
                    max_episode_steps=7)
    pair = _run_pair(sc, monkeypatch, acts, task=task, masked_reset=True)
    assert pair[1].launch_config()["lanes_per_env"] == LANES[name]


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [4, 8, 16, 32])
def test_specialised_matches_generic_every_lane_width(lanes, monkeypatch, tmp_path):
    monkeypatch.setenv("KB_JIT_CACHE", str(tmp_path))
    monkeypatch.setenv("KB_LANES_PER_ENV", str(lanes))
    sc = SC.c2_quad_assembly(16, degenerate=False)
    pair = _run_pair(sc, monkeypatch, SC.random_actions(sc, sc.num_envs, 8))
    assert pair[1].launch_config()["lanes_per_env"] == lanes


@pytest.mark.gpu
def test_specialised_matches_generic_direct_control(monkeypatch, tmp_path):
    monkeypatch.setenv("KB_JIT_CACHE", str(tmp_path))
    sc = SCENARIOS["direct"]()
    _run_pair(sc, monkeypatch, SC.random_kilobot_actions(sc, sc.num_envs, 8), mode=abi.KB_ACTION_KILOBOTS,
              masked_reset=True)


def _create_in_new_process(cache):
    """(specialised, jit_ms) of two C2 handles created one after the other in a fresh process (the kernel cache of a
    process lives as long as the process) with the disk cache at `cache`."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from gym_kilobots_b200 import _native as native, scenarios as SC\n"
            "sc = SC.c2_quad_assembly(8)\n"
            "for _ in range(2):\n"
            "    c = native.NativeBatch(sc.scenes, sc.num_envs, sc.env_scene, sc.max_contacts).launch_config()\n"
            "    print(c['specialised'], c['jit_ms'])\n") % root
    env = dict(os.environ, KB_JIT="1", KB_JIT_CACHE=str(cache))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    w = out.stdout.split()[-4:]
    return [(w[0] == "True", float(w[1])), (w[2] == "True", float(w[3]))]


@pytest.mark.gpu
def test_kernel_cache(tmp_path):
    """The first handle of a layout compiles, a second one in the same process takes the loaded kernel, a new process
    takes it from the disk cache, and a corrupted or truncated cache file is recompiled and rewritten."""
    (first, second) = _create_in_new_process(tmp_path)
    assert first[0] and first[1] > 0.0
    assert second == (True, 0.0)
    files = list(tmp_path.glob("step_*.cubin"))
    assert len(files) == 1
    intact = files[0].read_bytes()
    assert _create_in_new_process(tmp_path)[0] == (True, 0.0)
    bad = bytearray(intact)
    bad[len(bad) // 2] ^= 0xFF
    for broken in (bytes(bad), intact[: len(intact) // 3]):
        files[0].write_bytes(broken)
        spec, ms = _create_in_new_process(tmp_path)[0]
        assert spec and ms > 0.0
        assert files[0].read_bytes() == intact


@pytest.mark.gpu
def test_generic_on_request(monkeypatch):
    nb = _batch(SC.c2_quad_assembly(4), "0", monkeypatch)
    cfg = nb.launch_config()
    assert cfg["specialised"] is False and cfg["jit_reason"] == "KB_JIT=0" and cfg["jit_ms"] == 0.0
