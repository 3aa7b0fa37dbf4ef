"""Per-kilobot local observations in numpy: the contract of kb_local_observation (include/kb_b200.h), evaluated on the
CPU from what the batch reports -- the body state of `kb_get_bodies` and the observation of the last step.  Product
code: usable without a GPU (e.g. to build the observation of a recorded state), and the reference the device kernels
(csrc/kb_local.cuh) are tested against.  Float32 operations are evaluated one at a time as numpy does, which is what the
kernels do (no fused multiply-add), so the neighbour and object parts agree bit for bit; the light part is float64
arithmetic rounded to float32 (sin / cos of a linear light come from numpy, so it may differ by 1 float32 ulp)."""
import numpy as np

from . import _abi as abi

_F = np.float32


def _light_value_grad(light, ls, sx, sy):
    """lightValueGrad (csrc/kb_env.cuh) of one light, float64, vectorised over the sensor points."""
    if light.type == abi.KB_LIGHT_LINEAR:
        vx, vy = np.cos(ls[0]), np.sin(ls[0])
        return vx * sx + vy * sy, np.full_like(sx, vx), np.full_like(sy, vy)
    g0 = -1 * (sx - ls[0])
    g1 = -1 * (sy - ls[1])
    norm = np.sqrt(g0 * g0 + g1 * g1)
    radius = float(light.radius)
    v = 1.0 - norm / radius
    v = np.where(v < 1.0, v, 1.0)
    v = np.where(v > 0.0, v, 0.0) * 255
    with np.errstate(invalid="ignore", divide="ignore"):
        g0 = np.where(norm == 0.0, 0.0, g0 / norm)
        g1 = np.where(norm == 0.0, 0.0, g1 / norm)
    far = norm > radius
    return v, np.where(far, g0 * 0.0, g0), np.where(far, g1 * 0.0, g1)


def _light_part(scene, bodies_e, M, n, ls):
    """[n, 3]: light value and body-frame gradient at each present kilobot's sensor point."""
    xf = bodies_e[M:M + n]
    px, py, s, c = xf[:, 8], xf[:, 9], xf[:, 10], xf[:, 11]
    kinds = np.array([b.kind for b in scene.bodies[scene.num_objects:]], np.int64)
    # senseControl: the body origin of a SimplePhototaxisKilobot, else the rear point (0, -r) through b2Mul(xf, .)
    lx, ly = _F(25.0 * 0.0), _F(25.0 * -0.0165)
    wx = (c * lx - s * ly) + px
    wy = (s * lx + c * ly) + py
    simple = kinds == abi.KB_KILOBOT_SIMPLE_PHOTOTAXIS
    sx = np.where(simple, px, wx).astype(np.float64) / 25.0
    sy = np.where(simple, py, wy).astype(np.float64) / 25.0
    value = np.zeros(n)
    gx, gy = np.zeros(n), np.zeros(n)
    best = np.zeros(n)
    so = 0
    for l, light in enumerate(scene.lights):
        v, g0, g1 = _light_value_grad(light, ls[so:], sx, sy)
        if len(scene.lights) == 1:
            value, gx, gy = v, g0, g1
        else:
            value = value + v
            take = np.ones(n, bool) if l == 0 else v > best
            best = np.where(take, v, best)
            gx, gy = np.where(take, g0, gx), np.where(take, g1, gy)
        so += light.state_dim
    cd, sd = c.astype(np.float64), s.astype(np.float64)
    return np.stack([value, cd * gx + sd * gy, -sd * gx + cd * gy], axis=-1).astype(_F)


def local_observation_numpy(spec, bodies, obs_kilobots, obs_objects, light_state, scenes, env_scene=None):
    """float32 [E, Nmax, D] (D = spec.dim(Mmax)), what kb_local_observation writes.

    spec          scene.LocalObsSpec
    bodies        [E, B, 12] float32, NativeBatch.bodies() (kb_get_bodies): xf.p (b2 units) and xf.q = (sin, cos)
    obs_kilobots  [E, Nmax, 3] float32, obs_objects [E, Mmax, 3] float32: the step's observation (positions in metres)
    light_state   [E, L] float64: the light state (obs['light'])
    scenes        the batch's scene templates (scene.SceneSpec); env_scene [E]: the scene each env was last reset with
                  (None = all scene 0)"""
    bodies = np.asarray(bodies, _F)
    kb = np.asarray(obs_kilobots, _F)
    ob = np.asarray(obs_objects, _F)
    E, N = kb.shape[:2]
    M = ob.shape[1]
    if spec.objects and M == 0:
        raise ValueError("local observation: the objects part needs a batch with objects")
    if spec.light and not scenes[0].lights:
        raise ValueError("local observation: the light part needs a batch with lights")
    K = int(spec.max_neighbours)
    r2 = _F(spec.radius) * _F(spec.radius)
    sl = spec.slices(M)
    out = np.full((E, N, spec.dim(M)), np.nan, _F)
    es = np.zeros(E, np.int64) if env_scene is None else np.asarray(env_scene, np.int64)
    light_state = np.asarray(light_state, np.float64).reshape(E, -1)
    for e in range(E):
        scene = scenes[es[e]]
        n, m = scene.num_kilobots, scene.num_objects
        if n == 0:
            continue
        p = kb[e, :n, :2]
        s, c = bodies[e, M:M + n, 10], bodies[e, M:M + n, 11]
        row = out[e, :n]
        if spec.neighbours:
            dx = p[None, :, 0] - p[:, None, 0]          # [i, j]: p_j - p_i
            dy = p[None, :, 1] - p[:, None, 1]
            d2 = dx * dx + dy * dy
            hit = d2 <= r2
            np.fill_diagonal(hit, False)
            key = (d2.view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.arange(n, dtype=np.uint64)[None, :]
            key = np.where(hit, key, np.uint64(0xFFFFFFFFFFFFFFFF))
            key = np.sort(key, axis=1)[:, :K]
            nb = np.zeros((n, K, 4), _F)
            filled = key != np.uint64(0xFFFFFFFFFFFFFFFF)
            ii, kk = np.nonzero(filled)
            j = (key[ii, kk] & np.uint64(0xFFFFFFFF)).astype(np.int64)
            ddx, ddy = dx[ii, j], dy[ii, j]
            nb[ii, kk, 0] = c[ii] * ddx + s[ii] * ddy
            nb[ii, kk, 1] = -s[ii] * ddx + c[ii] * ddy
            nb[ii, kk, 2] = np.sqrt(d2[ii, j])
            nb[ii, kk, 3] = 1.0
            cols = sl["neighbours"]
            row[:, cols.start] = hit.sum(axis=1).astype(_F)
            row[:, cols.start + 1:cols.stop] = nb.reshape(n, 4 * K)
        if spec.objects:
            po = ob[e, :m, :2]
            so, co = bodies[e, :m, 10], bodies[e, :m, 11]
            obj = np.zeros((n, M, 5), _F)
            dx = po[None, :, 0] - p[:, None, 0]
            dy = po[None, :, 1] - p[:, None, 1]
            ci, si = c[:, None], s[:, None]
            obj[:, :m, 0] = ci * dx + si * dy
            obj[:, :m, 1] = -si * dx + ci * dy
            obj[:, :m, 2] = co[None, :] * ci + so[None, :] * si
            obj[:, :m, 3] = so[None, :] * ci - co[None, :] * si
            obj[:, :m, 4] = 1.0
            row[:, sl["objects"]] = obj.reshape(n, 5 * M)
        if spec.light:
            row[:, sl["light"]] = _light_part(scene, bodies[e], M, n, light_state[e])
    return out
