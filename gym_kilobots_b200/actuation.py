"""numpy mirror of the actuation model (include/kb_b200.h kb_set_actuation, csrc/kb_env.cuh).

The device draws every kilobot's actuation as a pure function of (seed, global env id, episode or step), so the draws
can be recomputed anywhere: for logging, for a privileged critic, or to check the device bit for bit.  Uniform
distributions only, so that the device, the oracle and numpy agree exactly.
"""
import numpy as np

from .philox import EnvRng, _to_double, philox4x32

STREAM_ACTUATION = 9          # per-episode draws: draw indices 2k, 2k + 1
STREAM_ACTUATION_NOISE = 10   # per-sub-step noise


def episode_draws(spec, env_ids, episodes, num_kilobots):
    """float32 [E, N, 4] = (g_v, g_w, d_w, alive) of every kilobot slot of the global envs `env_ids` in their actuation
    episodes (scalar or [E]).  spec: scene.ActuationSpec (its env_id_base is not used: env_ids are global)."""
    env_ids = np.asarray(env_ids, np.int64).reshape(-1)
    rng = EnvRng(spec.seed & 0xFFFFFFFFFFFFFFFF, env_ids.astype(np.uint64),
                 np.broadcast_to(np.asarray(episodes, np.uint64), env_ids.shape))
    k = np.arange(num_kilobots, dtype=np.uint64)[None, :]
    u0, u1 = rng.uniform2(STREAM_ACTUATION, np.broadcast_to(2 * k, (len(env_ids), num_kilobots)))
    u2, u3 = rng.uniform2(STREAM_ACTUATION, np.broadcast_to(2 * k + 1, (len(env_ids), num_kilobots)))
    out = np.empty((len(env_ids), num_kilobots, 4), np.float32)
    out[..., 0] = spec.gain_v_lo + (spec.gain_v_hi - spec.gain_v_lo) * u0
    out[..., 1] = spec.gain_w_lo + (spec.gain_w_hi - spec.gain_w_lo) * u1
    out[..., 2] = spec.drift_w * (2.0 * u2 - 1.0)
    out[..., 3] = np.where(u3 < spec.p_dead, 0.0, 1.0)
    return out


def substep_noise(spec, env_ids, step, substep, num_kilobots):
    """(xi_v, xi_w) float64 [E, N] in [-1, 1) of sub-step `substep` of the env-step whose step count (kb_step calls since
    kb_set_actuation) is `step`."""
    g = np.asarray(env_ids, np.int64).reshape(-1).astype(np.uint64)[:, None]
    k = np.arange(num_kilobots, dtype=np.uint64)[None, :]
    mask = np.uint64(0xFFFFFFFF)
    seed = int(spec.seed) & 0xFFFFFFFFFFFFFFFF
    c0 = k | np.uint64(int(substep) << 16)
    c1 = np.uint64(int(step) & 0xFFFFFFFF)
    c3 = (np.uint64(STREAM_ACTUATION_NOISE) | ((g >> np.uint64(32)) << np.uint64(8))) & mask
    r0, r1, r2, r3 = philox4x32(c0 & mask, c1, g & mask, c3, np.uint32(seed & 0xFFFFFFFF), np.uint32(seed >> 32))
    return 2.0 * _to_double(r0, r1) - 1.0, 2.0 * _to_double(r2, r3) - 1.0


def substep_factors(spec, env_ids, step, substep, num_kilobots):
    """(f_v, f_w) float32 [E, N]: the factors on speed and turn rate, (float)(1 + noise * xi); 1 without noise."""
    xv, xw = substep_noise(spec, env_ids, step, substep, num_kilobots)
    return (1.0 + spec.noise_v * xv).astype(np.float32), (1.0 + spec.noise_w * xw).astype(np.float32)
