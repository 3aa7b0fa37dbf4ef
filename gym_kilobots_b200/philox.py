"""Counter-based random numbers (Philox4x32-10) keyed by (seed, global env id, stream, draw index).

The reference draws its random scenes from numpy's global generator, one env at a time
(gym_kilobots/envs/yaml_kilobots_env.py:194-198,256-265,299,327-354).  A batched simulator needs draws
that do not depend on how many environments share a batch or a rank, so every draw here is a pure
function of (seed, env id, stream, index): the numpy implementation below and the device one in
csrc/kb_reset_sample.cuh evaluate the same function, a slice of a batch sees the same numbers as the
whole batch, and 1 GPU and 8 GPUs reset an environment identically.

Philox4x32-10: Salmon et al., "Parallel random numbers: as easy as 1, 2, 3" (SC'11); constants as in
Random123 / cuRAND / numpy.random.Philox.
"""
import numpy as np

_M0 = np.uint64(0xD2511F53)
_M1 = np.uint64(0xCD9E8D57)
_W0 = np.uint32(0x9E3779B9)
_W1 = np.uint32(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)

# streams (one per kind of quantity, so that adding a draw to one never shifts another)
STREAM_LIGHT = 1
STREAM_OBJECT = 2
STREAM_KILOBOT_POS = 3
STREAM_KILOBOT_ANGLE = 4
STREAM_SWARM = 5
STREAM_SHUFFLE = 6
STREAM_ACTION = 7
STREAM_CONFIG = 8      # the configuration of a reset in a batch that mixes several (sampler.SamplerMix)


def philox4x32(c0, c1, c2, c3, k0, k1):
    """Ten rounds of Philox4x32 on arrays of uint32 counters / keys (broadcast); returns 4 uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint32) for c in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = np.broadcast_to(np.asarray(k0, dtype=np.uint32), c0.shape).copy()
    k1 = np.broadcast_to(np.asarray(k1, dtype=np.uint32), c0.shape).copy()
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = c0.astype(np.uint64) * _M0
            p1 = c2.astype(np.uint64) * _M1
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & _MASK).astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & _MASK).astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0 = k0 + _W0
            k1 = k1 + _W1
    return c0, c1, c2, c3


def _to_double(hi, lo):
    """53-bit uniform in [0, 1) from two uint32 (the construction numpy and cuRAND use)."""
    return ((hi >> np.uint32(5)).astype(np.float64) * 67108864.0 + (lo >> np.uint32(6)).astype(np.float64)) / 9007199254740992.0


class EnvRng:
    """Per-env counter-based streams for a set of global env ids."""

    def __init__(self, seed, env_ids, episode=0):
        """episode: scalar or [E] -- the number of sampled resets the env has had (device: kb_sample.cuh)."""
        self.seed = int(seed)
        self.env = np.asarray(env_ids, dtype=np.uint64)
        self.episode = np.broadcast_to(np.asarray(episode, dtype=np.uint64), self.env.shape)

    def _raw(self, stream, index, sel=None):
        env = self.env if sel is None else self.env[sel]
        ep = self.episode if sel is None else self.episode[sel]
        idx = np.asarray(index, dtype=np.uint64)
        shp = (lambda a: a.reshape(a.shape + (1,) * (idx.ndim - 1)) if idx.ndim > 1 else a)
        env_b, ep_b, idx_b = np.broadcast_arrays(shp(env), shp(ep), idx)
        c1 = (np.uint64(stream) + (ep_b << np.uint64(8))) & _MASK
        return philox4x32(idx_b & _MASK, c1, env_b & _MASK, env_b >> np.uint64(32),
                          np.uint32(self.seed & 0xFFFFFFFF), np.uint32((self.seed >> 32) & 0xFFFFFFFF))

    def uniform2(self, stream, index, sel=None):
        """Two uniforms in [0, 1) per (env, index): arrays shaped like broadcast(env, index)."""
        r0, r1, r2, r3 = self._raw(stream, index, sel)
        return _to_double(r0, r1), _to_double(r2, r3)

    def normal2(self, stream, index, sel=None):
        """Two independent standard normals per (env, index) (Box-Muller on the two uniforms)."""
        u1, u2 = self.uniform2(stream, index, sel)
        r = np.sqrt(-2.0 * np.log(1.0 - u1))
        a = 6.283185307179586 * u2
        return r * np.cos(a), r * np.sin(a)
