"""The formats of the golden fixtures under tests/golden/ (written by tests/golden/gen_golden*.py), decoded once for the
CPU tier and the GPU tier.  numpy only: no torch, no CUDA.

Images are stored as np.packbits of their binary planes; rewards as the bit patterns (int64) of the float64 the
reference returned; a trace file holds one array per env e and key, named e<e>_<key>."""
import os

import numpy as np


def unpack(bits, shape):
    """float32 images of `shape` from packed bits [..., nbytes] (leading axes kept)."""
    n = int(np.prod(shape))
    return np.unpackbits(bits, axis=-1)[..., :n].reshape(bits.shape[:-1] + tuple(shape)).astype(np.float32)


def f64(bits):
    """The float64 whose bit pattern is `bits`."""
    return np.asarray(bits, dtype=np.int64).view(np.float64)


def reward_f32_bits(f64_bits):
    """The float32 bit pattern (uint32) of a float64 reward given by its bit pattern: what the batched API returns for
    a reward the reference returned.  A scalar or an array."""
    return f64(f64_bits).astype(np.float32).view(np.uint32)


def _replicate(small):
    """x7 replication of the 5x5 crops on the last two axes: the reference's 35x35 planes."""
    return np.repeat(np.repeat(small, 7, -2), 7, -1)


def fov_image(bits, visit):
    """lmaze-v4 / v5 (7,35,35) foveal images from the five packed binary crops [..., 16] and the two float visit
    crops [..., 2, 5, 5], which are channels 2 and 6."""
    b = unpack(bits, (5, 5, 5))
    small = np.stack([b[..., 0, :, :], b[..., 1, :, :], visit[..., 0, :, :], b[..., 2, :, :], b[..., 3, :, :],
                      b[..., 4, :, :], visit[..., 1, :, :]], axis=-3)
    return _replicate(small)


def loc_image(bits):
    """lmaze-v5 (4,35,35) local images from the packed binary crops [..., 13]."""
    return _replicate(unpack(bits, (4, 5, 5)))


def pack_v2_spawn(s5):
    """(bx, by, gx, gy, layout) rows [..., >=5] -> the oracle's 4-int spawn rows (layout in bits 5.. of the last)."""
    s5 = np.asarray(s5)
    return np.stack([s5[..., 0], s5[..., 1], s5[..., 2], s5[..., 3] | (s5[..., 4] << 5)], axis=-1)


class Traces(object):
    """<variant>_traces.npz: the arrays e<e>_<key> of n_envs recorded envs, and the file-level arrays (z[key]).
    T: steps per env of a step trace (every env has the same number); None for the v5 / v6 event traces, whose envs
    have different lengths."""

    def __init__(self, golden_dir, variant):
        self.z = np.load(os.path.join(golden_dir, variant + "_traces.npz"))
        self.n_envs = int(self.z["n_envs"])
        self.T = len(self.z["e0_actions"]) if "e0_actions" in self.z.files else None

    def __getitem__(self, key):
        return self.z[key]

    def env(self, e):
        """{key: array} of env e."""
        pre = "e%d_" % e
        return {k[len(pre):]: self.z[k] for k in self.z.files if k.startswith(pre)}

    def per_env(self, key):
        """[n_envs, ...]: key of every env."""
        return np.stack([self.z["e%d_%s" % (e, key)] for e in range(self.n_envs)])

    def per_step(self, key):
        """[T, n_envs, ...]: key of every env at every step."""
        return np.stack([self.z["e%d_%s" % (e, key)] for e in range(self.n_envs)], axis=1)
