"""numpy twins of the oracle's counter-based action streams (oracle/lmaze_oracle.c lmzo_rng_action, lmzo_rng_action25,
lmzo_rng_hier): the same Philox-4x32-10 blocks computed for a whole array of env ids at once, so that tests can drive a
whole-batch oracle with the actions the rollout kernels draw on the device."""
import numpy as np

_M32 = np.uint64(0xFFFFFFFF)


def _philox_np(c0, c1, c2, c3, k0, k1):
    """numpy Philox-4x32-10 over arrays of counters (same spec as DESIGN.md section 4)."""
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) for x in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & _M32, p1 >> np.uint64(32), p1 & _M32
        c0, c1, c2, c3 = (hi1 ^ c1 ^ k0) & _M32, lo1, (hi0 ^ c3 ^ k1) & _M32, lo0
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
    return c0, c1, c2, c3


def _block(seed, ids, blk, tag):
    """Philox block `blk` of every env id in `ids` (uint64 array): counter (id lo, id hi, blk lo, blk hi << 8 | tag)."""
    ids = np.asarray(ids, dtype=np.uint64)
    n = len(ids)
    seed, blk = int(seed), int(blk)
    return _philox_np(ids & _M32, ids >> np.uint64(32), np.full(n, blk & 0xFFFFFFFF, np.uint64),
                      np.full(n, (((blk >> 32) << 8) | tag) & 0xFFFFFFFF, np.uint64),
                      seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)


class ActionStream(object):
    """Actions of env ids `ids` at consecutive steps t, one Philox block computed per block boundary crossed.
    kind 4: lmzo_rng_action (v0 / v3, 64 two-bit actions per block); kind 25: lmzo_rng_action25 (v2 / v4, word t % 4
    of block t // 4, scaled to 0..24)."""

    def __init__(self, seed, ids, kind):
        assert kind in (4, 25)
        self.seed, self.ids, self.kind = seed, np.asarray(ids, dtype=np.uint64), kind
        self._blk, self._w = None, None

    def __call__(self, t):
        blk = t >> 6 if self.kind == 4 else t >> 2
        if blk != self._blk:
            self._blk, self._w = blk, _block(self.seed, self.ids, blk, 0x41 if self.kind == 4 else 0x42)
        if self.kind == 4:
            slot = t & 63
            return ((self._w[slot >> 4] >> np.uint64(2 * (slot & 15))) & np.uint64(3)).astype(np.int64)
        return ((self._w[t & 3] * np.uint64(25)) >> np.uint64(32)).astype(np.int64)


def _rng_actions(seed, ids, t):
    """lmzo_rng_action at step t for every env id in `ids`."""
    return ActionStream(seed, ids, 4)(t)


def rng_actions25(seed, ids, t):
    """lmzo_rng_action25 at step t for every env id in `ids`."""
    return ActionStream(seed, ids, 25)(t)


def rng_hier(seed, ids, t):
    """lmzo_rng_hier (v5 / v6): one block per step; goal from word 0 scaled to 0..24, action = top 2 bits of word 1."""
    w = _block(seed, ids, t, 0x48)
    return ((w[0] * np.uint64(25)) >> np.uint64(32)).astype(np.int64), (w[1] >> np.uint64(30)).astype(np.int64)
