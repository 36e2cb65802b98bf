"""CPU test: the numpy twins of the device action streams (tests/philox_np.py) equal the oracle's scalar functions.
The GPU tests drive whole-batch oracles with these twins, so a wrong twin would blame (or excuse) a kernel."""
import numpy as np
import pytest

from philox_np import ActionStream, _rng_actions, rng_actions25, rng_hier

SEEDS = [0, 7, 2027, (1 << 32) + 5, 0xDEADBEEF12345678, (1 << 64) - 1]
# env ids on both sides of 2^32 (the counter's low / high words) and near the top of the range
IDS = np.array([0, 1, 31, 32, 4095, 606_228, (1 << 32) - 2, (1 << 32) - 1, 1 << 32, (1 << 32) + 1, 1 << 33,
                10 ** 12 + 17, (1 << 63) + 3, (1 << 64) - 1], dtype=np.uint64)
# steps crossing the 4-step (Discrete(25)) and 64-step (Discrete(4)) block boundaries, and a block index past 2^32
TS = [0, 1, 2, 3, 4, 5, 15, 16, 17, 62, 63, 64, 65, 127, 128, 129, 1000, (1 << 32) + 3, (1 << 38) + 64 * 3 + 1]


@pytest.fixture(scope="module")
def O(oracle_mod):
    return oracle_mod


@pytest.mark.parametrize("seed", SEEDS)
def test_rng_action_twin(O, seed):
    for t in TS:
        want = [O.rng_action(seed, int(i), t) for i in IDS]
        assert _rng_actions(seed, IDS, t).tolist() == want, t


@pytest.mark.parametrize("seed", SEEDS)
def test_rng_action25_twin(O, seed):
    for t in TS:
        want = [O.rng_action25(seed, int(i), t) for i in IDS]
        assert rng_actions25(seed, IDS, t).tolist() == want, t


@pytest.mark.parametrize("seed", SEEDS)
def test_rng_hier_twin(O, seed):
    for t in TS:
        want = [O.rng_hier(seed, int(i), t) for i in IDS]
        g, a = rng_hier(seed, IDS, t)
        assert list(zip(g.tolist(), a.tolist())) == want, t


def test_twins_cover_their_value_ranges(O):
    """Over many envs every action / goal value occurs: the twins are not stuck on a constant word."""
    ids = np.arange(1 << 32, (1 << 32) + 4096, dtype=np.uint64)
    assert set(_rng_actions(9, ids, 70).tolist()) == set(range(4))
    assert set(rng_actions25(9, ids, 6).tolist()) == set(range(25))
    g, a = rng_hier(9, ids, 3)
    assert set(g.tolist()) == set(range(25)) and set(a.tolist()) == set(range(4))


@pytest.mark.parametrize("kind", [4, 25])
def test_action_stream_over_consecutive_steps(O, kind):
    """ActionStream reuses one block across the steps it covers: 140 consecutive steps (from t = 60, across block
    boundaries of both kinds) equal the scalar functions."""
    seed, ids = (3 << 32) + 9, IDS
    scalar = O.rng_action if kind == 4 else O.rng_action25
    stream = ActionStream(seed, ids, kind)
    for t in range(60, 200):
        assert stream(t).tolist() == [scalar(seed, int(i), t) for i in ids], t
