"""GPU tier: the single-maze compat classes replay the reference's golden traces in the reference's own
types (numpy obs, Python-float reward, bool done, info = the action passed)."""
import numpy as np
import pytest

from golden_io import Traces, unpack

pytestmark = pytest.mark.gpu


def test_lmaze_v0_drop_in(golden_dir):
    import gym_lmaze_b200 as g
    tr = Traces(golden_dir, "v0")
    env = g.make("lmaze-v0")
    assert isinstance(env, g.LmazeEnv) and env.action_space.n == 4 and tuple(env.observation_space.shape) == (4, 84, 84)
    for e in range(tr.n_envs):
        z = tr.env(e)
        obs = env.reset(spawn=tuple(z["spawn0"]))
        assert isinstance(obs, np.ndarray) and obs.dtype == np.float32 and obs.shape == (4, 84, 84)
        for t in range(tr.T):
            a = int(z["actions"][t])
            obs, r, d, info = env.step(a)
            assert type(r) is float and np.float64(r).view(np.int64) == z["reward_bits"][t], (e, t)
            assert type(d) is bool and d == bool(z["done"][t]) and info == a
            if d:
                obs = env.reset(spawn=tuple(z["spawn"][t]))
            assert np.array_equal(obs, unpack(z["obs"][t], (4, 84, 84))), (e, t)
    # float / numeric-string actions go through int() like the reference (lmaze_env.py:148)
    env.reset(spawn=(3, 3))
    assert env.step(1.9)[3] == 1 and env.step("3")[3] == 3
    env.close()


def test_lmaze_v3_drop_in_takes_strings(golden_dir):
    import gym_lmaze_b200 as g
    tr = Traces(golden_dir, "v3")
    env = g.make("lmaze-v3")
    spell = {0: ("left", "0"), 1: ("right", "1"), 2: ("up", "2"), 3: ("down", "3")}
    for e in range(2):
        z = tr.env(e)
        env.reset(spawn=tuple(z["spawn0"]))
        for t in range(tr.T):
            code = int(z["actions"][t])
            a = spell[code][t % 2] if code in spell else ("noop", 0, 3, "4")[t % 4]
            obs, r, d, info = env.step(a)
            assert np.float64(r).view(np.int64) == z["reward_bits"][t] and d == bool(z["done"][t])
            assert info == a
            if d:
                obs = env.reset(spawn=tuple(z["spawn"][t]))
            assert np.array_equal(obs, unpack(z["obs"][t], (3, 72, 72))), (e, t)
    o = env.reset(mode="test")
    assert env.state_vector[:4] == [7, 8, 8, 8] and o.shape == (3, 72, 72)
    env.close()


def test_lmaze_v2_v4_drop_in(golden_dir):
    import gym_lmaze_b200 as g
    tr = Traces(golden_dir, "v2")
    z = tr.env(0)
    env = g.make("lmaze-v2")
    assert env.action_space.n == 25 and tuple(env.observation_space.shape) == (5, 35, 35)
    init = z["init"]                                     # bx, by, gx, gy, layout, layout-before
    env._vec.set_state([[4, 4, 8, 8, 0, int(init[5]), 4 | (4 << 5), 0]])
    obs = env.reset(spawn=tuple(init[:5]))
    assert np.array_equal(obs, unpack(z["first_obs"], (5, 35, 35)))
    for t in range(tr.T):
        a = int(z["actions"][t])
        obs, r, d, info = env.step(a)
        assert np.float64(r).view(np.int64) == z["reward_bits"][t] and d == bool(z["done"][t]) and info == a
        if d:
            obs = env.reset(spawn=tuple(z["spawn"][t]))
        assert np.array_equal(obs, unpack(z["obs"][t], (5, 35, 35))), t
    with pytest.raises(IndexError):
        env.step(25)
    env.close()
    env4 = g.make("lmaze-v4")
    assert tuple(env4.observation_space.shape) == (7, 35, 35) and env4.step(12)[0].shape == (7, 35, 35)
    env4.close()
    vec = g.make("lmaze-vec-v0")
    assert isinstance(vec, g.LmazeVecCuda) and vec.num_envs == 4096
    vec.close()
