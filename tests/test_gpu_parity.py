"""GPU tier: the CUDA path (through the C ABI, via gym_lmaze_b200.LmazeVecCuda) against
(a) the golden fixtures produced by the unmodified reference and (b) the CPU oracle
on the same seeded inputs.  Everything is compared bit for bit: positions, reward
bit patterns, done flags and whole observation tensors, per step.
"""
import os

import numpy as np
import pytest
import torch

from golden_io import Traces, fov_image, pack_v2_spawn, reward_f32_bits, unpack
from gpu_helpers import REWARD_BITS, REWARD_F32, lmz, need_free, u32
from philox_np import _rng_actions

pytestmark = pytest.mark.gpu

INVALID = 7
RC = {0x8000000000000000: 0, 0xBFF0000000000000: 1, 0xBF847AE147AE147B: 2, 0x4059000000000000: 3}


def rcode_of_f64_bits(bits):
    return RC[int(np.int64(bits).view(np.uint64))]


# ---------------------------------------------------------------- golden fixtures (reference outputs)
@pytest.mark.parametrize("render_mode", ["tma", "st128"])
def test_v0_golden_table(lmz, golden_dir, render_mode):
    z = np.load(os.path.join(golden_dir, "v0_table.npz"))
    tab = np.concatenate([z["table"], z["edge"]])
    n = len(tab)
    env = lmz.LmazeVecCuda(n, "v0", autoreset=False, render_mode=render_mode)
    st = np.zeros((n, 8), np.int32)
    st[:, 0], st[:, 1], st[:, 2], st[:, 3] = tab[:, 0], tab[:, 1], 5, 5
    st[:, 4] = tab[:, 4]
    st[:, 5] = [rcode_of_f64_bits(b) for b in tab[:, 3]]
    st[:, 6] = 3
    env.set_state(st)
    obs, rew, done, info = env.step(torch.as_tensor(tab[:, 2]))
    out = env.get_state().cpu().numpy()
    assert np.array_equal(out[:, 0], tab[:, 5]) and np.array_equal(out[:, 1], tab[:, 6])
    assert np.array_equal(u32(rew), reward_f32_bits(tab[:, 7]))           # incl. -0.0 and the stale 'S' reward
    assert np.array_equal(done.cpu().numpy().astype(np.int64), tab[:, 8])
    assert np.array_equal(out[:, 6] - 3, tab[:, 9])        # goalCount delta
    assert np.array_equal(out[:, 4], tab[:, 10])           # stepCount
    assert torch.equal(info["action"].cpu(), torch.as_tensor(tab[:, 2]))
    # obs of each row = the reference render of its new position
    pos_index = {tuple(p): i for i, p in enumerate(z["positions"])}
    renders = torch.from_numpy(unpack(z["renders"], (4, 84, 84))).cuda()
    idx = torch.as_tensor([pos_index[(int(a), int(b))] for a, b in zip(tab[:, 5], tab[:, 6])]).cuda()
    assert torch.equal(obs, renders[idx])
    env.close()


def test_v3_golden_table(lmz, golden_dir):
    z = np.load(os.path.join(golden_dir, "v3_table.npz"))
    tab = np.concatenate([z["table"], z["edge"]])
    n = len(tab)
    env = lmz.LmazeVecCuda(n, "v3", autoreset=False)
    st = np.zeros((n, 8), np.int32)
    st[:, 0:4] = tab[:, 0:4]
    st[:, 4] = tab[:, 5]
    env.set_state(st)
    obs, rew, done, _ = env.step(torch.as_tensor(tab[:, 4]))
    out = env.get_state().cpu().numpy()
    assert np.array_equal(out[:, 0], tab[:, 6]) and np.array_equal(out[:, 1], tab[:, 7])
    assert np.array_equal(out[:, 2:4], tab[:, 2:4])
    assert np.array_equal(u32(rew), reward_f32_bits(tab[:, 8]))
    assert np.array_equal(done.cpu().numpy().astype(np.int64), tab[:, 9])
    assert np.array_equal(out[:, 4], tab[:, 10])
    # renders: set each (ball, goal) key and render without stepping
    keys = z["render_keys"]
    env2 = lmz.LmazeVecCuda(len(keys), "v3", autoreset=False)
    st2 = np.zeros((len(keys), 8), np.int32)
    st2[:, 0:4] = keys
    env2.set_state(st2)
    got = env2.render_obs()
    want = torch.from_numpy(unpack(z["renders"], (3, 72, 72))).cuda()
    assert torch.equal(got, want)
    env.close(); env2.close()


@pytest.mark.parametrize("variant", ["v0", "v3"])
@pytest.mark.parametrize("render_mode", ["tma", "st128"])
def test_golden_traces(lmz, golden_dir, variant, render_mode):
    """Recorded reference episodes (scripted spawns, invalid actions, timeouts, goals)."""
    tr = Traces(golden_dir, variant)
    shape = (4, 84, 84) if variant == "v0" else (3, 72, 72)
    env = lmz.LmazeVecCuda(tr.n_envs, variant, autoreset=True, render_mode=render_mode)
    sp0 = tr.per_env("spawn0")
    if variant == "v0":
        sp0 = np.concatenate([sp0, -np.ones_like(sp0)], 1)
    env.reset(spawn=sp0)
    acts, spawns, dref = tr.per_step("actions"), tr.per_step("spawn"), tr.per_step("done")
    want_r, obs_bits = reward_f32_bits(tr.per_step("reward_bits")), tr.per_step("obs")
    for t in range(tr.T):
        spawn = spawns[t]
        if variant == "v0":
            spawn = np.concatenate([spawn, -np.ones_like(spawn)], 1)
        spawn = np.where(dref[t][:, None] > 0, spawn, 1)
        obs, rew, done, _ = env.step(torch.as_tensor(acts[t]), spawn=spawn)
        assert np.array_equal(u32(rew), want_r[t]), t
        assert np.array_equal(done.cpu().numpy().astype(np.uint8), dref[t]), t
        assert np.array_equal(obs.cpu().numpy(), unpack(obs_bits[t], shape)), t
    s = env.stats()
    assert s["episodes"] == int(dref.sum()) and s["steps"] == tr.T * tr.n_envs
    env.close()


def test_v0_real_mt_trace(lmz, golden_dir):
    z = np.load(os.path.join(golden_dir, "v0_traces.npz"))
    env = lmz.LmazeVecCuda(1, "v0", autoreset=True)
    env.reset(spawn=[[z["mt_spawn0"][0], z["mt_spawn0"][1]]])
    for t in range(len(z["mt_actions"])):
        sp = z["mt_spawn"][t] if z["mt_done"][t] else (1, 1)
        obs, rew, done, _ = env.step(torch.as_tensor([z["mt_actions"][t]]), spawn=[[sp[0], sp[1]]])
        assert u32(rew)[0] == reward_f32_bits(z["mt_reward_bits"][t]) and bool(done[0]) == bool(z["mt_done"][t]), t
        if not z["mt_done"][t]:
            assert tuple(env.get_state()[0, :2].tolist()) == tuple(z["mt_pos"][t])
    env.close()


# ---------------------------------------------------------------- BASELINE config 2: 4,096 envs vs the oracle
def _spawn_cells(rows, variant):
    G = len(rows)
    if variant == "v0":
        return np.array([(x, y) for x in range(G) for y in range(G) if rows[x][y] in "BS"])
    return np.array([(x, y) for x in range(G) for y in range(G) if rows[x][y] != "W"])


def _random_spawn(rng, cells, n, variant):
    if variant == "v0":
        b = cells[rng.randint(len(cells), size=n)]
        return np.concatenate([b, -np.ones_like(b)], 1).astype(np.int32)
    gi = rng.randint(len(cells), size=n)
    bi = rng.randint(len(cells) - 1, size=n)
    bi = bi + (bi >= gi)
    return np.concatenate([cells[bi], cells[gi]], 1).astype(np.int32)


@pytest.mark.parametrize("variant,render_mode,T", [("v0", "tma", 256), ("v0", "st128", 64),
                                                   ("v3", "tma", 160), ("v3", "st128", 64)])
def test_config2_4096_envs_per_step_parity(lmz, oracle_mod, variant, render_mode, T):
    N = 4096
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    threads = os.cpu_count() or 1
    ora = oracle_mod.OracleVec(ov, N, autoreset=True, threads=threads)
    env = lmz.LmazeVecCuda(N, variant, autoreset=True, render_mode=render_mode)
    cells = _spawn_cells(oracle_mod.layout(ov), variant)
    rng = np.random.RandomState(1234)
    gen = torch.Generator().manual_seed(1234)
    sp = _random_spawn(rng, cells, N, variant)
    if variant == "v0":
        sp[:64, :2] = (1, 2)              # a block of envs next to the 'S' cell (stale-reward quirk)
    o_ref = ora.reset(spawn=sp)
    o_gpu = env.reset(spawn=sp)
    assert torch.equal(o_gpu.cpu(), torch.from_numpy(o_ref))
    actions = torch.randint(0, 4, (T, N), generator=gen)
    actions[torch.rand((T, N), generator=gen) < 0.03] = INVALID
    if variant == "v0":
        actions[0, :64] = 2               # (1,2) --left--> 'S': no branch taken
        actions[1, :32] = INVALID
    obs_buf = np.empty((N,) + oracle_mod.OBS_SHAPE[ov], np.float32)
    pinned = torch.from_numpy(obs_buf)
    for t in range(T):
        sp = _random_spawn(rng, cells, N, variant)
        a = actions[t]
        _, r_ref, d_ref = ora.step(a.numpy(), spawn=sp, obs_out=obs_buf)
        obs, rew, done, _ = env.step(a.to(torch.uint8) if t % 3 == 0 else (a.to(torch.int32) if t % 3 == 1 else a),
                                     spawn=sp)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)), t
        assert np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
        assert torch.equal(obs, pinned.cuda()), t
        if t % 16 == 0 or t == T - 1:
            st = env.get_state().cpu().numpy()
            pos, sc, gc, rw = ora.export()
            assert np.array_equal(st[:, 0:4], pos) if variant == "v3" else np.array_equal(st[:, 0:2], pos[:, 0:2])
            assert np.array_equal(st[:, 4], sc) and np.array_equal(st[:, 7], ora.episode)
            if variant == "v0":
                assert np.array_equal(st[:, 6], gc)
    s = env.stats()
    assert [s[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist()
    assert s["episodes"] >= N * (T // 101)          # every env timed out (or scored) at least T//101 times
    env.close()


# ---------------------------------------------------------------- device RNG, rollout, sharding
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_device_rng_spawn_matches_spec(lmz, oracle_mod, variant):
    N, T, seed, id0 = 2048, 230, 77, 1 << 33
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=seed, env_id0=id0, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0, autoreset=True)
    assert torch.equal(env.reset().cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(5)
    for t in range(T):
        a = torch.randint(0, 4, (N,), generator=gen)
        _, r_ref, d_ref = ora.step(a.numpy(), want_obs=False)
        _, rew, done, _ = env.step(a, )
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
    st = env.get_state().cpu().numpy()
    pos, sc, gc, _ = ora.export()
    assert np.array_equal(st[:, 0:2], pos[:, 0:2]) and np.array_equal(st[:, 4], sc)
    if variant == "v3":
        assert np.array_equal(st[:, 2:4], pos[:, 2:4])
    assert np.array_equal(st[:, 7], ora.episode) and ora.episode.min() >= 3
    assert torch.equal(env.render_obs().cpu(), torch.from_numpy(np.stack([ora.render_one(i) for i in range(N)])))
    env.close()


@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_rollout_kernel_parity(lmz, oracle_mod, variant):
    N, T, seed, id0 = 1500, 64, 11, 12345
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=seed, env_id0=id0, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0, autoreset=True)
    ora.reset(want_obs=False); env.reset()
    # (a) device-side Philox actions, two consecutive rollouts of uneven length (t0 continuity)
    t_global = 0
    for Tk in (64, 37, 64):
        rew, done = env.rollout(Tk)
        acts = np.array([[oracle_mod.rng_action(seed, id0 + i, t_global + t) for i in range(N)] for t in range(Tk)])
        for t in range(Tk):
            _, r_ref, d_ref = ora.step(acts[t], want_obs=False)
            assert np.array_equal(u32(rew[t]), r_ref.view(np.uint32)), (Tk, t)
            assert np.array_equal(done[t].cpu().numpy().view(np.uint8), d_ref), (Tk, t)
        t_global += Tk
    # (b) caller-supplied action buffer [T, N]
    gen = torch.Generator().manual_seed(3)
    a = torch.randint(0, 5, (T, N), generator=gen)        # 4 = invalid
    rew, done = env.rollout(T, actions=a.to(torch.uint8))
    for t in range(T):
        _, r_ref, d_ref = ora.step(a[t].numpy(), want_obs=False)
        assert np.array_equal(u32(rew[t]), r_ref.view(np.uint32)) and \
            np.array_equal(done[t].cpu().numpy().view(np.uint8), d_ref), t
    st = env.get_state().cpu().numpy()
    pos, sc, gc, _ = ora.export()
    assert np.array_equal(st[:, 0:2], pos[:, 0:2]) and np.array_equal(st[:, 4], sc) and np.array_equal(st[:, 7], ora.episode)
    s = env.stats()
    assert [s[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist()
    # final obs after a rollout comes from render_obs()
    assert torch.equal(env.render_obs().cpu(), torch.from_numpy(np.stack([ora.render_one(i) for i in range(N)])))
    env.close()


def test_shard_invariance(lmz):
    """Env i's trajectory does not depend on how the batch is split over handles/GPUs."""
    N, T, seed = 3000, 150, 9
    whole = lmz.LmazeVecCuda(N, "v0", seed=seed, env_id0=0)
    lo, hi = lmz.shard_range(N, 1, 3)
    part = lmz.LmazeVecCuda(hi - lo, "v0", seed=seed, env_id0=lo)
    assert torch.equal(whole.reset()[lo:hi], part.reset())
    r_w, d_w = whole.rollout(T)
    r_p, d_p = part.rollout(T)
    assert torch.equal(r_w[:, lo:hi].view(torch.int32), r_p.view(torch.int32)) and torch.equal(d_w[:, lo:hi], d_p)
    assert torch.equal(whole.get_state()[lo:hi], part.get_state())
    whole.close(); part.close()


# ---------------------------------------------------------------- reference behaviours with autoreset off
def test_no_autoreset_matches_reference_semantics(lmz, oracle_mod):
    N = 256
    ora = oracle_mod.OracleVec(oracle_mod.V0, N, autoreset=False)
    env = lmz.LmazeVecCuda(N, "v0", autoreset=False)
    cells = _spawn_cells(oracle_mod.layout(oracle_mod.V0), "v0")
    rng = np.random.RandomState(0)
    sp = _random_spawn(rng, cells, N, "v0")
    ora.reset(spawn=sp, want_obs=False); env.reset(spawn=sp)
    gen = torch.Generator().manual_seed(0)
    seen_101 = False
    for t in range(130):                     # stepping past done is legal: done at 100, not at 101 (Q4)
        a = torch.randint(0, 4, (N,), generator=gen)
        o_ref, r_ref, d_ref = ora.step(a.numpy())
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and np.array_equal(done.cpu().numpy().view(np.uint8), d_ref)
        assert torch.equal(obs.cpu(), torch.from_numpy(o_ref))
        if t == 100:
            seen_101 = True
            goal = u32(rew) == 0x42C80000
            assert not done.cpu().numpy()[~goal].any()
    assert seen_101
    # masked reset only touches the selected envs (state and obs)
    mask = torch.zeros(N, dtype=torch.bool); mask[::3] = True
    before = env.get_state().clone(); obs_before = env.obs.clone()
    sp = _random_spawn(rng, cells, N, "v0")
    env.reset(spawn=sp, mask=mask)
    after = env.get_state()
    assert torch.equal(after[~mask.cuda()], before[~mask.cuda()]) and torch.equal(env.obs[~mask.cuda()], obs_before[~mask.cuda()])
    assert (after[mask.cuda(), 4] == 0).all() and torch.equal(after[mask.cuda(), 0:2].cpu(), torch.from_numpy(sp[mask.numpy(), 0:2]))
    assert torch.equal(after[:, 6], before[:, 6])            # goalCount survives reset (Q5)
    env.close()


# ---------------------------------------------------------------- boundary behaviour
def test_abi_argument_validation(lmz):
    from gym_lmaze_b200._abi import LmzError
    env = lmz.LmazeVecCuda(64, "v0")
    env.reset()
    with pytest.raises(LmzError, match="shape"):
        env.step(torch.zeros(63, dtype=torch.int64, device="cuda"))
    with pytest.raises(LmzError, match="contiguous"):
        p, k = lmz.envs.lmaze_vec_cuda._abi.dl(torch.zeros(128, dtype=torch.int64, device="cuda")[::2])
        lmz.envs.lmaze_vec_cuda._abi.check(env._lib.lmz_step_dl(env._h, p, None, None))
    with pytest.raises(LmzError, match="CUDA device"):
        p, k = lmz.envs.lmaze_vec_cuda._abi.dl(torch.zeros(64, dtype=torch.int64))
        lmz.envs.lmaze_vec_cuda._abi.check(env._lib.lmz_step_dl(env._h, p, None, None))
    with pytest.raises(LmzError, match="dtype"):
        p, k = lmz.envs.lmaze_vec_cuda._abi.dl(torch.zeros(64, dtype=torch.float32, device="cuda"))
        lmz.envs.lmaze_vec_cuda._abi.check(env._lib.lmz_step_dl(env._h, p, None, None))
    # float / list / string actions are converted host-side like the reference's int(msg)
    env.step(torch.full((64,), 1.9, device="cuda"))
    env.step([0] * 64)
    # a spawn on a wall is rejected and reported
    env2 = lmz.LmazeVecCuda(4, "v0")
    env2.reset(spawn=[[0, 0], [5, 5], [1, 1], [2, 2]])
    with pytest.raises(ValueError, match="3 injected spawn"):
        env2.stats()
    env.close(); env2.close()
    with pytest.raises(KeyError):
        lmz.make("lmaze-v7")
    with pytest.raises(ValueError):
        lmz.LmazeVecCuda(4, "v5")


def test_raw_pointer_abi_and_host_step(lmz, oracle_mod):
    """The plain-pointer entry points and the HOST-buffer step (the end-to-end call)."""
    N = 1000
    env = lmz.LmazeVecCuda(N, "v0", seed=4)
    ora = oracle_mod.OracleVec(oracle_mod.V0, N, seed=4)
    env.reset(); ora.reset(want_obs=False)
    a = torch.randint(0, 4, (N,), dtype=torch.uint8).pin_memory()
    r = torch.empty(N, dtype=torch.float32).pin_memory()
    d = torch.empty(N, dtype=torch.uint8).pin_memory()
    o = torch.empty((N, 4, 84, 84), dtype=torch.float32).pin_memory()
    for _ in range(3):
        a.random_(0, 4)
        env.step_host(a, r, d, o)
        o_ref, r_ref, d_ref = ora.step(a.numpy().astype(np.int64))
        assert np.array_equal(r.numpy().view(np.uint32), r_ref.view(np.uint32)) and np.array_equal(d.numpy(), d_ref)
        assert np.array_equal(o.numpy(), o_ref)
    env.close()


def test_v3_string_actions(lmz, oracle_mod):
    env = lmz.LmazeVecCuda(4, "v3", autoreset=False)
    ora = oracle_mod.OracleVec(oracle_mod.V3, 4, autoreset=False)
    sp = [[7, 8, 8, 8]] * 4
    env.reset(spawn=sp); ora.reset(spawn=sp)
    obs, rew, done, _ = env.step(["left", "1", "up", "noop"])
    o_ref, r_ref, d_ref = ora.step(np.array([0, 1, 2, INVALID]))
    assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and torch.equal(obs.cpu(), torch.from_numpy(o_ref))
    env.close()


# ---------------------------------------------------------------- BASELINE config 3 scale: 2^20 envs, size-independent properties
def test_one_million_envs_properties(lmz, oracle_mod):
    N = 1 << 20
    need_free(N * 112896 + (4 << 30))
    env = lmz.LmazeVecCuda(N, "v0", seed=2026)
    obs = env.reset()
    gen = torch.Generator(device="cuda").manual_seed(1)
    for t in range(3):
        before = env.get_state()
        a = torch.randint(0, 4, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        obs, rew, done, _ = env.step(a)
    after = env.get_state()
    # every reward is one of the reference's four bit patterns
    rb = rew.view(torch.int32)
    allowed = torch.as_tensor(REWARD_BITS.view(np.int32)).cuda()
    assert torch.isin(rb, allowed).all()
    # per-env channel sums [49, 3528, 49, 3430] and ball block where the state says (chunked: obs is 118 GB)
    want = torch.tensor([49.0, 3528.0, 49.0, 3430.0], device="cuda")
    CH = 1 << 14
    for lo in range(0, N, CH):
        o = obs[lo:lo + CH]
        assert torch.equal(o.sum(dim=(2, 3)), want.expand(o.shape[0], 4))
        x = after[lo:lo + CH, 0].long(); y = after[lo:lo + CH, 1].long()
        idx = torch.arange(o.shape[0], device="cuda")
        assert (o[idx, 0, 7 * x, 7 * y] == 1).all() and (o[idx, 0, 7 * x + 6, 7 * y + 6] == 1).all()
        assert torch.equal(o[:, 1:], obs[0:1, 1:].expand(o.shape[0], 3, 84, 84))   # static channels identical
    # a random sample replayed through the oracle from the same pre-step state
    idx = torch.randperm(N, generator=torch.Generator().manual_seed(0))[:2048]
    b = before[idx.cuda()].cpu().numpy()
    ora = oracle_mod.OracleVec(oracle_mod.V0, len(idx), autoreset=False)
    for i, row in enumerate(b):
        ora.force(i, int(row[0]), int(row[1]), step_count=int(row[4]), reward=float(REWARD_F32[row[5]]), goal_count=int(row[6]))
    _, r_ref, d_ref = ora.step(a[idx.cuda()].cpu().numpy().astype(np.int64), want_obs=False)
    assert np.array_equal(u32(rew[idx.cuda()]), r_ref.view(np.uint32))
    assert np.array_equal(done[idx.cuda()].cpu().numpy().view(np.uint8), d_ref)
    nd = d_ref == 0                                 # envs that did not reset: position must match, obs must match
    pos = ora.export()[0]
    assert np.array_equal(after[idx.cuda()].cpu().numpy()[nd, 0:2], pos[nd, 0:2])
    sel = idx[torch.from_numpy(nd)][:256]
    ref_obs = np.stack([ora.render_one(int(i)) for i in np.nonzero(nd)[0][:256]])
    assert torch.equal(obs[sel.cuda()].cpu(), torch.from_numpy(ref_obs))
    s = env.stats()
    assert s["steps"] == 3 * N and s["wall_bumps"] + s["moves"] + s["stale"] == 3 * N
    env.close()


# ---------------------------------------------------------------- compact observations and render windows
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_compact_obs_reconstructs_reference_image(lmz, oracle_mod, variant):
    """obs_mode='compact' (u8 un-expanded layers): expand() must equal the oracle's full image, per step."""
    N, T = 1000, 130
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=21, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=21, autoreset=True, obs_mode="compact")
    assert env.obs.dtype == torch.uint8 and tuple(env.obs.shape[1:]) == ((4, 12, 12) if variant == "v0" else (3, 18, 18))
    assert torch.equal(env.expand(env.reset()).cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(8)
    for t in range(T):
        a = torch.randint(0, 5, (N,), generator=gen)
        o_ref, r_ref, d_ref = ora.step(a.numpy())
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and np.array_equal(done.cpu().numpy().view(np.uint8), d_ref)
        assert torch.equal(env.expand(obs).cpu(), torch.from_numpy(o_ref)), t
    s = env.stats()
    assert [s[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist()
    if variant == "v0":
        # reference initState(): raw un-expanded state layers (lmaze_env.py:243-244)
        state, rew, done, info = env.initState()
        assert info == {"newState": True} and state.shape == (N, 576)
        full = torch.from_numpy(np.stack([ora.render_one(i) for i in range(N)]))
        assert torch.equal(state.view(N, 4, 12, 12).cpu(), full[:, :, ::7, ::7])
    env.close()


@pytest.mark.parametrize("render_mode,obs_mode", [("tma", "full"), ("st128", "full"), ("tma", "compact")])
def test_render_window(lmz, oracle_mod, render_mode, obs_mode):
    """A window of W rows stands for envs [lo, lo+W): every env steps, only the window is rendered."""
    N, W = 1000, 300
    ora = oracle_mod.OracleVec(oracle_mod.V3, N, seed=5, autoreset=True)
    env = lmz.LmazeVecCuda(N, "v3", seed=5, autoreset=True, render_mode=render_mode, obs_mode=obs_mode, obs_window=W)
    assert env.obs.shape[0] == W
    ora.reset(want_obs=False); env.reset()
    gen = torch.Generator().manual_seed(2)
    for t in range(6):
        a = torch.randint(0, 4, (N,), generator=gen)
        o_ref, r_ref, d_ref = ora.step(a.numpy())
        lo = (t * 173) % (N - W + 1)
        env.set_window(lo)
        env.obs.fill_(7)                                   # sentinel: rows must be fully rewritten
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32))          # all N envs stepped
        assert torch.equal(env.expand(obs).cpu(), torch.from_numpy(o_ref[lo:lo + W])), t
        # walk the rest of the batch window by window without stepping
        for lo2 in (0, N - W, 350):
            assert torch.equal(env.expand(env.render_window(lo2)).cpu(), torch.from_numpy(o_ref[lo2:lo2 + W]))
    from gym_lmaze_b200._abi import LmzError
    with pytest.raises(LmzError, match="window"):
        env.set_window(N - W + 1)
    env.close()


def test_transition_only_mode(lmz, oracle_mod):
    """with_obs=False: nothing is rendered, transitions/stat counters are unchanged."""
    N = 2000
    ora = oracle_mod.OracleVec(oracle_mod.V0, N, seed=9)
    env = lmz.LmazeVecCuda(N, "v0", seed=9, with_obs=False)
    ora.reset(want_obs=False); assert env.reset() is None
    gen = torch.Generator().manual_seed(4)
    for t in range(120):
        a = torch.randint(0, 4, (N,), generator=gen)
        _, r_ref, d_ref = ora.step(a.numpy(), want_obs=False)
        obs, rew, done, _ = env.step(a)
        assert obs is None and np.array_equal(u32(rew), r_ref.view(np.uint32)) and \
            np.array_equal(done.cpu().numpy().view(np.uint8), d_ref)
    assert [env.stats()[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist()
    env.close()


# ---------------------------------------------------------------- lmaze-v2 (multi-layout foveal env)
def _v2_state_rows(L, bx, by, gx, gy, px, py, step, a=None):
    aux = px | (py << 5) | ((a << 10) | (1 << 15) if a is not None else 0)
    return [bx, by, gx, gy, step, L, aux, 0]


def test_v2_golden_table(lmz, golden_dir):
    z = np.load(os.path.join(golden_dir, "v2_table.npz"))
    tab = z["table"]
    n = len(tab)
    env = lmz.LmazeVecCuda(n, "v2", autoreset=False)
    assert env.num_actions == 25 and env.obs.shape[1:] == (5, 35, 35) and env.num_layouts == 5
    st = np.array([_v2_state_rows(r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[8]) for r in tab], np.int32)
    env.set_state(st)
    obs, rew, done, info = env.step(torch.as_tensor(tab[:, 7]))
    out = env.get_state().cpu().numpy()
    assert np.array_equal(out[:, 0], tab[:, 9]) and np.array_equal(out[:, 1], tab[:, 10])
    assert np.array_equal(u32(rew), reward_f32_bits(tab[:, 11]))
    assert np.array_equal(done.cpu().numpy().astype(np.int64), tab[:, 12])
    assert np.array_equal(out[:, 4], tab[:, 13])
    want = torch.from_numpy(unpack(z["obs"], (5, 35, 35)))
    # the device state has no room for an UNREACHABLE history (previous crop taken somewhere other than
    # the ball's cell), which half of the fixture rows use on purpose: compare their channels 0-2 only
    reachable = torch.from_numpy((tab[:, 1] == tab[:, 5]) & (tab[:, 2] == tab[:, 6]))
    assert reachable.sum() > 2000
    got = obs.cpu()
    assert torch.equal(got[reachable], want[reachable])
    assert torch.equal(got[~reachable][:, :3], want[~reachable][:, :3])
    # layouts exported by the library == the reference's five mazes
    zl = np.load(os.path.join(golden_dir, "v2_layouts.npz"))["layouts"]
    for k in range(5):
        assert env.layout(k + 1) == [str(r) for r in zl[k]]
    env.close()


def test_v2_golden_traces(lmz, golden_dir):
    tr = Traces(golden_dir, "v2")
    env = lmz.LmazeVecCuda(tr.n_envs, "v2", autoreset=True)
    init = tr.per_env("init")                                      # bx, by, gx, gy, layout, layout-before
    st = np.array([_v2_state_rows(r[5], 4, 4, 8, 8, 4, 4, 0) for r in init], np.int32)
    env.set_state(st)                                              # the maze the constructor rolled
    obs = env.reset(spawn=init[:, :5])
    assert np.array_equal(obs.cpu().numpy(), unpack(tr.per_env("first_obs"), (5, 35, 35)))
    acts, s5, dref = tr.per_step("actions"), tr.per_step("spawn"), tr.per_step("done")
    want_r, obs_bits = reward_f32_bits(tr.per_step("reward_bits")), tr.per_step("obs")
    for t in range(tr.T):
        obs, rew, done, _ = env.step(torch.as_tensor(acts[t]), spawn=np.where(dref[t][:, None] > 0, s5[t], 0))
        assert np.array_equal(u32(rew), want_r[t]), t
        assert np.array_equal(done.cpu().numpy().astype(np.uint8), dref[t]), t
        assert np.array_equal(obs.cpu().numpy(), unpack(obs_bits[t], (5, 35, 35))), t
    assert env.stats()["episodes"] == int(dref.sum())
    env.close()


@pytest.mark.parametrize("inject", [True, False])
def test_v2_4096_envs_vs_oracle(lmz, oracle_mod, inject):
    """Config-2-style parity for v2: per step reward bits, done, whole obs; injected or device-RNG resets."""
    N, T, seed = (512, 70, 31) if inject else (4096, 130, 31)
    ora = oracle_mod.OracleVec(oracle_mod.V2, N, seed=seed, env_id0=77, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, "v2", seed=seed, env_id0=77, autoreset=True)
    rng = np.random.RandomState(3)
    cands = []
    for k in range(1, 6):
        rows = oracle_mod.layout_v2(k)
        gc = [(x, y) for x in range(1, 17) for y in range(1, 17) if rows[x][y] not in "WS"]
        bc = [(x, y) for x in range(1, 17) for y in range(1, 17) if rows[x][y] not in "WX"]
        cands.append((gc, bc))

    def draw_spawn(cur_layouts):
        """what the reference's rejection loops could have produced on each env's CURRENT maze"""
        out = np.zeros((N, 5), np.int64)
        for i in range(N):
            gc, bc = cands[cur_layouts[i] - 1]
            g = gc[rng.randint(len(gc))]
            b = g
            while b == g:
                b = bc[rng.randint(len(bc))]
            out[i] = (b[0], b[1], g[0], g[1], rng.randint(1, 6))
        return out

    if inject:
        s5 = draw_spawn(np.ones(N, int))
        o_ref = ora.reset(spawn=pack_v2_spawn(s5)); o_gpu = env.reset(spawn=s5)
    else:
        o_ref = ora.reset(); o_gpu = env.reset()
    assert torch.equal(o_gpu.cpu(), torch.from_numpy(o_ref))
    gen = torch.Generator().manual_seed(9)
    obs_buf = np.empty((N, 5, 35, 35), np.float32)
    for t in range(T):
        a = torch.randint(0, 25, (N,), generator=gen)
        if inject:
            s5 = draw_spawn(ora.export_aux()[:, 0])
            _, r_ref, d_ref = ora.step(a.numpy(), spawn=pack_v2_spawn(s5), obs_out=obs_buf)
            obs, rew, done, _ = env.step(a, spawn=s5)
        else:
            _, r_ref, d_ref = ora.step(a.numpy(), obs_out=obs_buf)
            obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)), t
        assert np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
        assert torch.equal(obs.cpu(), torch.from_numpy(obs_buf)), t
    st = env.get_state().cpu().numpy()
    pos, sc, _, _ = ora.export()
    aux = ora.export_aux()
    assert np.array_equal(st[:, 0:4], pos) and np.array_equal(st[:, 4], sc) and np.array_equal(st[:, 5], aux[:, 0])
    assert np.array_equal(st[:, 7], ora.episode)
    s = env.stats()
    assert [s[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist()
    assert s["episodes"] >= N and s["goals"] > 0
    if not inject:
        assert torch.equal(env.render_obs().cpu(), torch.from_numpy(np.stack([ora.render_one(i) for i in range(N)])))
    env.close()


def test_v2_windows_and_masks(lmz, oracle_mod):
    """Partial tiles: batch tail (N % 32 != 0), render window edges, masked reset."""
    N, W = 1003, 333
    ora = oracle_mod.OracleVec(oracle_mod.V2, N, seed=2, autoreset=True)
    env = lmz.LmazeVecCuda(N, "v2", seed=2, autoreset=True, obs_window=W)
    ora.reset(want_obs=False); env.reset()
    gen = torch.Generator().manual_seed(1)
    for t in range(5):
        a = torch.randint(0, 25, (N,), generator=gen)
        o_ref, r_ref, d_ref = ora.step(a.numpy())
        lo = (t * 211) % (N - W + 1)
        env.set_window(lo)
        env.obs.fill_(5)
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32))
        assert torch.equal(obs.cpu(), torch.from_numpy(o_ref[lo:lo + W])), t
        assert torch.equal(env.render_window(N - W).cpu(), torch.from_numpy(o_ref[N - W:]))
    rew, done = env.rollout(4)                      # (round 2: the foveal variants have a rollout kernel too)
    assert tuple(rew.shape) == (4, N) and tuple(done.shape) == (4, N)
    env.close()
    # out-of-range actions are clamped and reported
    env = lmz.LmazeVecCuda(8, "v2", seed=1)
    env.reset()
    env.step(torch.tensor([0, 24, 25, -1, 7, 300, 12, 3]))
    with pytest.raises(ValueError, match="3 "):
        env.stats()
    env.close()


# ---------------------------------------------------------------- lmaze-v4 (v2 + float visit layer)
def test_v4_golden_table(lmz, golden_dir):
    """Reference outputs incl. the float visit layer, compared as f32 BIT patterns."""
    z = np.load(os.path.join(golden_dir, "v4_table.npz"))
    tab = z["table"]
    n = len(tab)
    env = lmz.LmazeVecCuda(n, "v4", autoreset=False)
    assert env.obs.shape[1:] == (7, 35, 35) and env.num_actions == 25
    st = np.array([_v2_state_rows(r[0], r[1], r[2], r[3], r[4], r[1], r[2], r[6]) for r in tab], np.int32)
    env.set_state(st)
    env.set_visit(z["pre_visit"])
    obs, rew, done, _ = env.step(torch.as_tensor(tab[:, 5]))
    out = env.get_state().cpu().numpy()
    assert np.array_equal(out[:, 0], tab[:, 7]) and np.array_equal(out[:, 1], tab[:, 8])
    assert np.array_equal(u32(rew), reward_f32_bits(tab[:, 9]))
    assert np.array_equal(done.cpu().numpy().astype(np.int64), tab[:, 10]) and np.array_equal(out[:, 4], tab[:, 11])
    assert np.array_equal(env.get_visit().cpu().numpy().view(np.uint32), z["post_visit"].view(np.uint32))
    want = fov_image(z["obs_bits"], z["obs_visit"])
    assert np.array_equal(obs.cpu().numpy().view(np.uint32), want.view(np.uint32))
    env.close()


def test_v4_golden_traces(lmz, golden_dir):
    tr = Traces(golden_dir, "v4")
    env = lmz.LmazeVecCuda(tr.n_envs, "v4", autoreset=True)
    obs = env.reset(spawn=tr.per_env("init"))                      # bx, by, gx, gy, layout
    assert np.array_equal(obs.cpu().numpy(), fov_image(tr.per_env("first_bits"), tr.per_env("first_visit")))
    acts, s5, dref = tr.per_step("actions"), tr.per_step("spawn"), tr.per_step("done")
    want_r = reward_f32_bits(tr.per_step("reward_bits"))
    obs_bits, obs_visit = tr.per_step("obs_bits"), tr.per_step("obs_visit")
    for t in range(tr.T):
        obs, rew, done, _ = env.step(torch.as_tensor(acts[t]), spawn=np.where(dref[t][:, None] > 0, s5[t], 0))
        assert np.array_equal(u32(rew), want_r[t]), t
        assert np.array_equal(done.cpu().numpy().astype(np.uint8), dref[t]), t
        assert np.array_equal(u32(obs), u32(fov_image(obs_bits[t], obs_visit[t]))), t
    assert np.array_equal(u32(env.get_visit()), u32(tr.per_env("final_visit")))
    env.close()


def test_v4_4096_envs_vs_oracle(lmz, oracle_mod):
    """Device-RNG resets, 130 steps, 4,099 envs (ragged last tile): reward bits, done, whole obs, visit layer."""
    N, T, seed = 4099, 130, 13
    ora = oracle_mod.OracleVec(oracle_mod.V4, N, seed=seed, env_id0=5, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, "v4", seed=seed, env_id0=5, autoreset=True)
    assert torch.equal(env.reset().cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(4)
    obs_buf = np.empty((N, 7, 35, 35), np.float32)
    for t in range(T):
        a = torch.randint(0, 25, (N,), generator=gen)
        _, r_ref, d_ref = ora.step(a.numpy(), obs_out=obs_buf)
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)), t
        assert np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
        assert torch.equal(obs.cpu().view(torch.int32), torch.from_numpy(obs_buf).view(torch.int32)), t
        if t % 25 == 0:
            assert np.array_equal(env.get_visit().cpu().numpy().view(np.uint32), ora.export_visit().view(np.uint32))
    st = env.get_state().cpu().numpy()
    pos, sc, _, _ = ora.export()
    assert np.array_equal(st[:, 0:4], pos) and np.array_equal(st[:, 4], sc) and np.array_equal(st[:, 7], ora.episode)
    s = env.stats()
    assert [s[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist() and s["episodes"] >= 2 * N
    # re-render and windowed render agree with the oracle as well
    full = torch.from_numpy(np.stack([ora.render_one(i) for i in range(N)]))
    assert torch.equal(env.render_obs().cpu(), full)
    env.close()


# ---------------------------------------------------------------- CUDA graph replay of the fused step
@pytest.mark.parametrize("variant,render_mode", [("v0", "tma"), ("v0", "st128"), ("v2", "tma")])
def test_cuda_graph_replay(lmz, oracle_mod, variant, render_mode):
    """One captured launch replayed 150 times (the work counter re-arms itself) == 150 oracle steps."""
    N = 4096
    ov = {"v0": oracle_mod.V0, "v2": oracle_mod.V2}[variant]
    ora = oracle_mod.OracleVec(ov, N, seed=6, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=6, autoreset=True, render_mode=render_mode)
    ora.reset(want_obs=False); env.reset()
    abuf = torch.zeros(N, dtype=torch.uint8, device="cuda")
    replay = env.capture_step(abuf)
    launches = env.launch_count
    gen = torch.Generator().manual_seed(12)
    for t in range(150):
        a = torch.randint(0, env.num_actions, (N,), generator=gen)
        abuf.copy_(a.to(torch.uint8))
        replay()
        o_ref, r_ref, d_ref = ora.step(a.numpy(), want_obs=(t % 30 == 0))
        assert np.array_equal(u32(env.reward), r_ref.view(np.uint32)), t
        assert np.array_equal(env.done.cpu().numpy().view(np.uint8), d_ref), t
        if t % 30 == 0:
            assert torch.equal(env.obs.cpu(), torch.from_numpy(o_ref)), t
    assert env.launch_count == launches          # no host-side launches happened during the replays
    assert env.stats()["steps"] == 150 * N       # capturing does not execute; the warm-up is a render, not a step
    env.close()


# ---------------------------------------------------------------- the reference's attribute switches
@pytest.mark.parametrize("variant,random_ball,random_goal", [("v0", False, True), ("v3", False, True),
                                                             ("v3", True, False), ("v3", False, False)])
def test_fixed_ball_and_goal_switches(lmz, oracle_mod, variant, random_ball, random_goal):
    """RANDOM_BALL / RANDOM_GOAL = False (lmaze_env.py:25,82-89; lmaze_env_v3.py:103-104,162-164)."""
    N = 600
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=3, random_ball=random_ball, random_goal=random_goal)
    env = lmz.LmazeVecCuda(N, variant, seed=3, random_ball=random_ball, random_goal=random_goal)
    assert torch.equal(env.reset().cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(1)
    for t in range(210):
        a = torch.randint(0, 4, (N,), generator=gen)
        o_ref, r_ref, d_ref = ora.step(a.numpy(), want_obs=(t % 20 == 0))
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
        if t % 20 == 0:
            assert torch.equal(obs.cpu(), torch.from_numpy(o_ref)), t
    st = env.get_state().cpu().numpy()
    pos = ora.export()[0]
    assert np.array_equal(st[:, 0:2], pos[:, 0:2])
    if variant == "v3":
        assert np.array_equal(st[:, 2:4], pos[:, 2:4])
        if not random_goal:
            assert (st[:, 2] == 8).all() and (st[:, 3] == 8).all()      # the 'X' cell
    env.close()


def test_v3_reset_test_mode(lmz, golden_dir):
    z = np.load(os.path.join(golden_dir, "v3_table.npz"))
    env = lmz.LmazeVecCuda(5, "v3")
    obs = env.reset(mode="test")
    st = env.get_state().cpu().numpy()
    assert (st[:, 0:4] == np.array(z["test_info"])).all()
    assert np.array_equal(obs[0].cpu().numpy(), unpack(z["test_obs"], (3, 72, 72)))
    env.close()
    with pytest.raises(ValueError):
        lmz.LmazeVecCuda(2, "v0").reset(mode="test")


# ---------------------------------------------------------------- incremental render into a persistent obs tensor
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_incremental_render_stays_bit_identical(lmz, oracle_mod, variant):
    """render_mode='incremental': only the moved ExE blocks are rewritten, yet after every step the whole
    obs tensor equals the oracle's full image (auto-resets, invalid actions, windows, set_state resync)."""
    N, T = 2500, 260
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=17, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=17, autoreset=True, render_mode="incremental")
    assert torch.equal(env.reset().cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(3)
    obs_buf = np.empty((N,) + oracle_mod.OBS_SHAPE[ov], np.float32)
    for t in range(T):
        a = torch.randint(0, 5, (N,), generator=gen)
        want_obs = t % 7 == 0 or t > T - 4
        _, r_ref, d_ref = ora.step(a.numpy(), obs_out=obs_buf if want_obs else None, want_obs=want_obs)
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
        if want_obs:
            assert torch.equal(obs.cpu(), torch.from_numpy(obs_buf)), t
        if t == 100:                              # move envs behind the tensor's back: must resync with a full render
            st = env.get_state()
            env.set_state(st.roll(1, 0))
            for i, row in enumerate(st.roll(1, 0).cpu().numpy()):
                ora.force(i, int(row[0]), int(row[1]), int(row[2]), int(row[3]), step_count=int(row[4]),
                          reward=float(REWARD_F32[row[5]]), goal_count=int(row[6]))
            ora.episode[:] = st.roll(1, 0).cpu().numpy()[:, 7]
        if t == 150:                              # masked reset in the middle (full render of the masked rows only)
            mask = torch.rand(N, generator=gen) < 0.3
            sp = _random_spawn(np.random.RandomState(t), _spawn_cells(oracle_mod.layout(ov), variant), N, variant)
            env.reset(spawn=sp, mask=mask)
            for i in np.nonzero(mask.numpy())[0]:
                oracle_mod.lib().lmzo_reset(ora._env(int(i)), int(sp[i, 0]), int(sp[i, 1]), int(sp[i, 2]), int(sp[i, 3]))
                ora.episode[i] += 1
    s = env.stats()
    assert s["steps"] == T * N and s["episodes"] == int(ora.stats[1])
    env.close()
    # windowed: the window is re-synced by a full render after every set_window
    env = lmz.LmazeVecCuda(N, variant, seed=17, render_mode="incremental", obs_window=700)
    ora = oracle_mod.OracleVec(ov, N, seed=17)
    env.reset(); ora.reset(want_obs=False)
    for t in range(12):
        a = torch.randint(0, 4, (N,), generator=gen)
        o_ref, _, _ = ora.step(a.numpy())
        if t % 4 == 0:
            env.set_window(300 * (t // 4))
        obs, _, _, _ = env.step(a)
        assert torch.equal(obs.cpu(), torch.from_numpy(o_ref[env.window_lo:env.window_lo + 700])), t
    env.close()


# ---------------------------------------------------------------- long soak: 65,536 envs x 1,000 steps
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_soak_rollout_65k_envs_1000_steps(lmz, oracle_mod, variant):
    """Device-RNG actions and spawns for 65.5 M env-steps: every reward / done of every step, the final
    states, goal counts, episode counters and the integer statistics must equal the oracle's."""
    N, T, calls, seed, id0 = 1 << 16, 250, 4, 2027, 10 ** 12
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=seed, env_id0=id0, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0, autoreset=True, with_obs=False)
    ora.reset(want_obs=False); env.reset()
    L = oracle_mod.lib()
    ids = np.arange(N, dtype=np.uint64) + np.uint64(id0)
    t_global = 0
    for c in range(calls):
        rew, done = env.rollout(T)
        rew_h = rew.cpu().numpy().view(np.uint32); done_h = done.cpu().numpy().view(np.uint8)
        for t in range(T):
            acts = np.fromiter((L.lmzo_rng_action(seed, int(g), t_global + t) for g in ids[:64]), dtype=np.int64)
            # the full action row comes from the vectorised twin below; the first 64 are cross-checked here
            row = _rng_actions(seed, ids, t_global + t)
            assert np.array_equal(row[:64], acts)
            _, r_ref, d_ref = ora.step(row, want_obs=False)
            assert np.array_equal(rew_h[t], r_ref.view(np.uint32)), (c, t)
            assert np.array_equal(done_h[t], d_ref), (c, t)
        t_global += T
    st = env.get_state().cpu().numpy()
    pos, sc, gc, _ = ora.export()
    assert np.array_equal(st[:, 0:2], pos[:, 0:2]) and np.array_equal(st[:, 4], sc) and np.array_equal(st[:, 7], ora.episode)
    if variant == "v0":
        assert np.array_equal(st[:, 6], gc)
    s = env.stats()
    assert [s[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist() and s["steps"] == N * T * calls
    env.close()

