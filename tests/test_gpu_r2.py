"""GPU tier, round 2: regressions for the round-1 review (ADVICE.md / VERDICT.md) and the paths added in round 2.
Everything goes through the C ABI (gym_lmaze_b200.LmazeVecCuda / LmazeHierCuda) and is compared bit for bit with the
CPU oracle or with the golden fixtures produced by the unmodified reference."""
import os

import numpy as np
import pytest
import torch

from golden_io import unpack
from gpu_helpers import REWARD_BITS, lmz, u32
from philox_np import _rng_actions

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------- ADVICE r1 (high): incremental render + rollout
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_incremental_render_resyncs_after_rollout(lmz, oracle_mod, variant):
    """lmz_rollout moves every ball (and auto-resets) without rendering; the next step of an incremental-render
    env must fall back to a full render, or the tensor keeps the pre-rollout blocks (lmaze_env.py:208-234 is a
    full image every step)."""
    N, seed, T = 1500, 23, 37
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=seed, autoreset=True)
    env = lmz.LmazeVecCuda(N, variant, seed=seed, autoreset=True, render_mode="incremental")
    assert torch.equal(env.reset().cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(5)
    t_roll = 0
    for it in range(3):
        for _ in range(3):                                     # steps on the incremental kernel
            a = torch.randint(0, 5, (N,), generator=gen)
            o_ref, r_ref, d_ref = ora.step(a.numpy())
            obs, rew, done, _ = env.step(a)
            assert np.array_equal(u32(rew), r_ref.view(np.uint32))
            assert torch.equal(obs.cpu(), torch.from_numpy(o_ref)), it
        rew, done = env.rollout(T)                             # no obs written
        for t in range(T):
            _, r_ref, d_ref = ora.step(_rng_actions(seed, np.arange(N), t_roll + t), want_obs=False)
            assert np.array_equal(u32(rew[t]), r_ref.view(np.uint32)), (it, t)
        t_roll += T
    a = torch.randint(0, 4, (N,), generator=gen)
    o_ref, _, _ = ora.step(a.numpy())
    obs, _, _, _ = env.step(a)
    assert torch.equal(obs.cpu(), torch.from_numpy(o_ref))
    env.close()


def test_incremental_graph_replay_guard(lmz, oracle_mod):
    """A graph captured while the tensor was in sync replays the incremental kernel; after set_state / rollout the
    replay must refuse to run until the tensor is re-rendered."""
    N, seed = 600, 3
    ora = oracle_mod.OracleVec(oracle_mod.V0, N, seed=seed)
    env = lmz.LmazeVecCuda(N, "v0", seed=seed, render_mode="incremental")
    assert torch.equal(env.reset().cpu(), torch.from_numpy(ora.reset()))
    abuf = torch.zeros(N, dtype=torch.uint8, device="cuda")
    replay = env.capture_step(abuf)
    gen = torch.Generator().manual_seed(9)
    for _ in range(4):
        a = torch.randint(0, 4, (N,), generator=gen)
        abuf.copy_(a)
        replay()
        o_ref, _, _ = ora.step(a.numpy())
        assert torch.equal(env.obs.cpu(), torch.from_numpy(o_ref))
    env.set_state(env.get_state())                             # anything that desyncs the tensor
    with pytest.raises(RuntimeError):
        replay()
    env.render_obs()                                           # full render: back in sync
    a = torch.randint(0, 4, (N,), generator=gen)
    abuf.copy_(a)
    replay()
    o_ref, _, _ = ora.step(a.numpy())
    assert torch.equal(env.obs.cpu(), torch.from_numpy(o_ref))
    env.close()


# ---------------------------------------------------------------- ADVICE r1 (low): test mode beats RANDOM_BALL = False
@pytest.mark.parametrize("random_ball,random_goal", [(False, True), (True, False), (False, False)])
def test_v3_test_mode_has_priority_over_fixed_flags(lmz, golden_dir, random_ball, random_goal):
    """lmaze_env_v3.py:145-146,154-155: mode == "test" is checked BEFORE RANDOM_GOAL / RANDOM_BALL."""
    z = np.load(os.path.join(golden_dir, "v3_table.npz"))
    env = lmz.LmazeVecCuda(7, "v3", random_ball=random_ball, random_goal=random_goal, seed=4)
    env.reset()                                                # a normal reset first (goal may have moved off 'X')
    obs = env.reset(mode="test")
    st = env.get_state().cpu().numpy()
    assert (st[:, 0:4] == np.array(z["test_info"])).all()      # ball (7,8), goal (8,8)
    assert np.array_equal(obs[3].cpu().numpy(), unpack(z["test_obs"], (3, 72, 72)))
    assert env.stats()["steps"] == 0                           # and no error was counted
    env.close()


def test_v3_test_mode_single_maze_class(lmz, golden_dir):
    z = np.load(os.path.join(golden_dir, "v3_table.npz"))
    env = lmz.LmazeEnv_v3(random_ball=False)
    obs = env.reset(mode="test")
    assert np.array_equal(obs, unpack(z["test_obs"], (3, 72, 72)))
    assert env.state_vector[0:4] == [int(v) for v in z["test_info"]]
    env.close()


# ---------------------------------------------------------------- VERDICT r1 8(c): set_state never repairs silently
def test_set_state_counts_unreachable_rows(lmz):
    env = lmz.LmazeVecCuda(6, "v0", autoreset=False)
    st = env.get_state()
    st[:, 0:2] = torch.tensor([[1, 1], [5, 5], [3, 3], [0, 4], [2, 2], [13, 1]], dtype=torch.int32)
    #                          'S' ok  'X' ok  'B' ok  border  wall    outside
    st[:, 5] = torch.tensor([0, 3, 2, 0, 0, 0], dtype=torch.int32)
    env.set_state(st)
    with pytest.raises(ValueError):
        env.stats()
    assert env.stats(check_errors=False)["steps"] == 0
    out = env.get_state().cpu().numpy()
    assert out[3, 0] == 1 and out[5, 0] == 10                  # clamped into the interior, and counted
    env.close()
    env = lmz.LmazeVecCuda(3, "v0", autoreset=False)
    st = env.get_state()
    st[:, 0:2] = torch.tensor([[1, 1], [5, 5], [10, 10]], dtype=torch.int32)
    env.set_state(st)
    env.stats()                                                # reachable rows: no error
    env.close()
    env = lmz.LmazeVecCuda(3, "v3", autoreset=False)
    st = env.get_state()
    st[:, 0:4] = torch.tensor([[4, 4, 8, 8], [4, 5, 0, 0], [4, 6, 8, 8]], dtype=torch.int32)   # row 1: goal on the border
    env.set_state(st)
    with pytest.raises(ValueError):
        env.stats()
    env.close()
    for variant in ("v2", "v4"):
        env = lmz.LmazeVecCuda(2, variant, autoreset=False)
        st = env.get_state()
        env.set_state(st)
        env.stats()
        st[1, 0] = 1                                           # the ball never leaves [2, 15]
        env.set_state(st)
        with pytest.raises(ValueError):
            env.stats()
        env.close()
    h = lmz.LmazeHierCuda(2, "v5", autoreset=False)
    h.reset()
    st = h.get_state()
    h.set_state(st)
    h.stats()
    st[0, 12] = 31                                             # foveal goal cell outside 0..24
    h.set_state(st)
    with pytest.raises(ValueError):
        h.stats()
    h.close()


# ---------------------------------------------------------------- bit-packed observations (SURVEY 8d(ii): 72 B per v0 env)
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_bits_obs_reconstructs_reference_image(lmz, oracle_mod, variant):
    """obs_mode='bits': 1 bit per cell of the un-expanded layers; unpack + xE replication is the oracle's full image
    every step (auto-resets, invalid actions, a masked reset, a render window, the batch tail)."""
    N, T = 3001, 230
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=11, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=11, autoreset=True, obs_mode="bits")
    assert env.obs.dtype == torch.uint8 and tuple(env.obs.shape) == (N, 72 if variant == "v0" else 124)
    assert torch.equal(env.expand(env.reset()).cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(2)
    for t in range(T):
        a = torch.randint(0, 5, (N,), generator=gen)
        want = t % 5 == 0 or t > T - 3
        o_ref, r_ref, d_ref = ora.step(a.numpy(), want_obs=want)
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
        if want:
            assert torch.equal(env.expand(obs).cpu(), torch.from_numpy(o_ref)), t
        if variant == "v3":
            assert int((obs[:, 121] >> 4).max()) == 0 and int(obs[:, 122:].max()) == 0     # pad bits stay zero
    # compact twin: the bits are exactly the compact bytes
    twin = lmz.LmazeVecCuda(N, variant, seed=11, obs_mode="compact")
    twin.set_state(env.get_state())
    assert torch.equal(env.unpack_bits(env.render_obs()), twin.render_obs())
    twin.close()
    # masked reset: only the masked rows change
    before = env.obs.clone()
    mask = torch.rand(N, generator=gen) < 0.25
    env.reset(mask=mask)
    assert torch.equal(env.obs[~mask.cuda()], before[~mask.cuda()])
    env.close()
    # render window
    env = lmz.LmazeVecCuda(N, variant, seed=11, obs_mode="bits", obs_window=1000)
    ora = oracle_mod.OracleVec(ov, N, seed=11)
    env.reset(); ora.reset(want_obs=False)
    for t in range(6):
        a = torch.randint(0, 4, (N,), generator=gen)
        o_ref, _, _ = ora.step(a.numpy())
        if t % 2 == 0:
            env.set_window(777 * (t // 2) + 1)
        obs, _, _, _ = env.step(a)
        assert torch.equal(env.expand(obs).cpu(), torch.from_numpy(o_ref[env.window_lo:env.window_lo + 1000])), t
    env.close()
    with pytest.raises(Exception):
        lmz.LmazeVecCuda(4, "v2", obs_mode="bits")


# ---------------------------------------------------------------- rollout with 1-byte reward codes
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_rollout_reward_codes(lmz, variant):
    N, T = 5000, 150
    a = lmz.LmazeVecCuda(N, variant, seed=5, with_obs=False)
    b = lmz.LmazeVecCuda(N, variant, seed=5, with_obs=False)
    a.reset(); b.reset()
    table = a.reward_table("cuda")
    assert u32(table).tolist() == REWARD_BITS.tolist()
    for it in range(2):
        rew, done_a = a.rollout(T)
        codes, done_b = b.rollout(T, reward_codes=True)
        assert codes.dtype == torch.uint8 and int(codes.max()) <= 3
        assert torch.equal(table[codes.long()].view(torch.int32), rew.view(torch.int32))
        assert torch.equal(done_a, done_b)
    assert torch.equal(a.get_state(), b.get_state()) and a.stats() == b.stats()
    acts = torch.randint(0, 6, (T, N), device="cuda", dtype=torch.uint8)
    rew, _ = a.rollout(T, actions=acts)
    codes, _ = b.rollout(T, actions=acts, reward_codes=torch.empty((T, N), dtype=torch.uint8, device="cuda"))
    assert torch.equal(table[codes.long()].view(torch.int32), rew.view(torch.int32))
    a.close(); b.close()


# ---------------------------------------------------------------- double-buffered host pipeline
@pytest.mark.parametrize("variant,obs_mode", [("v0", "compact"), ("v0", "bits"), ("v3", "bits"), ("v0", "full")])
def test_host_pipeline_matches_oracle(lmz, oracle_mod, variant, obs_mode):
    """lmz_step_host_async / _wait: every output of every step (obs included) lands in pinned host memory one
    submit later and equals the oracle's; the full f32 observation stays on the device (with_obs=False)."""
    N, T = 4099, 40
    ov = oracle_mod.V0 if variant == "v0" else oracle_mod.V3
    ora = oracle_mod.OracleVec(ov, N, seed=21, autoreset=True)
    env = lmz.LmazeVecCuda(N, variant, seed=21, autoreset=True, obs_mode=obs_mode)
    env.reset(); ora.reset(want_obs=False)
    if obs_mode == "full":
        with pytest.raises(ValueError):
            env.host_pipeline()
    pipe = env.host_pipeline(with_obs=obs_mode != "full")
    gen = torch.Generator().manual_seed(4)
    acts = [torch.randint(0, 5, (N,), generator=gen, dtype=torch.uint8).pin_memory() for _ in range(T)]
    refs = []

    def check(res, ref):
        o_ref, r_ref, d_ref = ref
        assert np.array_equal(res.reward.numpy().view(np.uint32), r_ref.view(np.uint32))
        assert np.array_equal(res.done.numpy(), d_ref)
        if res.obs is not None:
            assert torch.equal(env.expand(res.obs.cuda()).cpu(), torch.from_numpy(o_ref))
    for t in range(T):
        refs.append(ora.step(acts[t].numpy().astype(np.int64)))
        res = pipe.submit(acts[t])
        assert (res is None) == (t == 0)
        if res is not None:
            check(res, refs[t - 1])
    check(pipe.drain(), refs[-1])
    assert pipe.drain() is None
    # the pipeline can be resumed after a drain, and the serial host call still works beside it
    refs.append(ora.step(acts[0].numpy().astype(np.int64)))
    assert pipe.submit(acts[0]) is None
    check(pipe.drain(), refs[-1])
    r = torch.empty(N, dtype=torch.float32).pin_memory(); d = torch.empty(N, dtype=torch.uint8).pin_memory()
    o_ref, r_ref, d_ref = ora.step(acts[1].numpy().astype(np.int64))
    env.step_host(acts[1], r, d)
    assert np.array_equal(r.numpy().view(np.uint32), r_ref.view(np.uint32)) and np.array_equal(d.numpy(), d_ref)
    assert torch.equal(env.expand(env.obs).cpu(), torch.from_numpy(o_ref))
    assert env.stats()["steps"] == (T + 2) * N
    env.close()


# ---------------------------------------------------------------- the visit layer kept as its HISTORY (v4 / v5), edge cases
@pytest.mark.parametrize("obs_mode", ["full", "compact"])
def test_v4_visit_layer_long_episode_without_reset(lmz, oracle_mod, obs_mode):
    """autoreset off and no reset for 330 steps: the layer is averaged 330 times in a row, far past the 64 entries
    the visit history holds (the 65th averaging materialises the layer and goes to direct mode) and deep into the
    float32 denormals (values halve down to 2^-149 and round to zero step by step).  Whole layer + whole observation
    vs the oracle, bit for bit."""
    N, T = 777, 330
    ora = oracle_mod.OracleVec(oracle_mod.V4, N, seed=31, autoreset=False, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, "v4", seed=31, autoreset=False, obs_mode=obs_mode)
    assert torch.equal(env.expand(env.reset()).cpu(), torch.from_numpy(ora.reset()))
    gen = torch.Generator().manual_seed(8)
    small = 0
    for t in range(T):
        # keep most envs in one corner so that the far cells are never visited again and decay all the way down
        a = torch.randint(0, 25, (N,), generator=gen)
        a[N // 2:] = 12
        o_ref, r_ref, d_ref = ora.step(a.numpy())
        obs, rew, done, _ = env.step(a)
        assert np.array_equal(u32(rew), r_ref.view(np.uint32)) and np.array_equal(done.cpu().numpy().view(np.uint8), d_ref), t
        assert np.array_equal(u32(env.expand(obs)), u32(o_ref)), t
        if t % 20 == 19 or t in (61, 62, 63, 64, 65, 66, 148, 149, 150, 151):
            vref = ora.export_visit()
            assert np.array_equal(u32(env.get_visit()), u32(vref)), t
            small = max(small, int(((vref > 0) & (vref < 1.2e-38)).sum()))
    assert small > 0                                           # denormals really occurred
    # a reset returns to the history form and everything still matches
    assert np.array_equal(u32(env.expand(env.reset())), u32(ora.reset()))
    for t in range(30):
        a = torch.randint(0, 25, (N,), generator=gen)
        o_ref, _, _ = ora.step(a.numpy())
        obs, _, _, _ = env.step(a)
        assert np.array_equal(u32(env.expand(obs)), u32(o_ref)), t
    assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit()))
    env.close()


def test_v4_set_visit_arbitrary_values_then_steps(lmz, oracle_mod):
    """lmz_set_visit takes arbitrary values, which have no history (direct mode until the next reset): tiny and
    denormal values are averaged exactly like the oracle's float64 expression."""
    N, T = 300, 60
    ora = oracle_mod.OracleVec(oracle_mod.V4, N, seed=2, autoreset=False)
    env = lmz.LmazeVecCuda(N, "v4", seed=2, autoreset=False)
    env.reset(); ora.reset(want_obs=False)
    rng = np.random.RandomState(0)
    vis = (rng.rand(N, 18, 18).astype(np.float32) * np.float32(2.0) ** rng.randint(-149, 1, size=(N, 18, 18))).astype(np.float32)
    vis[rng.rand(N, 18, 18) < 0.3] = 0.0
    env.set_visit(vis)
    for i in range(N):
        ora.set_visit(i, vis[i])
    assert np.array_equal(u32(env.get_visit()), u32(vis))
    for t in range(T):
        a = rng.randint(0, 25, size=N)
        o_ref, _, _ = ora.step(a)
        obs, _, _, _ = env.step(a)
        assert np.array_equal(u32(obs), u32(o_ref)), t
        assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit())), t
    # checkpoint round trip in the middle of an episode: state + TRUE visit values into a fresh handle
    env2 = lmz.LmazeVecCuda(N, "v4", seed=2, autoreset=False)
    env2.set_state(env.get_state()); env2.set_visit(env.get_visit())
    for t in range(10):
        a = rng.randint(0, 25, size=N)
        o1, _, _, _ = env.step(a); o2, _, _, _ = env2.step(a)
        assert torch.equal(o1.view(torch.int32), o2.view(torch.int32))
    assert torch.equal(env.get_visit().view(torch.int32), env2.get_visit().view(torch.int32))
    env.close(); env2.close()


def test_v5_visit_layer_many_averagings_without_planner(lmz, oracle_mod):
    """lmaze-v5 averages the layer on EVERY step while the local episode is over (lmaze_env_v5.py:308-312): an actor
    that keeps stepping without plannerStep averages it hundreds of times -- past the 64 history entries and into the
    denormals."""
    N, T = 600, 260
    ora = oracle_mod.OracleHier(N, seed=9)
    env = lmz.LmazeHierCuda(N, "v5", seed=9, autoreset=False)
    assert np.array_equal(u32(env.reset()), u32(ora.reset()))
    rng = np.random.RandomState(1)
    g = rng.randint(0, 25, size=N)
    env.plannerStep(g); ora.planner_step(g)
    for t in range(T):
        a = rng.randint(0, 4, size=N)
        fov, loc, gr, lr, gd, ld, _, _ = env.step(a, goal_plane=False)
        f_ref, l_ref, gr_ref, lr_ref, gd_ref, ld_ref, err = ora.step(a)
        assert np.array_equal(u32(fov), u32(f_ref)), t
        assert np.array_equal(ld.cpu().numpy(), ld_ref.astype(bool)), t
        if t % 20 == 19 or t in (70, 71, 72, 73, 74, 75, 76):
            assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit())), t
    assert int(ld_ref.sum()) > N // 2                          # most envs sat in "local episode over" for ~250 steps
    vref = ora.export_visit()
    assert int(((vref > 0) & (vref < 1.2e-38)).sum()) > 0      # denormals occurred
    env.close()


# ---------------------------------------------------------------- rollout kernels of the foveal variants
@pytest.mark.parametrize("variant", ["v2", "v4"])
def test_foveal_rollout_kernel_parity(lmz, oracle_mod, variant):
    """lmz_rollout for lmaze-v2 / v4: T fused steps per launch, Philox actions (spec: DESIGN.md section 4) or a
    [T,N] action buffer; per-step reward bits / done flags, final state, episode counters, v4's visit layer and
    the observation rendered afterwards, all against the oracle stepped one call at a time."""
    N, seed, T = 1537, 77, 70
    ov = oracle_mod.V2 if variant == "v2" else oracle_mod.V4
    ora = oracle_mod.OracleVec(ov, N, seed=seed, env_id0=3, autoreset=True, threads=os.cpu_count() or 1)
    env = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=3, autoreset=True)
    assert np.array_equal(u32(env.reset()), u32(ora.reset()))
    t_glob = 0
    for rnd in range(3):
        if rnd == 1:                                           # caller-supplied actions (incl. a few out of range: clamped + counted)
            acts = np.random.RandomState(rnd).randint(0, 25, size=(T, N))
            acts[5, :7] = 30
            rew, done = env.rollout(T, actions=torch.as_tensor(acts))
        elif rnd == 2:
            acts = np.array([[oracle_mod.rng_action25(seed, 3 + i, t_glob + t) for i in range(N)] for t in range(T)])
            codes, done = env.rollout(T, reward_codes=True)
            rew = env.reward_table("cuda")[codes.long()]
        else:
            acts = np.array([[oracle_mod.rng_action25(seed, 3 + i, t_glob + t) for i in range(N)] for t in range(T)])
            rew, done = env.rollout(T)
        t_glob += T
        for t in range(T):
            _, r_ref, d_ref = ora.step(acts[t], want_obs=False)
            assert np.array_equal(u32(rew[t]), r_ref.view(np.uint32)), (rnd, t)
            assert np.array_equal(done[t].cpu().numpy().view(np.uint8), d_ref), (rnd, t)
        st = env.get_state().cpu().numpy()
        pos, sc, _, _ = ora.export()
        assert np.array_equal(st[:, 0:4], pos) and np.array_equal(st[:, 4], sc) and np.array_equal(st[:, 7], ora.episode)
        if variant == "v4":
            assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit())), rnd
        full = np.stack([ora.render_one(i) for i in range(N)])
        assert np.array_equal(u32(env.render_obs()), u32(full)), rnd
    # short rollouts too (T = 5, 1, 7)
    for T_short in (5, 1, 7):
        acts = np.array([[oracle_mod.rng_action25(seed, 3 + i, t_glob + t) for i in range(N)] for t in range(T_short)])
        rew, done = env.rollout(T_short)
        t_glob += T_short
        for t in range(T_short):
            _, r_ref, d_ref = ora.step(acts[t], want_obs=False)
            assert np.array_equal(u32(rew[t]), r_ref.view(np.uint32)) and np.array_equal(done[t].cpu().numpy().view(np.uint8), d_ref)
    if variant == "v4":
        assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit()))
    s = env.stats(check_errors=False)
    assert [s[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist() and s["episodes"] > N
    # ... and ordinary steps continue from the rolled-out state
    a = np.random.RandomState(9).randint(0, 25, size=N)
    o_ref, r_ref, _ = ora.step(a)
    obs, rew, _, _ = env.step(a)
    assert np.array_equal(u32(obs), u32(o_ref)) and np.array_equal(u32(rew), r_ref.view(np.uint32))
    env.close()


@pytest.mark.parametrize("philox", [True, False])
def test_hier_rollout_kernel_parity(lmz, oracle_mod, philox):
    """lmz_hier_rollout (lmaze-v5 / v6): per step plannerStep for the envs waiting for their planner, then step(),
    auto-reset on globalDone; both rewards and both done flags per step, final state words and visit layer."""
    N, seed, T = 1201, 5, 90
    ora = oracle_mod.OracleHier(N, seed=seed, env_id0=40)
    env = lmz.LmazeHierCuda(N, "v5", seed=seed, env_id0=40, autoreset=True)
    assert np.array_equal(u32(env.reset()), u32(ora.reset()))
    t_glob = 0
    for rnd in range(2):
        if philox:
            ga = np.array([[oracle_mod.rng_hier(seed, 40 + i, t_glob + t) for i in range(N)] for t in range(T)])
            goals, acts = ga[:, :, 0], ga[:, :, 1]
            gr, lr, gd, ld = env.rollout(T)
        else:
            rs = np.random.RandomState(rnd)
            goals, acts = rs.randint(0, 25, size=(T, N)), rs.randint(0, 5, size=(T, N))     # 4 = unmatched action: no move
            gr, lr, gd, ld = env.rollout(T, goals=torch.as_tensor(goals), actions=torch.as_tensor(acts))
        t_glob += T
        for t in range(T):
            st = ora.export()
            need = (((st[:, 15] >> 1) & 1) | (st[:, 14] == 0)).astype(np.uint8)          # localDone, or no plannerStep since reset
            if need.any():
                ora.planner_step(goals[t], mask=need)
            _, _, gr_ref, lr_ref, gd_ref, ld_ref, _ = ora.step(acts[t])
            assert np.array_equal(u32(gr[t]), gr_ref.view(np.uint32)) and np.array_equal(u32(lr[t]), lr_ref.view(np.uint32)), (rnd, t)
            assert np.array_equal(gd[t].cpu().numpy(), gd_ref.astype(bool)) and np.array_equal(ld[t].cpu().numpy(), ld_ref.astype(bool)), (rnd, t)
            if gd_ref.any():
                ora.reset(mask=gd_ref, want_obs=False)
        st, ref = env.get_state().cpu().numpy(), ora.export()
        assert np.array_equal(st[:, :13], ref[:, :13]) and np.array_equal(st[:, 15], ref[:, 15])
        assert np.array_equal(np.minimum(st[:, 13:15], 255), np.minimum(ref[:, 13:15], 255))
        assert np.array_equal(st[:, 16].astype(np.uint32), ora.episode)
        assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit())), rnd
        fov_ref, loc_ref, err_ref = ora.render()
        env.render_obs()
        assert np.array_equal(u32(env.obs), u32(fov_ref)) and np.array_equal(u32(env.loc_obs), u32(loc_ref))
        if rnd == 0:                                       # a short rollout in between
            ga = np.array([[oracle_mod.rng_hier(seed, 40 + i, t_glob + t) for i in range(N)] for t in range(6)])
            gr6, lr6, gd6, ld6 = env.rollout(6) if philox else env.rollout(6, goals=torch.as_tensor(ga[:, :, 0]), actions=torch.as_tensor(ga[:, :, 1]))
            t_glob += 6
            for t in range(6):
                st6 = ora.export()
                need = (((st6[:, 15] >> 1) & 1) | (st6[:, 14] == 0)).astype(np.uint8)
                if need.any():
                    ora.planner_step(ga[t, :, 0], mask=need)
                _, _, gr_ref, lr_ref, gd_ref, ld_ref, _ = ora.step(ga[t, :, 1])
                assert np.array_equal(u32(gr6[t]), gr_ref.view(np.uint32)) and np.array_equal(ld6[t].cpu().numpy(), ld_ref.astype(bool)), t
                if gd_ref.any():
                    ora.reset(mask=gd_ref, want_obs=False)
            assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit()))
    assert env.stats(check_errors=False)["steps"] == (2 * T + 6) * N
    env.close()


@pytest.mark.parametrize("variant", ["v2", "v4", "v5"])
def test_foveal_rollout_soak_and_shards(lmz, variant):
    """65,536 envs x 600 rolled-out steps in chunks == the same envs stepped through the fused step kernel with the
    same action stream (the two kernels share one transition), and two half-batch handles == the whole batch."""
    N, T, chunks = 1 << 16, 120, 5
    hier = variant == "v5"
    mk = (lambda n, id0: lmz.LmazeHierCuda(n, "v5", seed=12, env_id0=id0, obs_mode="compact")) if hier else \
         (lambda n, id0: lmz.LmazeVecCuda(n, variant, seed=12, env_id0=id0, obs_mode="compact"))
    whole, lo, hi = mk(N, 0), mk(N // 2, 0), mk(N // 2, N // 2)
    for e in (whole, lo, hi):
        e.reset()
    for c in range(chunks):
        outs = [e.rollout(T) for e in (whole, lo, hi)]
        for k in range(len(outs[0])):
            assert torch.equal(outs[0][k], torch.cat([outs[1][k], outs[2][k]], dim=1)), (c, k)
    assert torch.equal(whole.get_state(), torch.cat([lo.get_state(), hi.get_state()]))
    sw = whole.stats(check_errors=False)
    sl, sh = lo.stats(check_errors=False), hi.stats(check_errors=False)
    assert all(sw[k] == sl[k] + sh[k] for k in sw) and sw["steps"] == N * T * chunks and sw["episodes"] > N
    # replay the first chunk of a fresh handle through the step kernel with the recorded... Philox stream
    if not hier:
        from oracle import oracle as O
        a = mk(4096, 0); b = mk(4096, 0)
        a.reset(); b.reset()
        rew, done = a.rollout(40)
        ids = np.arange(4096, dtype=np.uint64)
        for t in range(40):
            acts = np.array([O.rng_action25(12, int(i), t) for i in ids[:4096]])
            _, r, d, _ = b.step(acts)
            assert torch.equal(r.view(torch.int32), rew[t].view(torch.int32)) and torch.equal(d, done[t]), t
        assert torch.equal(a.get_state(), b.get_state())
        if variant == "v4":
            assert torch.equal(a.get_visit().view(torch.int32), b.get_visit().view(torch.int32))
        a.close(); b.close()
    for e in (whole, lo, hi):
        e.close()
