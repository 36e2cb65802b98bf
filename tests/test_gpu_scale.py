"""GPU tier, BASELINE.json's full sizes off the default path (VERDICT r1 item 9): the ST128 render at 2^20 envs,
lmaze-v3 at 8 M envs through a render window, lmaze-v5 at 2^20 envs with the device-side planner mask.  At these
sizes the oracle cannot step every env, so each test checks (a) size-independent properties of EVERY row of the
tensors and (b) a contiguous block of 1,024 envs from the middle of the batch replayed by the oracle from reset
with the same global env ids (the device RNG is keyed by global id), bit for bit, every step."""
import numpy as np
import pytest
import torch

from gpu_helpers import REWARD_BITS, lmz, need_free, u32

pytestmark = pytest.mark.gpu


def test_one_million_envs_st128_render(lmz, oracle_mod):
    """configs[2] size on the 128-bit vector-store render path (LMZ_RENDER_ST128): 2^20 envs x 112,896 B."""
    N, B, LO, seed = 1 << 20, 1024, 555_555, 77
    need_free(N * 112896 + (4 << 30))
    env = lmz.LmazeVecCuda(N, "v0", seed=seed, render_mode="st128")
    ora = oracle_mod.OracleVec(oracle_mod.V0, B, seed=seed, env_id0=LO)
    obs = env.reset()
    assert np.array_equal(u32(obs[LO:LO + B]), u32(ora.reset()))
    gen = torch.Generator(device="cuda").manual_seed(1)
    for t in range(4):
        a = torch.randint(0, 5, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        obs, rew, done, _ = env.step(a)
        o_ref, r_ref, d_ref = ora.step(a[LO:LO + B].cpu().numpy().astype(np.int64))
        assert np.array_equal(u32(rew[LO:LO + B]), r_ref.view(np.uint32)), t
        assert np.array_equal(done[LO:LO + B].cpu().numpy().view(np.uint8), d_ref), t
        assert np.array_equal(u32(obs[LO:LO + B]), u32(o_ref)), t
    st = env.get_state()
    assert torch.isin(rew.view(torch.int32), torch.as_tensor(REWARD_BITS.view(np.int32)).cuda()).all()
    want = torch.tensor([49.0, 3528.0, 49.0, 3430.0], device="cuda")          # per-env channel sums (SURVEY 8a, a10)
    CH = 1 << 14
    for lo in range(0, N, CH):
        o = obs[lo:lo + CH]
        assert torch.equal(o.sum(dim=(2, 3)), want.expand(o.shape[0], 4))
        x, y = st[lo:lo + CH, 0].long(), st[lo:lo + CH, 1].long()
        idx = torch.arange(o.shape[0], device="cuda")
        assert (o[idx, 0, 7 * x, 7 * y] == 1).all() and (o[idx, 0, 7 * x + 6, 7 * y + 6] == 1).all()
        assert torch.equal(o[:, 1:], obs[0:1, 1:].expand(o.shape[0], 3, 84, 84))   # static channels identical
    s = env.stats()
    assert s["steps"] == 4 * N and s["wall_bumps"] + s["moves"] + s["stale"] == 4 * N
    env.close()


def test_v3_eight_million_envs_through_a_window(lmz, oracle_mod):
    """BASELINE configs[3] on ONE GPU: 8 M lmaze-v3 envs (498 GB of observations) consumed through a 1 M-env render
    window -- a step advances every env and renders window 0, lmz_render re-renders the other seven."""
    N, W, B, LO, seed = 1 << 23, 1 << 20, 1024, 5 * (1 << 20) + 333_333, 5
    need_free(W * 62208 + (4 << 30))
    env = lmz.LmazeVecCuda(N, "v3", seed=seed, obs_window=W)
    ora = oracle_mod.OracleVec(oracle_mod.V3, B, seed=seed, env_id0=LO)
    env.reset()
    ora.reset(want_obs=False)
    gen = torch.Generator(device="cuda").manual_seed(2)
    for t in range(3):
        a = torch.randint(0, 5, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        env.set_window(0)
        obs, rew, done, _ = env.step(a)
        o_ref, r_ref, d_ref = ora.step(a[LO:LO + B].cpu().numpy().astype(np.int64))
        assert np.array_equal(u32(rew[LO:LO + B]), r_ref.view(np.uint32)), t
        assert np.array_equal(done[LO:LO + B].cpu().numpy().view(np.uint8), d_ref), t
    st = env.get_state()
    assert torch.isin(rew.view(torch.int32), torch.as_tensor(REWARD_BITS[[1, 2, 3]].view(np.int32)).cuda()).all()    # v3 never returns -0.0
    free = 73 * 16.0                                        # 73 free cells x 4 x 4 (lmaze_env_v3.py:166)
    want = torch.tensor([free, 16.0, 16.0], device="cuda")
    total_ball = 0.0
    for w in range(N // W):                                 # all 8 windows rendered and checked
        obs = env.obs if w == 0 else env.render_window(w * W)
        CH = 1 << 15
        for lo in range(0, W, CH):
            o = obs[lo:lo + CH]
            sums = o.sum(dim=(2, 3))
            assert torch.equal(sums, want.expand(o.shape[0], 3)), (w, lo)
            total_ball += float(sums[:, 1].sum())
            s = st[w * W + lo:w * W + lo + CH]
            idx = torch.arange(o.shape[0], device="cuda")
            assert (o[idx, 1, 4 * s[:, 0].long(), 4 * s[:, 1].long()] == 1).all()          # ball block (lmaze_env_v3.py:167)
            assert (o[idx, 2, 4 * s[:, 2].long() + 3, 4 * s[:, 3].long() + 3] == 1).all()  # goal block (:182)
            assert torch.equal(o[:, 0], obs[0:1, 0].expand(o.shape[0], 72, 72))
        if w == LO // W:
            assert np.array_equal(u32(obs[LO - w * W:LO - w * W + B]), u32(o_ref))          # the oracle's block, last step
    assert total_ball == 16.0 * N                           # checksum of checksums over the whole batch
    assert env.stats()["steps"] == 3 * N
    env.close()


def test_v5_one_million_envs_auto_planner(lmz, oracle_mod):
    """lmaze-v5 at 2^20 envs on its default CTA configuration: plannerStep with the device-side "waiting for the
    planner" mask + step + same-step auto-reset, both observation tensors."""
    N, B, LO, seed = 1 << 20, 1024, 700_001, 9
    need_free(N * (34300 + 19600 + 1296) + (4 << 30))
    env = lmz.LmazeHierCuda(N, "v5", seed=seed, autoreset=True)
    ora = oracle_mod.OracleHier(B, seed=seed, env_id0=LO)
    fov = env.reset()
    assert np.array_equal(u32(fov[LO:LO + B]), u32(ora.reset()))
    gen = torch.Generator(device="cuda").manual_seed(3)
    n_reset = n_err = 0
    for t in range(14):
        goals = torch.randint(0, 25, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        acts = torch.randint(0, 4, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        env.plannerStep(goals, mask="auto")
        fov, loc, gr, lr, gd, ld, fg, _ = env.step(acts, goal_plane=False)
        st = ora.export()
        need = (((st[:, 15] >> 1) & 1) | (st[:, 14] == 0)).astype(np.uint8)
        if need.any():
            ora.planner_step(goals[LO:LO + B].cpu().numpy().astype(np.int64), mask=need)
        f_ref, l_ref, gr_ref, lr_ref, gd_ref, ld_ref, err_ref = ora.step(acts[LO:LO + B].cpu().numpy().astype(np.int64))
        if gd_ref.any():                                    # the framework's same-step reset: both rows show the new episode
            ora.reset(mask=gd_ref, want_obs=False)
            ora.render(mask=gd_ref, fov=f_ref, loc=l_ref)
            err_ref[gd_ref.astype(bool)] = 0
            n_reset += int(gd_ref.sum())
        n_err += int(err_ref.sum())
        assert np.array_equal(u32(gr[LO:LO + B]), gr_ref.view(np.uint32)) and np.array_equal(u32(lr[LO:LO + B]), lr_ref.view(np.uint32)), t
        assert np.array_equal(gd[LO:LO + B].cpu().numpy(), gd_ref.astype(bool)) and np.array_equal(ld[LO:LO + B].cpu().numpy(), ld_ref.astype(bool)), t
        assert np.array_equal(u32(fov[LO:LO + B]), u32(f_ref)), t
        assert np.array_equal(u32(loc[LO:LO + B]), u32(l_ref)), t
    assert n_reset > 0
    assert np.array_equal(u32(env.get_visit()[LO:LO + B]), u32(ora.export_visit()))
    # properties of every row: the fovealGoal plane (ch 3) is one 7x7 block; the free-cell crop (ch 0) shows the ball's
    # own cell; binary channels are binary; the visit crops (ch 2, 6) lie in [0, 1]; IndexError rows of loc are zero
    allowed = torch.as_tensor(REWARD_BITS.view(np.int32)).cuda()
    assert torch.isin(gr.view(torch.int32), allowed).all() and torch.isin(lr.view(torch.int32), allowed).all()
    CH = 1 << 14
    for lo in range(0, N, CH):
        f, l = fov[lo:lo + CH], loc[lo:lo + CH]
        assert torch.equal(f[:, 3].sum(dim=(1, 2)), torch.full((f.shape[0],), 49.0, device="cuda"))
        assert (f[:, 0, 17, 17] == 1).all()
        b = f[:, [0, 1, 3, 4, 5]]
        assert ((b == 0) | (b == 1)).all() and (f[:, [2, 6]] >= 0).all() and (f[:, [2, 6]] <= 1).all()
        err = env.loc_err[lo:lo + CH]
        assert (l[err].sum() == 0) and ((l == 0) | (l == 1)).all()
        assert torch.equal(l[~err][:, 3].sum(dim=(1, 2)), torch.full((int((~err).sum()),), 49.0, device="cuda"))
    s = env.stats(check_errors=False)
    assert s["steps"] == 14 * N and s["episodes"] > 0
    env.close()
