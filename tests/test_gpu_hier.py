"""GPU tier, lmaze-v5 / lmaze-v6 (planner / actor env): the CUDA path through the C ABI against
(a) the golden traces recorded from the unmodified reference and (b) the CPU oracle on the same
seeded inputs -- every returned value per call, bit for bit (both observation tensors, both rewards'
bit patterns, both done flags, the IndexError flag, the packed state and the float visit layer).
"""
import numpy as np
import pytest
import torch

from golden_io import Traces, fov_image, loc_image, reward_f32_bits
from gpu_helpers import lmz, need_free, u32

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------- golden traces (reference outputs)
@pytest.mark.parametrize("variant", ["v5", "v6", "v5_edge"])
def test_hier_golden_traces(lmz, golden_dir, variant):
    """Every value the reference returned from reset / plannerStep / step over 4 x ~730 recorded events."""
    tr = Traces(golden_dir, variant)
    n_events = 0
    for e in range(tr.n_envs):
        env = lmz.LmazeHierCuda(1, variant[:2], autoreset=False)
        z = tr.env(e)
        ev = z["events"]
        for k, row in enumerate(ev):
            kind, arg, grb, orb, gd, ld, bx, by = (int(v) for v in row[:8])
            sp = [int(v) for v in row[8:13]]
            if kind == 0:
                fov = env.reset(spawn=[sp])
                assert np.array_equal(u32(fov[0]), u32(fov_image(z["fov_bits"][k], z["fov_visit"][k]))), (e, k)
            elif kind == 1:
                loc = env.plannerStep([arg])
                assert not bool(env.loc_err.item())
                assert np.array_equal(u32(loc[0]), u32(loc_image(z["loc_bits"][k]))), (e, k)
            else:
                fov, loc, gr, lr, gdo, ldo, fg, act = env.step([arg])
                assert not bool(env.loc_err.item())
                assert u32(gr)[0] == reward_f32_bits(grb), (e, k)
                assert u32(lr)[0] == reward_f32_bits(orb), (e, k)
                assert (int(gdo.item()), int(ldo.item())) == (gd, ld), (e, k)
                assert np.array_equal(u32(fov[0]), u32(fov_image(z["fov_bits"][k], z["fov_visit"][k]))), (e, k)
                assert np.array_equal(u32(loc[0]), u32(loc_image(z["loc_bits"][k]))), (e, k)
                assert fg.shape == (1, 1, 5, 5) and float(fg.sum()) == 1.0 and int(act.item()) == arg
            st = env.get_state()[0].tolist()
            assert (st[0], st[1]) == (bx, by), (e, k)
            if k % 16 == 0 or kind == 0:
                assert float(env.get_visit()[0].cpu().numpy().astype(np.float64).sum()) == z["visit_sum"][k], (e, k)
            n_events += 1
        assert env.stats()["steps"] == int((ev[:, 0] == 2).sum())
        env.close()
    assert n_events > (400 if variant == "v5_edge" else 2500)


def test_v6_safe_goal_golden(lmz, golden_dir, oracle_mod):
    """safeFovealGoal (lmaze_env_v6.py:505-523) with the reference's own np.random draws injected."""
    tr = Traces(golden_dir, "v6")
    rows = [str(r) for r in tr["safe_layout"]]
    k = [i for i in range(1, 6) if oracle_mod.layout_v2(i) == rows][0]
    res = tr["safe_results"]
    n = len(res)
    env = lmz.LmazeHierCuda(n, "v6", autoreset=False)
    env.reset()
    st = env.get_state()
    st[:, 0] = torch.as_tensor(res[:, 0]); st[:, 1] = torch.as_tensor(res[:, 1])
    st[:, 15] = k << 4
    env.set_state(st)
    draws = np.zeros((n, 40), np.int64)
    pos = 0
    for i, (bx, by, want, used) in enumerate(res):
        chunk = tr["safe_draws"][pos:pos + 40]
        draws[i, :len(chunk)] = chunk
        pos += int(used)
    goals, used = env.safeFovealGoal(draws)
    assert np.array_equal(goals.cpu().numpy().astype(np.int64), res[:, 2])
    assert np.array_equal(used.cpu().numpy().astype(np.int64), res[:, 3])
    # device RNG: always a non-wall cell of the window, and every non-wall cell comes up
    env2 = lmz.LmazeHierCuda(8192, "v6", autoreset=False, seed=5)
    env2.reset()
    st = env2.get_state()
    st[:, 0], st[:, 1], st[:, 15] = int(res[0, 0]), int(res[0, 1]), k << 4
    env2.set_state(st)
    g = env2.safeFovealGoal().cpu().numpy().astype(np.int64)
    bx, by = int(res[0, 0]), int(res[0, 1])
    free = np.array([rows[bx - 2 + a // 5][by - 2 + a % 5] != "W" for a in range(25)])
    counts = np.bincount(g, minlength=25)
    assert counts[~free].sum() == 0 and (counts[free] > 0).all()
    expect = 8192 / free.sum()
    assert (np.abs(counts[free] - expect) < 6 * np.sqrt(expect)).all()
    env.close(); env2.close()


# ---------------------------------------------------------------- batched parity vs the oracle
def _drive(lmz, oracle_mod, n, iters, seed, autoreset):
    env = lmz.LmazeHierCuda(n, "v5", seed=seed, autoreset=autoreset, env_id0=1000)
    ora = oracle_mod.OracleHier(n, seed=seed, env_id0=1000)
    rng = np.random.RandomState(seed)
    fov = env.reset()
    fov_ref = ora.reset()
    assert np.array_equal(u32(fov), u32(fov_ref))
    need_plan = np.ones(n, np.uint8)
    n_err = n_gd = n_ld = 0
    for it in range(iters):
        goals = rng.randint(0, 25, size=n)
        if need_plan.any():
            loc = env.plannerStep(goals, mask=need_plan)
            loc_ref, err_ref = ora.planner_step(goals, mask=need_plan)
            m = need_plan.astype(bool)
            assert np.array_equal(u32(loc)[m], u32(loc_ref)[m]), it
            assert np.array_equal(env.loc_err.cpu().numpy()[m], err_ref[m].astype(bool)), it
        acts = rng.randint(0, 4, size=n)
        acts[rng.rand(n) < 0.05] = 7                       # unmatched action: no move (lmaze_env_v5.py:203-217)
        fov, loc, gr, lr, gd, ld, fg, _ = env.step(torch.as_tensor(acts), goal_plane=False)
        fov_ref, loc_ref, gr_ref, lr_ref, gd_ref, ld_ref, err_ref = ora.step(acts)
        assert np.array_equal(u32(gr), u32(gr_ref)) and np.array_equal(u32(lr), u32(lr_ref)), it
        assert np.array_equal(gd.cpu().numpy(), gd_ref.astype(bool)), it
        assert np.array_equal(ld.cpu().numpy(), ld_ref.astype(bool)), it
        gdm = gd_ref.astype(bool)
        if autoreset and gdm.any():
            # the framework's same-step reset: both rows show the new episode (Philox spawn, same spec both sides)
            ora.reset(mask=gdm.astype(np.uint8), want_obs=False)
            ora.render(mask=gdm.astype(np.uint8), fov=fov_ref, loc=loc_ref)
            err_ref[gdm] = 0
        assert np.array_equal(env.loc_err.cpu().numpy(), err_ref.astype(bool)), it
        assert np.array_equal(u32(fov), u32(fov_ref)), it
        assert np.array_equal(u32(loc), u32(loc_ref)), it            # IndexError rows are all zero on both sides
        n_err += int(err_ref.sum()); n_gd += int(gdm.sum()); n_ld += int(ld_ref.sum())
        if not autoreset and gdm.any():
            fov = env.reset(mask=gdm)
            fov_ref2 = ora.reset(mask=gdm.astype(np.uint8))
            assert np.array_equal(u32(fov)[gdm], u32(fov_ref2)[gdm]), it
        need_plan = (ld_ref | gd_ref).astype(np.uint8)
        if it % 10 == 9 or it == iters - 1:
            st = env.get_state().cpu().numpy()
            ref = ora.export()
            assert np.array_equal(st[:, :13], ref[:, :13]), it
            assert np.array_equal(np.minimum(st[:, 13:15], 255), np.minimum(ref[:, 13:15], 255)), it
            assert np.array_equal(st[:, 15], ref[:, 15]), it
            assert np.array_equal(st[:, 16].astype(np.uint32), ora.episode), it
            assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit())), it
            assert np.array_equal(env.foveal_goal.cpu().numpy().astype(np.int32), ref[:, 12]), it
    stats = env.stats(check_errors=False)
    assert stats["steps"] == n * iters and stats["episodes"] == n_gd
    env.close()
    return n_err, n_gd, n_ld


@pytest.mark.parametrize("autoreset", [False, True])
def test_hier_batched_parity(lmz, oracle_mod, autoreset):
    n_err, n_gd, n_ld = _drive(lmz, oracle_mod, 4099, 140, 11 + int(autoreset), autoreset)
    assert n_err > 50 and n_gd > 500 and n_ld > 20000      # the IndexError rows, resets and planner cycles all occurred


def test_hier_state_roundtrip_and_render(lmz, oracle_mod):
    n = 1000
    env = lmz.LmazeHierCuda(n, "v5", seed=3, autoreset=False)
    ora = oracle_mod.OracleHier(n, seed=3)
    env.reset(); ora.reset()
    rng = np.random.RandomState(0)
    for it in range(25):
        g = rng.randint(0, 25, size=n)
        m = np.ones(n, np.uint8) if it == 0 else (rng.rand(n) < 0.3).astype(np.uint8)
        env.plannerStep(g, mask=m); ora.planner_step(g, mask=m)
        a = rng.randint(0, 4, size=n)
        env.step(a, goal_plane=False); ora.step(a)
    st, vis = env.get_state(), env.get_visit()
    fov_ref, loc_ref, err_ref = ora.render()
    # a second handle restored from the checkpoint renders the same two tensors
    env2 = lmz.LmazeHierCuda(n, "v5", seed=3, autoreset=False)
    env2.set_state(st); env2.set_visit(vis)
    env2.render_obs()
    assert np.array_equal(u32(env2.obs), u32(fov_ref)) and np.array_equal(u32(env2.loc_obs), u32(loc_ref))
    assert np.array_equal(env2.loc_err.cpu().numpy(), err_ref.astype(bool))
    assert torch.equal(env2.get_state(), st)
    # ... and continues identically
    g = rng.randint(0, 25, size=n); a = rng.randint(0, 4, size=n)
    for e_ in (env, env2):
        e_.plannerStep(g); e_.step(a, goal_plane=False)
    assert torch.equal(env.obs, env2.obs) and torch.equal(env.loc_obs, env2.loc_obs)
    assert torch.equal(env.get_visit(), env2.get_visit()) and torch.equal(env.get_state(), env2.get_state())
    env.close(); env2.close()


def test_hier_compat_classes(lmz, golden_dir):
    """LmazeEnv_v5 / LmazeEnv_v6 with the reference's exact call surface and return types."""
    z = Traces(golden_dir, "v6").env(0)
    env = lmz.make("lmaze-v6")
    assert type(env).__name__ == "LmazeEnv_v6"
    ev = z["events"]
    for k, row in enumerate(ev[:120]):
        kind, arg, grb, orb, gd, ld = (int(v) for v in row[:6])
        if kind == 0:
            fov = env.reset(spawn=[int(v) for v in row[8:13]])
            assert isinstance(fov, np.ndarray) and fov.shape == (7, 35, 35) and fov.dtype == np.float32
        elif kind == 1:
            loc = env.plannerStep(arg)
            assert loc.shape == (4, 35, 35) and np.array_equal(loc, loc_image(z["loc_bits"][k]))
        else:
            out = env.step(arg)
            assert len(out) == 8
            assert isinstance(out[2], float) and np.float64(out[2]).view(np.int64) == grb
            assert isinstance(out[3], float) and np.float64(out[3]).view(np.int64) == orb
            assert out[4] is bool(gd) and out[5] is bool(ld) and out[6].shape == (1, 5, 5) and out[7] == arg
            assert np.array_equal(u32(out[0]), u32(fov_image(z["fov_bits"][k], z["fov_visit"][k])))
    assert 0 <= env.safeFovealGoal() <= 24
    with pytest.raises(IndexError):
        env.plannerStep(25)
    env.close()
    vec = lmz.make("lmaze-vec-v5", num_envs=64)
    assert type(vec).__name__ == "LmazeHierCuda" and vec.reset().shape == (64, 7, 35, 35)
    with pytest.raises(ValueError):
        lmz.LmazeVecCuda(4, "v5")
    vec.close()


def test_hier_auto_mask_and_host_step(lmz, oracle_mod):
    """plannerStep(mask="auto") picks exactly the envs that wait for their planner (localDone set, or no
    plannerStep since reset -- incl. envs that auto-reset in the previous step); step_host is the same pair
    of launches through host buffers."""
    n, seed = 3000, 21
    env = lmz.LmazeHierCuda(n, "v5", seed=seed, autoreset=True)
    ora = oracle_mod.OracleHier(n, seed=seed)
    env.reset(); ora.reset()
    rng = np.random.RandomState(3)
    want_mask = np.ones(n, np.uint8)
    pin = lambda t: t.pin_memory()
    gr_h, lr_h = pin(torch.empty(n, dtype=torch.float32)), pin(torch.empty(n, dtype=torch.float32))
    gd_h, ld_h = pin(torch.empty(n, dtype=torch.uint8)), pin(torch.empty(n, dtype=torch.uint8))
    for it in range(80):
        goals = rng.randint(0, 25, size=n); acts = rng.randint(0, 4, size=n)
        if it % 2 == 0:
            env.plannerStep(goals, mask="auto")
            env.step(acts, goal_plane=False)
            gr, lr, gd, ld = env.reward.cpu(), env.local_reward.cpu(), env._done_u8.cpu(), env._ldone_u8.cpu()
        else:
            env.step_host(pin(torch.as_tensor(goals, dtype=torch.uint8)), pin(torch.as_tensor(acts, dtype=torch.uint8)),
                          gr_h, lr_h, gd_h, ld_h)
            gr, lr, gd, ld = gr_h.clone(), lr_h.clone(), gd_h.clone(), ld_h.clone()
        loc_p, _ = ora.planner_step(goals, mask=want_mask)
        fov_ref, loc_ref, gr_ref, lr_ref, gd_ref, ld_ref, err_ref = ora.step(acts)
        assert np.array_equal(u32(gr), u32(gr_ref)) and np.array_equal(u32(lr), u32(lr_ref)), it
        assert np.array_equal(gd.numpy(), gd_ref) and np.array_equal(ld.numpy(), ld_ref), it
        gdm = gd_ref.astype(bool)
        if gdm.any():
            ora.reset(mask=gdm.astype(np.uint8), want_obs=False)
            ora.render(mask=gdm.astype(np.uint8), fov=fov_ref, loc=loc_ref)
        assert np.array_equal(u32(env.obs), u32(fov_ref)) and np.array_equal(u32(env.loc_obs), u32(loc_ref)), it
        want_mask = (gd_ref | ld_ref).astype(np.uint8)
    assert np.array_equal(env.get_state().cpu().numpy()[:, :13], ora.export()[:, :13])
    env.close()


@pytest.mark.parametrize("flags", [(False, True), (True, False), (False, False)])
def test_foveal_random_flags(lmz, oracle_mod, flags):
    """RANDOM_BALL / RANDOM_GOAL False (lmaze_env_v2.py:51-52,278-299; same in v4, v5): the ball starts on the
    maze's 'S' cell, the goal sits on its 'X' cell -- device-RNG resets, v2 + v4 + v5 against the oracle."""
    rb, rg = flags
    n = 700
    for variant, ov in (("v2", oracle_mod.V2), ("v4", oracle_mod.V4)):
        env = lmz.LmazeVecCuda(n, variant, seed=8, autoreset=True, random_ball=rb, random_goal=rg)
        ora = oracle_mod.OracleVec(ov, n, seed=8, autoreset=True, random_ball=rb, random_goal=rg)
        assert np.array_equal(u32(env.reset()), u32(ora.reset()))
        gen = torch.Generator().manual_seed(1)
        for t in range(60):
            a = torch.randint(0, 25, (n,), generator=gen)
            obs, rew, done, _ = env.step(a)
            o_ref, r_ref, d_ref = ora.step(a.numpy())
            assert np.array_equal(u32(rew), u32(r_ref)) and np.array_equal(done.cpu().numpy(), d_ref.astype(bool)), (variant, t)
            assert np.array_equal(u32(obs), u32(o_ref)), (variant, t)
        st = env.get_state().cpu().numpy()
        if not rb:
            assert ((st[:, 4] > 0) | ((st[:, 0] == 4) & (st[:, 1] == 4))).all()     # fresh episodes start on 'S'
        assert env.stats()["episodes"] > 0
        env.close()
    env = lmz.LmazeHierCuda(n, "v5", seed=8, autoreset=True, random_ball=rb, random_goal=rg)
    ora = oracle_mod.OracleHier(n, seed=8, random_ball=rb, random_goal=rg)
    assert np.array_equal(u32(env.reset()), u32(ora.reset()))
    rng = np.random.RandomState(2)
    mask = np.ones(n, np.uint8)
    for t in range(60):
        g = rng.randint(0, 25, size=n); a = rng.randint(0, 4, size=n)
        env.plannerStep(g, mask=mask); ora.planner_step(g, mask=mask)
        fov, loc, gr, lr, gd, ld, _, _ = env.step(a, goal_plane=False)
        fov_ref, loc_ref, gr_ref, lr_ref, gd_ref, ld_ref, err_ref = ora.step(a)
        gdm = gd_ref.astype(bool)
        if gdm.any():
            ora.reset(mask=gdm.astype(np.uint8), want_obs=False)
            ora.render(mask=gdm.astype(np.uint8), fov=fov_ref, loc=loc_ref)
        assert np.array_equal(u32(gr), u32(gr_ref)) and np.array_equal(u32(fov), u32(fov_ref)), t
        assert np.array_equal(u32(loc), u32(loc_ref)), t
        mask = (gd_ref | ld_ref).astype(np.uint8)
    st = env.get_state().cpu().numpy()
    if not rg:                                             # the goal is the maze's 'X' cell
        xs = {k: [(x, r.index("X")) for x, r in enumerate(oracle_mod.layout_v2(k)) if "X" in r][0] for k in range(1, 6)}
        assert all((st[i, 6], st[i, 7]) == xs[st[i, 15] >> 4] for i in range(n))
    env.close()


def test_hier_one_million_envs(lmz, oracle_mod):
    """Full size (2^20 envs, 57 GB of observations): two blocks of envs at both ends of the batch are replayed
    by the oracle from the same seeds (the device RNG is keyed by global env id), and size-independent
    properties hold over the whole batch."""
    N = 1 << 20
    need_free(N * 53900 + (6 << 30))
    seed, B = 4242, 384
    env = lmz.LmazeHierCuda(N, "v5", seed=seed, autoreset=True)
    blocks = [(0, oracle_mod.OracleHier(B, seed=seed, env_id0=0)), (N - B - 37, oracle_mod.OracleHier(B, seed=seed, env_id0=N - B - 37))]
    fov = env.reset()
    for lo, ora in blocks:
        assert np.array_equal(u32(fov[lo:lo + B]), u32(ora.reset()))
    gen = torch.Generator(device="cuda").manual_seed(5)
    masks = [np.ones(B, np.uint8) for _ in blocks]
    for t in range(12):
        goals = torch.randint(0, 25, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        acts = torch.randint(0, 4, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        env.plannerStep(goals, mask="auto")
        fov, loc, gr, lr, gd, ld, _, _ = env.step(acts, goal_plane=False)
        for k, (lo, ora) in enumerate(blocks):
            ora.planner_step(goals[lo:lo + B].cpu().numpy(), mask=masks[k])
            fov_ref, loc_ref, gr_ref, lr_ref, gd_ref, ld_ref, err_ref = ora.step(acts[lo:lo + B].cpu().numpy())
            gdm = gd_ref.astype(bool)
            if gdm.any():
                ora.reset(mask=gdm.astype(np.uint8), want_obs=False)
                ora.render(mask=gdm.astype(np.uint8), fov=fov_ref, loc=loc_ref)
            assert np.array_equal(u32(gr[lo:lo + B]), u32(gr_ref)) and np.array_equal(u32(lr[lo:lo + B]), u32(lr_ref)), (t, lo)
            assert np.array_equal(u32(fov[lo:lo + B]), u32(fov_ref)) and np.array_equal(u32(loc[lo:lo + B]), u32(loc_ref)), (t, lo)
            masks[k] = (gd_ref | ld_ref).astype(np.uint8)
    # whole batch: rewards are among the reference's constants; every 35x35 plane is a x7 replication; the
    # fovealGoal channel is one-hot; binary channels hold only 0 / 1
    allowed_g = torch.tensor([0x42C80000, 0xBC23D70A, 0xBF800000], dtype=torch.int64, device="cuda")
    assert torch.isin(gr.view(torch.int32).long() & 0xFFFFFFFF, allowed_g).all()
    CH = 1 << 15
    for lo in range(0, N, CH):
        f, l = fov[lo:lo + CH], loc[lo:lo + CH]
        small = f[:, :, ::7, ::7]
        assert torch.equal(small.repeat_interleave(7, 2).repeat_interleave(7, 3), f)
        assert torch.equal(l[:, :, ::7, ::7].repeat_interleave(7, 2).repeat_interleave(7, 3), l)
        assert (small[:, 3].sum(dim=(1, 2)) == 1).all() and (small[:, 0, 2, 2] == 1).all()      # goal plane one-hot; the ball's own cell is free
        binary = small[:, [0, 1, 3, 4, 5]]
        assert ((binary == 0) | (binary == 1)).all() and ((l == 0) | (l == 1)).all()
        ok = ~env.loc_err[lo:lo + CH]
        assert (l[ok][:, 3, ::7, ::7].sum(dim=(1, 2)) == 1).all() and (l[~ok].sum(dim=(1, 2, 3)) == 0).all()
    s = env.stats(check_errors=False)
    assert s["steps"] == 12 * N and s["wall_bumps"] + s["moves"] == 12 * N
    env.close()


def test_hier_shard_invariance_and_graph_replay(lmz):
    """Trajectories do not depend on how the batch is split over handles / GPUs, and a captured
    plannerStep(auto) + step pair replays correctly."""
    N, seed = 3000, 9
    whole = lmz.LmazeHierCuda(N, "v5", seed=seed, env_id0=0)
    lo, hi = lmz.shard_range(N, 1, 3)
    part = lmz.LmazeHierCuda(hi - lo, "v5", seed=seed, env_id0=lo)
    assert torch.equal(whole.reset()[lo:hi], part.reset())
    gen = torch.Generator(device="cuda").manual_seed(2)
    g_buf = torch.zeros(hi - lo, dtype=torch.uint8, device="cuda")
    a_buf = torch.zeros(hi - lo, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    part.plannerStep(g_buf, mask="auto"); part.step(a_buf, goal_plane=False)       # warm the launch paths ...
    part.set_state(whole.get_state()[lo:hi].clone()); part.set_visit(whole.get_visit()[lo:hi].clone())   # ... and rewind
    torch.cuda.synchronize()
    with torch.cuda.graph(graph):
        part.plannerStep(g_buf, mask="auto")
        part.step(a_buf, goal_plane=False)
    for t in range(40):
        g = torch.randint(0, 25, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        a = torch.randint(0, 4, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        whole.plannerStep(g, mask="auto"); whole.step(a, goal_plane=False)
        g_buf.copy_(g[lo:hi]); a_buf.copy_(a[lo:hi])
        graph.replay()
        assert torch.equal(whole.obs[lo:hi], part.obs) and torch.equal(whole.loc_obs[lo:hi], part.loc_obs), t
        assert torch.equal(whole.reward[lo:hi].view(torch.int32), part.reward.view(torch.int32)), t
    st_w, st_p = whole.get_state()[lo:hi], part.get_state()
    assert torch.equal(st_w, st_p) and torch.equal(whole.get_visit()[lo:hi], part.get_visit())
    whole.close(); part.close()


def test_foveal_compact_and_transition_only(lmz, oracle_mod):
    """obs_mode='compact' on the foveal variants: the f32 5x5 crops, whose x7 replication is exactly the reference
    image (every step, incl. v4's float visit planes and v5's two tensors); and the launch with no observation
    bound keeps the same trajectories."""
    n = 2500
    for variant, ov in (("v2", oracle_mod.V2), ("v4", oracle_mod.V4)):
        env = lmz.LmazeVecCuda(n, variant, seed=6, obs_mode="compact")
        bare = lmz.LmazeVecCuda(n, variant, seed=6, with_obs=False)
        ora = oracle_mod.OracleVec(ov, n, seed=6, autoreset=True)
        assert env.obs.shape == (n, env.full_obs_shape[0], 5, 5) and env.obs.dtype == torch.float32
        assert np.array_equal(u32(env.expand(env.reset())), u32(ora.reset()))
        bare.reset()
        gen = torch.Generator().manual_seed(4)
        for t in range(70):
            a = torch.randint(0, 25, (n,), generator=gen)
            obs, rew, done, _ = env.step(a)
            _, rew_b, done_b, _ = bare.step(a)
            o_ref, r_ref, d_ref = ora.step(a.numpy())
            assert np.array_equal(u32(rew), u32(r_ref)) and np.array_equal(done.cpu().numpy(), d_ref.astype(bool)), (variant, t)
            assert np.array_equal(u32(env.expand(obs)), u32(o_ref)), (variant, t)
            assert torch.equal(rew_b.view(torch.int32), rew.view(torch.int32)) and torch.equal(done_b, done), (variant, t)
        assert torch.equal(env.get_state(), bare.get_state())
        if variant == "v4":
            assert torch.equal(env.get_visit(), bare.get_visit())
            assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit()))
        assert [env.stats()[k] for k in oracle_mod.STAT_NAMES] == ora.stats.tolist()
        env.close(); bare.close()
    env = lmz.LmazeHierCuda(n, "v5", seed=6, obs_mode="compact")
    ora = oracle_mod.OracleHier(n, seed=6)
    assert env.obs.shape == (n, 7, 5, 5) and env.loc_obs.shape == (n, 4, 5, 5)
    assert np.array_equal(u32(env.expand(env.reset())), u32(ora.reset()))
    rng = np.random.RandomState(7)
    mask = np.ones(n, np.uint8)
    for t in range(70):
        g = rng.randint(0, 25, size=n); a = rng.randint(0, 4, size=n)
        loc = env.plannerStep(g, mask="auto" if t % 2 else mask)
        loc_ref, _ = ora.planner_step(g, mask=mask)
        m = mask.astype(bool)
        assert np.array_equal(u32(env.expand_local(loc))[m], u32(loc_ref)[m]), t
        fov, loc, gr, lr, gd, ld, _, _ = env.step(a, goal_plane=False)
        fov_ref, loc_ref, gr_ref, lr_ref, gd_ref, ld_ref, err_ref = ora.step(a)
        gdm = gd_ref.astype(bool)
        if gdm.any():
            ora.reset(mask=gdm.astype(np.uint8), want_obs=False)
            ora.render(mask=gdm.astype(np.uint8), fov=fov_ref, loc=loc_ref)
        assert np.array_equal(u32(gr), u32(gr_ref)) and np.array_equal(u32(lr), u32(lr_ref)), t
        assert np.array_equal(u32(env.expand(fov)), u32(fov_ref)), t
        assert np.array_equal(u32(env.expand_local(loc)), u32(loc_ref)), t
        mask = (gd_ref | ld_ref).astype(np.uint8)
    assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit()))
    env.close()


def test_hier_out_of_range_inputs_are_counted(lmz, oracle_mod):
    """plannerStep goals outside 0..24 raise IndexError in the reference (lmaze_env_v5.py:168); the batched API
    clamps them and bumps the error counter, exactly like the oracle's batched driver.  Step actions outside 0..3
    are legal no-moves (:203-217)."""
    n = 256
    env = lmz.LmazeHierCuda(n, "v5", seed=2, autoreset=False)
    ora = oracle_mod.OracleHier(n, seed=2)
    env.reset(); ora.reset()
    goals = np.arange(n, dtype=np.int64) - 100            # -100 .. 155
    loc = env.plannerStep(torch.as_tensor(goals))
    loc_ref, _ = ora.planner_step(goals)
    assert np.array_equal(u32(loc), u32(loc_ref))
    bad = int(((goals < 0) | (goals > 24)).sum())
    with pytest.raises(ValueError):
        env.stats()
    acts = np.arange(n, dtype=np.int64) - 50
    fov, loc, gr, lr, gd, ld, _, _ = env.step(torch.as_tensor(acts), goal_plane=False)
    fov_ref, loc_ref, gr_ref, lr_ref, gd_ref, ld_ref, err_ref = ora.step(acts)
    assert np.array_equal(u32(fov), u32(fov_ref)) and np.array_equal(u32(loc), u32(loc_ref))
    assert np.array_equal(u32(gr), u32(gr_ref)) and np.array_equal(u32(lr), u32(lr_ref))
    import ctypes
    from gym_lmaze_b200 import _abi
    out = (ctypes.c_int64 * _abi.NUM_STATS)(); err = ctypes.c_int64()
    _abi.check(env._lib.lmz_stats(env._h, ctypes.byref(out), ctypes.byref(err), env._stream()))
    assert err.value == bad + int(err_ref.sum())
    env.close()
