"""GPU tier: the persistent and grid-stride kernels at batch sizes where every resident warp or thread handles SEVERAL
work units.  The pipelining of these kernels (a tile's state words, actions and visit histories loaded one tile ahead,
refilled input buffers, double-buffered value planes, tiles grabbed ahead from a work counter, a rollout thread's
second and later envs) only runs from a worker's second unit on; at the sizes of the other parity tests every worker
gets at most one.

Sizing rule: R = SMs x 2048 is the most threads the device holds resident (64 warps per SM); the multi-tile tests use
N = 2R + 21 (606,229 envs on a 148-SM B200), so that at any occupancy every resident warp or thread gets at least two
units on average, the last tile is partial and the tile count is odd.  Everything is compared bit for bit with the
CPU oracle (whole batch where it fits, 1,024-env blocks replayed from reset with the same global ids otherwise) or
with a second handle whose kernel the oracle checks."""
import os

import numpy as np
import pytest
import torch

from oracle.oracle import STAT_NAMES
from philox_np import ActionStream, rng_hier

pytestmark = pytest.mark.gpu

RC_BITS = np.array([0x80000000, 0xBF800000, 0xBC23D70A, 0x42C80000], dtype=np.uint32).view(np.int32)
THREADS = os.cpu_count() or 1
CH = 1 << 14                                   # rows per chunk of the whole-tensor checks on the device


@pytest.fixture(scope="module")
def lmz():
    import gym_lmaze_b200 as g
    from gym_lmaze_b200 import _abi
    _abi.load()
    assert torch.cuda.is_available()
    return g


def u32(t):
    return (t.detach().cpu().numpy() if torch.is_tensor(t) else t).view(np.uint32)


def i32(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _need(nbytes):
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    free_b = torch.cuda.mem_get_info()[0]
    if free_b < nbytes:
        pytest.fail("B200 expected: %d GiB free, need %d GiB" % (free_b >> 30, nbytes >> 30))


def _resident():
    return torch.cuda.get_device_properties(0).multi_processor_count * 2048


def _multi(k=2, tail=21):
    R = _resident()
    N = k * R + tail
    assert N >= k * R
    return N


def _rows(N, seed):
    """The first tile, a middle tile, the last (partial) tile and 512 random rows."""
    mid = (N // 64) * 32
    rng = np.random.RandomState(seed)
    return np.unique(np.concatenate([np.arange(32), np.arange(mid, mid + 32), np.arange((N - 1) // 32 * 32, N),
                                     rng.randint(0, N, 512)]))


def _check(rew, done, r_ref, d_ref, what):
    assert np.array_equal(u32(rew), r_ref.view(np.uint32)), what
    assert np.array_equal(done.detach().cpu().numpy().view(np.uint8), d_ref), what


def _oracle(O, variant, n, **kw):
    ora = O.OracleVec(variant, n, threads=THREADS, lazy_init=True, **kw)
    ora.reset(want_obs=False)
    return ora


def _sampled(ora, rows):
    return torch.from_numpy(np.stack([ora.render_one(int(i)) for i in rows]))


def _expand_equal(comp, full_obs, expand):
    """expand(compact rows) == the full render, every row, on the device."""
    for lo in range(0, full_obs.shape[0], CH):
        assert torch.equal(i32(expand(comp[lo:lo + CH])), i32(full_obs[lo:lo + CH])), lo


def _end_state(env, ora, variant, past_limit=False):
    """Final state words, goal counts, episode counters and statistics.  past_limit: envs stepped far past their step
    limit without a reset; the foveal state word keeps the step counter in 6 bits, saturating at 63 (its episode-length
    statistic counts the saturated value), so those two are compared as saturated / left out."""
    st = env.get_state().cpu().numpy()
    pos, sc, gc, _ = ora.export()
    if variant == "v0":
        assert np.array_equal(st[:, 0:2], pos[:, 0:2]) and np.array_equal(st[:, 6], gc)
    else:
        assert np.array_equal(st[:, 0:4], pos)
    assert np.array_equal(st[:, 4], np.minimum(sc, 63) if past_limit else sc)
    assert np.array_equal(st[:, 7], ora.episode)
    s = env.stats(check_errors=False)
    names = [k for k in STAT_NAMES if not (past_limit and k == "eplen_sum")]
    assert [s[k] for k in names] == [int(ora.stats[STAT_NAMES.index(k)]) for k in names]


def _foveal_properties(obs, variant):
    """Every row of a full foveal render: 7x7-block replication of a 5x5 crop, binary planes binary, the goal / ball /
    previous-crop planes hold at most one hot cell, visit planes in [0, 1]."""
    vis = [2, 6] if variant in ("v4", "v5") else []
    binary = [c for c in range(obs.shape[1]) if c not in vis]
    hot = [1, 2, 4] if variant == "v2" else [1, 3, 5]
    for lo in range(0, obs.shape[0], CH):
        o = obs[lo:lo + CH]
        small = o[:, :, ::7, ::7]
        assert torch.equal(small.repeat_interleave(7, 2).repeat_interleave(7, 3), o), lo
        b = small[:, binary]
        assert ((b == 0) | (b == 1)).all(), lo
        assert (small[:, hot].sum(dim=(2, 3)) <= 1).all(), lo
        if vis:
            assert (small[:, vis] >= 0).all() and (small[:, vis] <= 1).all(), lo


# ---------------------------------------------------------------- 1. v0 / v3 compact family and incremental render
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_compact_bits_transition_incremental_multitile(lmz, oracle_mod, variant):
    """lmz_env_compact_kernel (compact, bits, transition-only) and lmz_env_incr_kernel, stepped with the same actions
    for 130 steps past the 101-step episode limit (auto-resets de-synchronise the envs) against one whole-batch
    oracle: reward bits and done flags of every env every step, sampled observation rows every 10th step, the final
    state words, goal counts, episode counters and statistics."""
    O = oracle_mod
    N, T, seed, id0 = _multi(), 130, 41, 7
    ov = O.V0 if variant == "v0" else O.V3
    _need(N * 4 * int(np.prod(O.OBS_SHAPE[ov])) + (8 << 30))
    ora = _oracle(O, ov, N, seed=seed, env_id0=id0)

    def mk(**kw):
        return lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0, autoreset=True, **kw)
    envs = {"compact": mk(obs_mode="compact"), "bits": mk(obs_mode="bits"), "transition": mk(with_obs=False),
            "incremental": mk(render_mode="incremental")}
    for e in envs.values():
        e.reset()
    rows = _rows(N, 1)
    rows_d = torch.as_tensor(rows, device="cuda")
    gen = torch.Generator().manual_seed(11)
    for t in range(T):
        a = torch.randint(0, 5, (N,), generator=gen)           # 4: the reference's unmatched action
        _, r_ref, d_ref = ora.step(a.numpy(), want_obs=False)
        a_d = a.to("cuda", torch.uint8)
        for name, e in envs.items():
            _, rew, done, _ = e.step(a_d)
            _check(rew, done, r_ref, d_ref, (name, t))
        if t % 10 == 9 or t == T - 1:
            want = _sampled(ora, rows)
            for name in ("compact", "bits", "incremental"):
                e = envs[name]
                assert torch.equal(e.expand(e.obs[rows_d]).cpu(), want), (name, t)
    assert ora.episode.min() >= 2
    for e in envs.values():
        _end_state(e, ora, variant)
    # the incremental tensor, every row: ball (and goal) blocks where the state says, the static channels
    env = envs["incremental"]
    obs, st = env.obs, env.get_state()
    for lo in range(0, N, CH):
        o, s = obs[lo:lo + CH], st[lo:lo + CH]
        idx = torch.arange(o.shape[0], device="cuda")
        x, y = s[:, 0].long(), s[:, 1].long()
        if variant == "v0":
            assert torch.equal(o.sum(dim=(2, 3)), torch.tensor([49.0, 3528.0, 49.0, 3430.0], device="cuda").expand(o.shape[0], 4))
            assert (o[idx, 0, 7 * x, 7 * y] == 1).all() and (o[idx, 0, 7 * x + 6, 7 * y + 6] == 1).all()
            assert torch.equal(o[:, 1:], obs[0:1, 1:].expand(o.shape[0], 3, 84, 84)), lo
        else:
            assert torch.equal(o.sum(dim=(2, 3)), torch.tensor([73 * 16.0, 16.0, 16.0], device="cuda").expand(o.shape[0], 3))
            assert (o[idx, 1, 4 * x, 4 * y] == 1).all()
            assert (o[idx, 2, 4 * s[:, 2].long() + 3, 4 * s[:, 3].long() + 3] == 1).all()
            assert torch.equal(o[:, 0], obs[0:1, 0].expand(o.shape[0], 72, 72)), lo
    for e in envs.values():
        e.close()


# ---------------------------------------------------------------- 2. v2 / v4 foveal step kernels
@pytest.mark.parametrize("variant", ["v2", "v4"])
def test_foveal_step_kernels_multitile(lmz, oracle_mod, variant):
    """lmz_fov_small_kernel (compact) and lmz_env_fov_kernel (full render) stepped with the same actions for 130 steps
    (STEP_LIMIT 50: every env resets at least twice, history lengths spread over 0..51 in every warp): reward bits and
    done flags of every env against the oracle, expand(compact) == full for every row every step, sampled rows
    against the oracle's render every 10 steps.  v4: the whole visit layer at checkpoints, and from step 60 on a mix of
    direct-mode lanes (set_visit(get_visit()) puts every env in direct mode until its next reset) and history lanes."""
    O = oracle_mod
    N, T, seed, id0 = _multi(), 130, 23, 1000
    ov = O.V2 if variant == "v2" else O.V4
    _need(2 * N * 4 * int(np.prod(O.OBS_SHAPE[ov])) + (8 << 30))
    ora = _oracle(O, ov, N, seed=seed, env_id0=id0)
    full = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0)
    comp = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0, obs_mode="compact")
    full.reset(); comp.reset()
    rows = _rows(N, 2)
    rows_d = torch.as_tensor(rows, device="cuda")
    gen = torch.Generator().manual_seed(12)
    for t in range(T):
        a = torch.randint(0, 25, (N,), generator=gen)
        _, r_ref, d_ref = ora.step(a.numpy(), want_obs=False)
        a_d = a.to("cuda", torch.uint8)
        for name, e in (("full", full), ("compact", comp)):
            _, rew, done, _ = e.step(a_d)
            _check(rew, done, r_ref, d_ref, (name, t))
        _expand_equal(comp.obs, full.obs, comp.expand)
        if t % 10 == 9 or t == T - 1:
            assert np.array_equal(u32(full.obs[rows_d]), u32(_sampled(ora, rows))), t
        if variant == "v4" and t in (9, 59, 64, 99, T - 1):
            vref = u32(ora.export_visit())
            assert np.array_equal(u32(full.get_visit()), vref), t
            assert np.array_equal(u32(comp.get_visit()), vref), t
        if variant == "v4" and t == 60:
            for e in (full, comp):
                e.set_visit(e.get_visit())
    assert ora.episode.min() >= 3
    for e in (full, comp):
        _end_state(e, ora, variant)
    _foveal_properties(full.obs, variant)
    full.close(); comp.close()


def test_v4_masked_reset_mixes_history_lengths(lmz, oracle_mod):
    """autoreset off, a masked reset of a random 40 % at step 35, 80 steps: the envs that were not reset cross 64
    history entries (the warp-cooperative materialisation) inside tiles whose other lanes are still in history mode."""
    O = oracle_mod
    N, T, seed, id0 = _multi(), 80, 31, 0
    _need(2 * N * 34300 + (8 << 30))
    ora = _oracle(O, O.V4, N, seed=seed, env_id0=id0, autoreset=False)
    full = lmz.LmazeVecCuda(N, "v4", seed=seed, env_id0=id0, autoreset=False)
    comp = lmz.LmazeVecCuda(N, "v4", seed=seed, env_id0=id0, autoreset=False, obs_mode="compact")
    full.reset(); comp.reset()
    rows = _rows(N, 3)
    rows_d = torch.as_tensor(rows, device="cuda")
    gen = torch.Generator().manual_seed(13)
    for t in range(T):
        if t == 35:
            mask = torch.rand(N, generator=gen) < 0.4
            ora.reset_masked(mask.numpy())
            for e in (full, comp):
                e.reset(mask=mask)
        a = torch.randint(0, 25, (N,), generator=gen)
        _, r_ref, d_ref = ora.step(a.numpy(), want_obs=False)
        a_d = a.to("cuda", torch.uint8)
        for name, e in (("full", full), ("compact", comp)):
            _, rew, done, _ = e.step(a_d)
            _check(rew, done, r_ref, d_ref, (name, t))
        _expand_equal(comp.obs, full.obs, comp.expand)
        if t in (34, 62, 63, 64, 65, 66, T - 1):
            vref = u32(ora.export_visit())
            assert np.array_equal(u32(full.get_visit()), vref), t
            assert np.array_equal(u32(comp.get_visit()), vref), t
    assert np.array_equal(u32(full.obs[rows_d]), u32(_sampled(ora, rows)))
    for e in (full, comp):
        _end_state(e, ora, "v4", past_limit=True)
    full.close(); comp.close()


# ---------------------------------------------------------------- 3. v5: planner + actor, compact against full
def _hier_blocks(O, N, seed, B=1024):
    los = [0, N // 2 - B // 2 + 5, N - B]
    return [(lo, O.OracleHier(B, seed=seed, env_id0=lo)) for lo in los]


def _hier_oracle_step(ora, goals, acts):
    """plannerStep for the envs waiting for their planner, step, the framework's same-step reset."""
    st = ora.export()
    need = (((st[:, 15] >> 1) & 1) | (st[:, 14] == 0)).astype(np.uint8)
    if need.any():
        ora.planner_step(goals, mask=need)
    f, l, gr, lr, gd, ld, err = ora.step(acts)
    if gd.any():
        ora.reset(mask=gd, want_obs=False)
        ora.render(mask=gd, fov=f, loc=l)
        err[gd.astype(bool)] = 0
    return f, l, gr, lr, gd, ld, err


def test_v5_compact_and_full_multitile(lmz, oracle_mod):
    """130 steps of plannerStep(mask="auto") + step with autoreset: the full twin (lmz_planner_kernel +
    lmz_env_fov_kernel<V5>) against the compact handle (lmz_fov_small_kernel in both modes) over the whole batch every
    step, and three 1,024-env oracle blocks (the first, a middle one, the one ending at the last env) every step."""
    O = oracle_mod
    N, T, seed = _multi(), 130, 19
    _need(N * (34300 + 19600) + (8 << 30))
    full = lmz.LmazeHierCuda(N, "v5", seed=seed, autoreset=True)
    comp = lmz.LmazeHierCuda(N, "v5", seed=seed, autoreset=True, obs_mode="compact")
    f0 = full.reset(); comp.reset()
    _expand_equal(comp.obs, full.obs, comp.expand)
    blocks = _hier_blocks(O, N, seed)
    for lo, ora in blocks:
        assert np.array_equal(u32(f0[lo:lo + ora.n]), u32(ora.reset()))
    gen = torch.Generator(device="cuda").manual_seed(14)
    n_reset = 0
    for t in range(T):
        goals = torch.randint(0, 25, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        acts = torch.randint(0, 4, (N,), generator=gen, device="cuda", dtype=torch.uint8)
        for e in (full, comp):
            e.plannerStep(goals, mask="auto")
            e.step(acts, goal_plane=False)
        _expand_equal(comp.obs, full.obs, comp.expand)
        _expand_equal(comp.loc_obs, full.loc_obs, comp.expand_local)
        for k in ("reward", "local_reward", "_done_u8", "_ldone_u8", "_loc_err_u8", "foveal_goal"):
            assert torch.equal(i32(getattr(comp, k)), i32(getattr(full, k))), (k, t)
        g_h, a_h = goals.cpu().numpy().astype(np.int64), acts.cpu().numpy().astype(np.int64)
        for lo, ora in blocks:
            B = ora.n
            f, l, gr, lr, gd, ld, err = _hier_oracle_step(ora, g_h[lo:lo + B], a_h[lo:lo + B])
            n_reset += int(gd.sum())
            assert np.array_equal(u32(full.reward[lo:lo + B]), gr.view(np.uint32)), (lo, t)
            assert np.array_equal(u32(full.local_reward[lo:lo + B]), lr.view(np.uint32)), (lo, t)
            assert np.array_equal(full._done_u8[lo:lo + B].cpu().numpy(), gd), (lo, t)
            assert np.array_equal(full._ldone_u8[lo:lo + B].cpu().numpy(), ld), (lo, t)
            assert np.array_equal(full._loc_err_u8[lo:lo + B].cpu().numpy(), err), (lo, t)
            assert np.array_equal(u32(full.obs[lo:lo + B]), u32(f)), (lo, t)
            assert np.array_equal(u32(full.loc_obs[lo:lo + B]), u32(l)), (lo, t)
        if t in (49, 99, T - 1):
            assert torch.equal(comp.get_state(), full.get_state()), t
            assert torch.equal(i32(comp.get_visit()), i32(full.get_visit())), t
    assert n_reset > 0
    for lo, ora in blocks:
        assert np.array_equal(u32(full.get_visit()[lo:lo + ora.n]), u32(ora.export_visit())), lo
    sf, sc = full.stats(check_errors=False), comp.stats(check_errors=False)
    assert sf == sc and sf["steps"] == T * N
    _foveal_properties(full.obs, "v5")
    full.close(); comp.close()


# ---------------------------------------------------------------- 4. every CTA shape tune= selects
def _lockstep(mk, variant, T, seed_gen):
    """A default-configured handle and a tuned one from reset, T steps with the same inputs, bit for bit."""
    hier = variant == "v5"
    ref, tun = mk(None), mk(True)
    o1, o2 = ref.reset(), tun.reset()
    if o1 is not None:
        assert torch.equal(i32(o1), i32(o2))
    gen = torch.Generator(device="cuda").manual_seed(seed_gen)
    na = 4 if hier else ref.num_actions
    for t in range(T):
        a = torch.randint(0, na + (0 if hier else 1), (ref.num_envs,), generator=gen, device="cuda", dtype=torch.uint8)
        if variant in ("v2", "v4"):
            a = a.clamp_(max=24)
        if hier:
            g = torch.randint(0, 25, (ref.num_envs,), generator=gen, device="cuda", dtype=torch.uint8)
            for e in (ref, tun):
                e.plannerStep(g, mask="auto")
                e.step(a, goal_plane=False)
            names = ("obs", "loc_obs", "reward", "local_reward", "_done_u8", "_ldone_u8", "_loc_err_u8", "foveal_goal")
        else:
            for e in (ref, tun):
                e.step(a)
            names = ("obs", "reward", "_done_u8")
        for k in names:
            x, y = getattr(ref, k), getattr(tun, k)
            if x is not None:
                assert torch.equal(i32(x), i32(y)), (k, t)
    assert torch.equal(ref.get_state(), tun.get_state())
    if variant in ("v4", "v5"):
        assert torch.equal(i32(ref.get_visit()), i32(tun.get_visit()))
    assert ref.stats(check_errors=False) == tun.stats(check_errors=False)
    ref.close(); tun.close()


def _mk(lmz, variant, N, tune, **kw):
    def mk(tuned):
        t = tune if tuned else None
        if variant == "v5":
            return lmz.LmazeHierCuda(N, "v5", seed=3, env_id0=11, tune=t, **kw)
        return lmz.LmazeVecCuda(N, variant, seed=3, env_id0=11, tune=t, **kw)
    return mk


@pytest.mark.parametrize("variant", ["v2", "v4", "v5"])
def test_full_foveal_kernel_every_cta_size(lmz, variant):
    """lmz_env_fov_kernel at every tune[0] the library builds besides the default 128 threads, R + 21 envs, 60 steps,
    against the default handle (which the tests above check against the oracle)."""
    N = _multi(k=1)
    _need(2 * N * (34300 + 19600) + (8 << 30))
    for thr in (160, 192, 224, 256, 512, 1024):
        _lockstep(_mk(lmz, variant, N, (thr, 0, 0, 0)), variant, 60, thr)


@pytest.mark.parametrize("variant", ["v2", "v4", "v5"])
def test_compact_foveal_kernel_every_cta_shape(lmz, variant):
    """lmz_fov_small_kernel with 2 and 8 warps per CTA, one and two CTAs per SM (tune[2] = 1 also makes every warp
    work through many more tiles)."""
    N = _multi(k=1)
    _need(8 << 30)
    for thr in (64, 256):
        for cap in (1, 2):
            _lockstep(_mk(lmz, variant, N, (thr, 0, cap, 0), obs_mode="compact"), variant, 60, thr + cap)


@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_compact_and_incremental_cta_caps(lmz, variant):
    """tune[2] (CTAs per SM) on the compact / transition-only launch and on the incremental render."""
    N = _multi(k=1)
    _need(2 * N * 112896 + (8 << 30))
    for kw in (dict(obs_mode="compact"), dict(with_obs=False), dict(render_mode="incremental")):
        for cap in (1, 2):
            _lockstep(_mk(lmz, variant, N, (0, 0, cap, 0), **kw), variant, 60, cap)


# ---------------------------------------------------------------- 5. grid-stride rollouts
def _rollout_against_oracle(env, ora, ids, seed, kind, n_dev_steps, buf_T, codes_T):
    """Philox rollouts of lengths n_dev_steps (t0 carried over), one caller-supplied [T, N] action buffer and one
    reward_codes=True rollout, every step's whole-batch rewards and dones against the oracle."""
    stream = ActionStream(seed, ids, kind)
    N = len(ids)
    table = env.reward_table("cuda")
    tg = 0
    for Tk in n_dev_steps:
        rew, done = env.rollout(Tk)
        rew_h, done_h = u32(rew), done.cpu().numpy().view(np.uint8)
        for t in range(Tk):
            _, r_ref, d_ref = ora.step(stream(tg + t), want_obs=False)
            assert np.array_equal(rew_h[t], r_ref.view(np.uint32)), (Tk, t)
            assert np.array_equal(done_h[t], d_ref), (Tk, t)
        tg += Tk
    gen = torch.Generator().manual_seed(5)
    acts = torch.randint(0, kind + 1, (buf_T, N), generator=gen, dtype=torch.uint8)
    if kind == 25:
        acts.clamp_(max=24)
    rew, done = env.rollout(buf_T, actions=acts.cuda())
    for t in range(buf_T):
        _, r_ref, d_ref = ora.step(acts[t].numpy().astype(np.int64), want_obs=False)
        _check(rew[t], done[t], r_ref, d_ref, ("buffer", t))
    tg += buf_T                                               # the device stream's t0 counts every rolled-out step
    codes, done = env.rollout(codes_T, reward_codes=True)
    rew = table[codes.long()]
    for t in range(codes_T):
        _, r_ref, d_ref = ora.step(stream(tg + t), want_obs=False)
        _check(rew[t], done[t], r_ref, d_ref, ("codes", t))


@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_rollout_kernel_several_envs_per_thread(lmz, oracle_mod, variant):
    """lmz_rollout_kernel at N = 3R + 5 (3-4 envs per resident thread), env ids crossing 2^32 inside the batch and a
    seed with a non-zero high word: rollouts of T = 64, 1, 17, 50 (t0 crosses the 64-step Philox blocks, T not a
    multiple of 16), a caller-supplied action buffer, reward codes; final state, statistics and sampled renders."""
    O = oracle_mod
    N = _multi(k=3, tail=5)
    seed, id0 = (5 << 32) + 77, (1 << 32) - 100_003
    ov = O.V0 if variant == "v0" else O.V3
    _need(4 << 30)
    ora = _oracle(O, ov, N, seed=seed, env_id0=id0)
    env = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0, obs_mode="compact")
    env.reset()
    ids = np.arange(N, dtype=np.uint64) + np.uint64(id0)
    _rollout_against_oracle(env, ora, ids, seed, 4, (64, 1, 17, 50), 12, 12)
    _end_state(env, ora, variant)
    rows = _rows(N, 4)
    assert torch.equal(env.expand(env.render_obs()[torch.as_tensor(rows, device="cuda")]).cpu(), _sampled(ora, rows))
    env.close()


@pytest.mark.parametrize("variant", ["v2", "v4"])
def test_foveal_rollout_kernel_several_envs_per_thread(lmz, oracle_mod, variant):
    """lmz_fov_rollout_kernel at N = 2R + 21: each thread reloads and stores back the visit history of every env it
    takes.  Rollouts of T = 30, 1, 17, 20 (t0 inside a 4-step Philox block), an action buffer, reward codes; the whole
    v4 visit layer, final state and sampled renders against the oracle."""
    O = oracle_mod
    N = _multi()
    seed, id0 = (3 << 32) + 9, (1 << 32) - 300_001
    ov = O.V2 if variant == "v2" else O.V4
    _need(4 << 30)
    ora = _oracle(O, ov, N, seed=seed, env_id0=id0)
    env = lmz.LmazeVecCuda(N, variant, seed=seed, env_id0=id0, obs_mode="compact")
    env.reset()
    ids = np.arange(N, dtype=np.uint64) + np.uint64(id0)
    _rollout_against_oracle(env, ora, ids, seed, 25, (30, 1, 17, 20), 8, 8)
    _end_state(env, ora, variant)
    if variant == "v4":
        assert np.array_equal(u32(env.get_visit()), u32(ora.export_visit()))
    rows = _rows(N, 5)
    assert np.array_equal(u32(env.expand(env.render_obs()[torch.as_tensor(rows, device="cuda")])), u32(_sampled(ora, rows)))
    env.close()


def test_hier_rollout_several_envs_per_thread(lmz, oracle_mod):
    """lmz_hier_rollout at N = 2R + 21 with device Philox goals / actions: three 1,024-env oracle blocks driven by the
    numpy twin, and the whole batch against a compact handle stepped through plannerStep(mask="auto") + step with
    the same goals and actions; then a rollout with caller-supplied goals= / actions= buffers against the same."""
    O = oracle_mod
    N, seed = _multi(), 21
    _need(8 << 30)
    roll = lmz.LmazeHierCuda(N, "v5", seed=seed, obs_mode="compact")
    step = lmz.LmazeHierCuda(N, "v5", seed=seed, obs_mode="compact")
    roll.reset(); step.reset()
    blocks = _hier_blocks(O, N, seed)
    for _, ora in blocks:
        ora.reset(want_obs=False)
    ids = np.arange(N, dtype=np.uint64)
    tg = 0
    for Tk in (20, 1, 13):
        gr, lr, gd, ld = roll.rollout(Tk)
        for t in range(Tk):
            g, a = rng_hier(seed, ids, tg + t)
            step.plannerStep(torch.as_tensor(g, device="cuda"), mask="auto")
            step.step(torch.as_tensor(a, device="cuda"), goal_plane=False)
            for x, y in ((gr[t], step.reward), (lr[t], step.local_reward), (gd[t], step.done), (ld[t], step.local_done)):
                assert torch.equal(i32(x), i32(y)), (Tk, t)
            for lo, ora in blocks:
                B = ora.n
                _, _, gr_r, lr_r, gd_r, ld_r, _ = _hier_oracle_step(ora, g[lo:lo + B], a[lo:lo + B])
                assert np.array_equal(u32(gr[t, lo:lo + B]), gr_r.view(np.uint32)), (lo, Tk, t)
                assert np.array_equal(u32(lr[t, lo:lo + B]), lr_r.view(np.uint32)), (lo, Tk, t)
                assert np.array_equal(gd[t, lo:lo + B].cpu().numpy(), gd_r.astype(bool)), (lo, Tk, t)
                assert np.array_equal(ld[t, lo:lo + B].cpu().numpy(), ld_r.astype(bool)), (lo, Tk, t)
        tg += Tk
    T = 16
    gen = torch.Generator(device="cuda").manual_seed(6)
    goals = torch.randint(0, 25, (T, N), generator=gen, device="cuda", dtype=torch.uint8)
    acts = torch.randint(0, 5, (T, N), generator=gen, device="cuda", dtype=torch.uint8)     # 4: no move
    gr, lr, gd, ld = roll.rollout(T, goals=goals, actions=acts)
    for t in range(T):
        step.plannerStep(goals[t], mask="auto")
        step.step(acts[t], goal_plane=False)
        for x, y in ((gr[t], step.reward), (lr[t], step.local_reward), (gd[t], step.done), (ld[t], step.local_done)):
            assert torch.equal(i32(x), i32(y)), ("buffer", t)
    st_r, st_s = roll.get_state(), step.get_state()
    assert torch.equal(st_r[:, :13], st_s[:, :13]) and torch.equal(st_r[:, 15:], st_s[:, 15:])
    assert torch.equal(st_r[:, 13:15].clamp(max=255), st_s[:, 13:15].clamp(max=255))
    assert torch.equal(i32(roll.get_visit()), i32(step.get_visit()))
    sr, ss = roll.stats(check_errors=False), step.stats(check_errors=False)
    assert sr["steps"] == ss["steps"] == (34 + T) * N and sr["episodes"] == ss["episodes"]
    roll.close(); step.close()


# ---------------------------------------------------------------- 6. the sizes the bench quotes
BENCH_SIZES = [("v2", "full", 1 << 22, 701_300), ("v4", "full", 1 << 21, 500_900), ("v4", "compact", 1 << 23, 6_627_990),
               ("v5", "compact", 1 << 23, 7_777_777), ("v0", "bits", 1 << 24, 16_000_001)]


@pytest.mark.parametrize("variant,obs_mode,N,LO", BENCH_SIZES, ids=["v2-full-4M", "v4-full-2M", "v4-compact-8M",
                                                                   "v5-compact-8M", "v0-bits-16M"])
def test_bench_sizes(lmz, oracle_mod, variant, obs_mode, N, LO):
    """The batch sizes bench.py quotes, 120 steps: a 1,024-env oracle block replayed from reset, compared every step
    (the full-render blocks start past float index 2^32 of the observation tensor; the v4 compact block straddles
    the env where the visit layer's offset passes 2^31 floats, and from step 100 on runs in direct mode), then
    per-row properties of every env."""
    O = oracle_mod
    T, B, seed = 120, 1024, 2026
    hier = variant == "v5"
    per_env = {"v2": 24500, "v4": 34300}.get(variant, 0) if obs_mode == "full" else 2048
    _need(N * (per_env + 2048) + (8 << 30))
    if hier:
        env = lmz.LmazeHierCuda(N, "v5", seed=seed, obs_mode=obs_mode)
        ora = O.OracleHier(B, seed=seed, env_id0=LO)
    else:
        env = lmz.LmazeVecCuda(N, variant, seed=seed, obs_mode=obs_mode)
        ora = O.OracleVec({"v0": O.V0, "v2": O.V2, "v4": O.V4}[variant], B, seed=seed, env_id0=LO)
    env.reset(); ora.reset(want_obs=False)
    sl = slice(LO, LO + B)
    gen = torch.Generator(device="cuda").manual_seed(7)
    for t in range(T):
        if hier:
            goals = torch.randint(0, 25, (N,), generator=gen, device="cuda", dtype=torch.uint8)
            acts = torch.randint(0, 4, (N,), generator=gen, device="cuda", dtype=torch.uint8)
            env.plannerStep(goals, mask="auto")
            env.step(acts, goal_plane=False)
            f, l, gr, lr, gd, ld, err = _hier_oracle_step(ora, goals[sl].cpu().numpy().astype(np.int64),
                                                          acts[sl].cpu().numpy().astype(np.int64))
            assert np.array_equal(u32(env.reward[sl]), gr.view(np.uint32)) and np.array_equal(u32(env.local_reward[sl]), lr.view(np.uint32)), t
            assert np.array_equal(env._done_u8[sl].cpu().numpy(), gd) and np.array_equal(env._ldone_u8[sl].cpu().numpy(), ld), t
            assert np.array_equal(u32(env.expand(env.obs[sl])), u32(f)), t
            assert np.array_equal(u32(env.expand_local(env.loc_obs[sl])), u32(l)), t
        else:
            a = torch.randint(0, env.num_actions, (N,), generator=gen, device="cuda", dtype=torch.uint8)
            obs, rew, done, _ = env.step(a)
            o_ref, r_ref, d_ref = ora.step(a[sl].cpu().numpy().astype(np.int64))
            _check(rew[sl], done[sl], r_ref, d_ref, t)
            assert np.array_equal(u32(env.expand(obs[sl])), u32(o_ref)), t
        if variant == "v4" and obs_mode == "compact" and t == 99:
            assert np.array_equal(u32(env.get_visit()[sl]), u32(ora.export_visit()))
            env.set_visit(env.get_visit())
    if variant in ("v4", "v5"):
        assert np.array_equal(u32(env.get_visit()[sl]), u32(ora.export_visit()))
    assert int(ora.episode.min()) >= (1 if hier else 2) and int(ora.episode.max()) >= 2
    # every row
    allowed = torch.as_tensor(RC_BITS).cuda()
    assert torch.isin(env.reward.view(torch.int32), allowed).all()
    if hier:
        assert torch.isin(env.local_reward.view(torch.int32), allowed).all()
    if obs_mode == "full":
        _foveal_properties(env.obs, variant)
    elif variant == "v0":
        for lo in range(0, N, CH):
            c = env.unpack_bits(env.obs[lo:lo + CH])
            assert torch.equal(c.sum(dim=(2, 3)).int(), torch.tensor([1, 72, 1, 70], device="cuda", dtype=torch.int32).expand(c.shape[0], 4))
    else:
        for lo in range(0, N, CH):
            o = env.obs[lo:lo + CH]
            vis = [2, 6]
            binary = [c for c in range(o.shape[1]) if c not in vis]
            assert ((o[:, binary] == 0) | (o[:, binary] == 1)).all() and (o[:, vis] >= 0).all() and (o[:, vis] <= 1).all()
            if hier:
                assert torch.equal(o[:, 3].sum(dim=(1, 2)), torch.ones(o.shape[0], device="cuda"))
    if variant in ("v4", "v5"):
        vis_all = env.get_visit()
        assert (vis_all >= 0).all() and (vis_all <= 1).all()
        del vis_all
    s = env.stats(check_errors=False)
    assert s["steps"] == N * T and s["episodes"] > 0
    env.close()
