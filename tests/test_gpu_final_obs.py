"""GPU tier: final observations under auto-reset (lmz_bind_final, LmazeVecCuda(final_obs=True)).

The row an env ends its episode in is compared bit for bit with the CPU oracle stepped WITHOUT autoreset (its
observation after the terminal step), then re-spawned with the device-RNG reset the kernel's auto-reset uses.  A twin
handle without a final buffer shows that binding one changes nothing else."""
import ctypes
import os

import numpy as np
import pytest
import torch

from gpu_helpers import lmz, same_bytes

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1
FULL_VIEW = ("v0", "v3")
STEP_LIMIT_STEPS = {"v0": 100, "v3": 101, "v2": 51, "v4": 51}       # the step whose done flag ends a no-goal episode
NO_MOVE = {"v0": 7, "v3": 7, "v2": 12, "v4": 12}                     # an action that never reaches the goal
CASES = [(v, m) for v in FULL_VIEW for m in ("tma", "st128", "incremental", "compact", "bits")] + \
        [(v, m) for v in ("v2", "v4") for m in ("full", "compact")]


def make(lmz, variant, mode, n, seed=0, **kw):
    """mode: a render mode of the full f32 observation ('tma', 'st128', 'incremental', 'full' = tma) or an obs mode"""
    render_mode = mode if mode in ("tma", "st128", "incremental") else "tma"
    obs_mode = mode if mode in ("compact", "bits") else "full"
    return lmz.LmazeVecCuda(n, variant, seed=seed, render_mode=render_mode, obs_mode=obs_mode, **kw)


def oracle_variant(O, variant):
    return {"v0": O.V0, "v3": O.V3, "v2": O.V2, "v4": O.V4}[variant]


def compact_of(variant, full):
    """the un-expanded layers of full reference images [n, C, S, S]: every E-th pixel on both axes"""
    e = 7 if variant in ("v0", "v2", "v4") else 4
    crop = full[:, :, ::e, ::e]
    return crop.astype(np.uint8) if variant in FULL_VIEW else np.ascontiguousarray(crop)


def final_rows(env, idx):
    """the final rows of envs idx as the compact layers (bit-packed rows unpacked), numpy"""
    rows = env.final_obs[torch.as_tensor(idx, device=env.device, dtype=torch.long)]
    if env.obs_mode == "bits":
        rows = env.unpack_bits(rows)
    return rows.cpu().numpy()


def actions_with_invalid(rng, variant, n):
    """random actions with out-of-range values sprinkled in (v0/v3: the no-op branch; v2/v4: counted errors)"""
    hi = 4 if variant in FULL_VIEW else 25
    a = rng.randint(0, hi, size=n).astype(np.int64)
    bad = rng.rand(n) < 0.02
    a[bad] = rng.choice([-3, hi, 255], size=int(bad.sum()))
    return a


def stats_with_errors(env):
    from gym_lmaze_b200 import _abi
    out, err = (ctypes.c_int64 * _abi.NUM_STATS)(), ctypes.c_int64()
    _abi.check(env._lib.lmz_stats(env._h, ctypes.byref(out), ctypes.byref(err), env._stream()))
    return list(out), err.value


# ---------------------------------------------------------------- 1 + 2: oracle parity, nothing else changes
@pytest.mark.parametrize("variant,mode", CASES)
def test_final_rows_match_oracle_terminal_obs(lmz, oracle_mod, variant, mode):
    N, seed = 4096, 11
    T = 230 if variant in FULL_VIEW else 120
    ora = oracle_mod.OracleVec(oracle_variant(oracle_mod, variant), N, seed=seed, autoreset=False, threads=THREADS)
    env = make(lmz, variant, mode, N, seed=seed, final_obs=True)
    twin = make(lmz, variant, mode, N, seed=seed)
    ora.reset(want_obs=False); env.reset(); twin.reset()
    rng = np.random.RandomState(5)
    finished, direct_done = 0, False
    for t in range(T):
        if variant == "v4" and t == 30:
            # direct mode (lmz_set_visit): every env until its reset; env 0 with arbitrary values of its own
            vis = env.get_visit()
            vis[0] = torch.from_numpy(rng.rand(18, 18).astype(np.float32))
            env.set_visit(vis); twin.set_visit(vis); ora.set_visit(0, vis[0].cpu().numpy())
        a = actions_with_invalid(rng, variant, N)
        _, r_ref, d_ref = ora.step(a, want_obs=False)
        obs, rew, done, info = env.step(torch.from_numpy(a))
        obs2, rew2, done2, _ = twin.step(torch.from_numpy(a))
        d = done.cpu().numpy()
        assert np.array_equal(d.view(np.uint8), d_ref), t
        assert np.array_equal(rew.cpu().numpy().view(np.uint32), r_ref.view(np.uint32)), t
        idx = np.nonzero(d)[0]
        if len(idx):
            ref = compact_of(variant, np.stack([ora.render_one(int(i)) for i in idx]))
            got = final_rows(env, idx)
            assert np.array_equal(got.view(np.uint8), ref.view(np.uint8)), (t, idx[:8])
            finished += len(idx)
            direct_done = direct_done or (variant == "v4" and t >= 30 and bool(d[0]))
        ora.reset_masked(d_ref)
        # the twin without a final buffer: every output and all state bit-identical
        assert same_bytes(obs, obs2) and same_bytes(rew, rew2) and torch.equal(done, done2), t
        assert torch.equal(env.get_state(), twin.get_state()), t
        if variant == "v4":
            assert same_bytes(env.get_visit(), twin.get_visit()), t
        assert info["_final_obs"] is env.done and info["final_obs"] is env.final_obs
    assert finished >= N                                  # every env finished at least one episode
    assert stats_with_errors(env) == stats_with_errors(twin)
    assert stats_with_errors(env)[1] > 0 or variant in FULL_VIEW     # the invalid actions were counted, once
    assert direct_done or variant != "v4"                 # env 0 finished the episode it was put in direct mode in
    env.close(); twin.close()


# ---------------------------------------------------------------- 3: rows of envs that did not finish stay untouched
@pytest.mark.parametrize("variant,mode", [("v0", "compact"), ("v3", "bits"), ("v2", "full"), ("v4", "compact")])
def test_rows_without_done_keep_the_callers_values(lmz, variant, mode):
    N, W = 4096, 1024
    env = make(lmz, variant, mode, N, seed=3, final_obs=True, obs_window=W)
    env.reset()
    sentinel = 0xA5
    fin = env.final_obs.view(torch.uint8)
    fin.fill_(sentinel)
    rng = np.random.RandomState(1)
    for t in range(130):
        if t % 40 == 0:
            env.set_window((t // 40) % (N // W) * W)
        _, _, done, _ = env.step(torch.from_numpy(actions_with_invalid(rng, variant, N)))
        rows = fin.reshape(N, -1)
        assert bool((rows[~done] == sentinel).all()), t
        rows[done] = sentinel
    env.close()


# ---------------------------------------------------------------- 4: the synchronised time-out step writes every row
@pytest.mark.parametrize("variant,n", [("v0", 1 << 20), ("v2", 1 << 22)])
def test_synchronised_timeout_step_writes_every_row(lmz, variant, n):
    """After a batch reset, an action that never reaches the goal makes every env time out in the same step.  It
    does not move the ball either, so the terminal observation is the observation of the step before."""
    env = make(lmz, variant, "compact", n, seed=8, final_obs=True)
    env.reset()
    a = torch.full((n,), NO_MOVE[variant], dtype=torch.uint8, device=env.device)
    for _ in range(STEP_LIMIT_STEPS[variant] - 1):
        _, _, done, _ = env.step(a)
        assert not bool(done.any())
    before = env.obs.clone()
    env.final_obs.view(torch.uint8).fill_(0xA5)
    _, _, done, info = env.step(a)
    assert bool(done.all()) and not bool(info["terminated"].any()) and bool(info["truncated"].all())
    assert same_bytes(env.final_obs, before)
    assert not same_bytes(env.obs, before)                 # the obs rows show the new episodes
    env.close()


# ---------------------------------------------------------------- 5: CUDA graph replays and the host step
@pytest.mark.parametrize("variant,mode", [("v0", "tma"), ("v3", "incremental"), ("v4", "compact")])
def test_graph_replay_and_step_host_write_final_rows(lmz, variant, mode):
    N, seed = 4096, 21
    ref = make(lmz, variant, mode, N, seed=seed, final_obs=True)
    gr = make(lmz, variant, mode, N, seed=seed, final_obs=True)
    host = make(lmz, variant, mode, N, seed=seed, final_obs=True)
    for e in (ref, gr, host):
        e.reset()
    abuf = torch.zeros(N, dtype=torch.int64, device=gr.device)
    replay = gr.capture_step(abuf)
    a_host = torch.zeros(N, dtype=torch.int64).pin_memory()
    r_host = torch.zeros(N, dtype=torch.float32).pin_memory()
    d_host = torch.zeros(N, dtype=torch.uint8).pin_memory()
    rng = np.random.RandomState(2)
    finished = 0
    for t in range(120):
        a = torch.from_numpy(actions_with_invalid(rng, variant, N))
        _, _, done, _ = ref.step(a)
        abuf.copy_(a)
        replay()
        a_host.copy_(a)
        host.step_host(a_host, r_host, d_host)
        assert torch.equal(gr.done, done) and torch.equal(d_host.to(done.device).bool(), done), t
        m = done
        finished += int(m.sum())
        assert same_bytes(gr.final_obs[m], ref.final_obs[m]) and same_bytes(host.final_obs[m], ref.final_obs[m]), t
    assert finished > 0
    for e in (ref, gr, host):
        e.close()


# ---------------------------------------------------------------- 6: terminated / truncated
@pytest.mark.parametrize("variant", ["v0", "v3", "v2", "v4"])
def test_terminated_and_truncated_match_the_episode_counters(lmz, variant):
    N = 2048
    env = make(lmz, variant, "compact", N, seed=4, final_obs=True)
    env.reset()
    before = env.stats()
    gen = torch.Generator().manual_seed(0)
    term = trunc = 0
    for _ in range(250):
        _, _, done, info = env.step(torch.randint(0, env.num_actions, (N,), generator=gen))
        assert torch.equal(info["terminated"] | info["truncated"], done)
        assert not bool((info["terminated"] & info["truncated"]).any())
        term += int(info["terminated"].sum()); trunc += int(info["truncated"].sum())
    after = env.stats()
    assert term == after["goals"] - before["goals"] and trunc == after["timeouts"] - before["timeouts"]
    assert term > 0 and trunc > 0
    env.close()


# ---------------------------------------------------------------- 7: refusals, unbinding
def test_refusals_and_unbinding(lmz):
    from gym_lmaze_b200 import _abi
    N = 256
    with pytest.raises(ValueError, match="autoreset"):
        lmz.LmazeVecCuda(N, "v0", autoreset=False, final_obs=True)
    L = _abi.load()

    def bind(env, t, mode):
        with pytest.raises(_abi.LmzError) as ei:
            _abi.call(L.lmz_bind_final_dl, env._h, t, mode)
        return ei.value.code

    dev = torch.device("cuda")
    u8 = lambda *s: torch.empty(s, dtype=torch.uint8, device=dev)
    plain = lmz.LmazeVecCuda(N, "v0", autoreset=False, obs_mode="compact")
    assert bind(plain, u8(N, 4, 12, 12), _abi.OBS_COMPACT) == -3                      # LMZ_ERR_STATE: no autoreset
    plain.close()
    hier = lmz.LmazeHierCuda(N, "v5")
    assert bind(hier, torch.empty((N, 7, 5, 5), device=dev), _abi.OBS_COMPACT) == -4   # v5 / v6
    hier.close()
    v2 = lmz.LmazeVecCuda(N, "v2", obs_mode="compact")
    assert bind(v2, u8(N, 72), _abi.OBS_BITS) == -4                                   # bits on a foveal variant
    assert bind(v2, torch.empty((N, 5, 35, 35), device=dev), _abi.OBS_FULL) == -4     # full anywhere
    assert bind(v2, u8(N, 5, 5, 5), _abi.OBS_COMPACT) == -1                           # dtype
    v2.close()
    env = lmz.LmazeVecCuda(N, "v0", obs_mode="compact", final_obs=True)
    assert bind(env, torch.empty((N, 4, 84, 84), device=dev), _abi.OBS_FULL) == -4
    assert bind(env, torch.empty((N, 4, 12, 12), device=dev), _abi.OBS_COMPACT) == -1  # dtype
    assert bind(env, u8(N - 1, 4, 12, 12), _abi.OBS_COMPACT) == -1                      # rows
    assert bind(env, u8(N, 3, 12, 12), _abi.OBS_COMPACT) == -1                          # row shape
    assert bind(env, u8(N, 72), _abi.OBS_COMPACT) == -1
    off = u8(N * 576 + 16)[1:1 + N * 576].view(N, 4, 12, 12)
    assert bind(env, off, _abi.OBS_COMPACT) == -1                                       # 16-byte alignment
    assert bind(env, u8(N, 4, 12, 12), 7) == -1                                         # unknown mode
    # host pipeline and lmz_step_host_async refuse while bound
    with pytest.raises(ValueError, match="final"):
        env.host_pipeline()
    a_host = torch.zeros(N, dtype=torch.uint8).pin_memory()
    r_host = torch.zeros(N, dtype=torch.float32).pin_memory()
    d_host = torch.zeros(N, dtype=torch.uint8).pin_memory()
    ticket = ctypes.c_int32(-1)
    rc = L.lmz_step_host_async(env._h, a_host.data_ptr(), 0, r_host.data_ptr(), d_host.data_ptr(), None,
                               env._stream(), ctypes.byref(ticket))
    assert rc == -4 and b"final" in L.lmz_last_error()
    # bound: two launches per step (pre-pass + step kernel); unbound (NULL): one, and the buffer is not written
    env.reset()
    a = torch.full((N,), 7, dtype=torch.uint8, device=dev)
    k = env.launch_count
    env.step(a)
    assert env.launch_count == k + 2
    fin = env.final_obs
    _abi.call(L.lmz_bind_final_dl, env._h, None, _abi.OBS_COMPACT)
    env.final_obs = None
    fin.fill_(0xA5)
    k = env.launch_count
    done_any = False
    for _ in range(100):
        _, _, done, info = env.step(a)
        done_any = done_any or bool(done.any())
        assert set(info) == {"action"}
    assert done_any and env.launch_count == k + 100 and bool((fin == 0xA5).all())
    pipe = env.host_pipeline(with_obs=False)
    pipe.submit(a_host)
    assert pipe.drain() is not None
    env.close()
