"""GPU tier: observation tensors in compressible device memory (lmz_alloc_obs, DESIGN.md §2).

Full-render observation tensors are allocated by the library in memory the L2 may keep compressed.  Compression is
lossless and invisible to kernels and copies, so every output must be bit for bit what the same handle writes into a
plain torch.empty tensor.  A 2^20-env v0 observation tensor is 118 GB, so two of them do not fit side by side: each case
runs twice from the same seed and actions, once per kind of memory, and compares per-row digests of the observations
and every reward, done flag and state word."""
import gc

import pytest
import torch

pytestmark = pytest.mark.gpu

STEPS = 130
CHECKPOINTS = (1, 64, STEPS)
CH = 1 << 14                            # rows per chunk of a digest


@pytest.fixture(scope="module")
def lmz():
    import gym_lmaze_b200 as g
    from gym_lmaze_b200 import _abi
    _abi.load()
    assert torch.cuda.is_available()
    return g


@pytest.fixture(scope="module")
def supported(lmz):
    """Does this device and driver grant compressible memory at all?"""
    from gym_lmaze_b200 import _abi
    t, compressed_bytes = _abi.obs_empty((1 << 22,), torch.float32, "cuda", True)
    del t
    return compressed_bytes > 0


def digest(t):
    """int64 per row: a weighted sum of the row's 32-bit words (u8 rows: bytes) -- no overflow, position-sensitive"""
    rows = t.reshape(t.shape[0], -1)
    words = rows.view(torch.int32) if rows.dtype == torch.float32 else rows
    gen = torch.Generator(device=t.device).manual_seed(5)
    w = torch.randint(1, 1 << 16, (words.shape[1],), generator=gen, device=t.device, dtype=torch.int64)
    out = torch.empty(rows.shape[0], dtype=torch.int64, device=t.device)
    for lo in range(0, rows.shape[0], CH):
        out[lo:lo + CH] = (words[lo:lo + CH].to(torch.int64) * w).sum(1)
    return out


def make_plain(lmz, env):
    """Rebind `env` to plain torch tensors of the same shapes (the path every output is compared against)."""
    from gym_lmaze_b200 import _abi
    shape, dtype = env.obs.shape, env.obs.dtype
    env.obs = None
    if isinstance(env, lmz.LmazeHierCuda):
        loc_shape = env.loc_obs.shape
        env.loc_obs = env.fov_obs = None
        gc.collect()
        env.loc_obs = torch.zeros(loc_shape, dtype=torch.float32, device=env.device)
        _abi.call(env._lib.lmz_bind_local_dl, env._h, env.loc_obs, env.local_reward, env._ldone_u8,
                  env._loc_err_u8, env.foveal_goal)
    env.obs = torch.empty(shape, dtype=dtype, device=env.device)
    if isinstance(env, lmz.LmazeHierCuda):
        env.fov_obs = env.obs
    env._bind()


def run(lmz, variant, n, plain, steps=STEPS, **kw):
    """`steps` steps of one seeded handle; returns what it computed: obs digests at CHECKPOINTS, every reward / done,
    the final state (and v5's local obs / reward / done)"""
    hier = variant == "v5"
    env = lmz.LmazeHierCuda(n, "v5", seed=11, **kw) if hier else lmz.LmazeVecCuda(n, variant, seed=11, **kw)
    if plain:
        make_plain(lmz, env)
    gen = torch.Generator(device="cuda").manual_seed(3)
    out = {"reward": [], "done": [], "obs": {}, "compressed": env.obs_compressed}
    env.reset()
    for i in range(1, steps + 1):
        a = torch.randint(0, env.num_actions, (n,), generator=gen, device="cuda", dtype=torch.uint8)
        if hier:
            env.plannerStep(torch.randint(0, 25, (n,), generator=gen, device="cuda", dtype=torch.uint8), mask="auto")
            env.step(a, goal_plane=False)
        else:
            env.step(a)
        out["reward"].append(env.reward.clone())
        out["done"].append(env.done.clone())
        if hier:
            out["reward"].append(env.local_reward.clone())
            out["done"].append(env.local_done.clone())
        if i in CHECKPOINTS:
            out["obs"][i] = digest(env.obs)
            if hier:
                out["obs"][-i] = digest(env.loc_obs)
    out["state"] = env.get_state()
    env.close()
    del env
    gc.collect()
    torch.cuda.empty_cache()
    return out


def assert_same(a, b):
    assert a["obs"].keys() == b["obs"].keys()
    for k in a["obs"]:
        assert torch.equal(a["obs"][k], b["obs"][k]), "observation digests differ at checkpoint %d" % k
    for name in ("reward", "done"):
        for t, (x, y) in enumerate(zip(a[name], b[name])):
            assert torch.equal(x.view(torch.uint8), y.view(torch.uint8)), "%s differs at step %d" % (name, t)
    assert torch.equal(a["state"], b["state"])


# (variant, envs, constructor keywords, whether the env puts its observations in compressible memory)
CASES = {
    "v0_tma": ("v0", 1 << 20, {}, True),
    "v3_tma": ("v3", 1 << 20, {}, True),
    "v0_st128": ("v0", 1 << 18, {"render_mode": "st128"}, True),
    "v0_window": ("v0", 1 << 18, {"obs_window": 40000}, True),
    "v5_full": ("v5", 1 << 16, {}, True),
    "v0_compact": ("v0", 1 << 18, {"obs_mode": "compact"}, False),
    "v0_incremental": ("v0", 1 << 16, {"render_mode": "incremental"}, False),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_obs_compressed_by_mode(lmz, supported, case):
    variant, n, kw, compressible = CASES[case]
    n = min(n, 1 << 16)                   # small batches, but large enough for the render window of v0_window
    env = lmz.LmazeHierCuda(n, "v5", **kw) if variant == "v5" else lmz.LmazeVecCuda(n, variant, **kw)
    assert env.obs_compressed == (compressible and supported)
    env.close()


@pytest.mark.parametrize("case", [c for c in sorted(CASES) if CASES[c][3]])
def test_compressible_obs_gives_the_same_outputs(lmz, supported, case):
    variant, n, kw, _ = CASES[case]
    new = run(lmz, variant, n, plain=False, **kw)
    assert new["compressed"] == supported
    ref = run(lmz, variant, n, plain=True, **kw)
    assert_same(new, ref)


def test_graph_replay_on_compressible_obs(lmz):
    n = 1 << 16
    outs = []
    for plain in (False, True):
        env = lmz.LmazeVecCuda(n, "v0", seed=5)
        if plain:
            make_plain(lmz, env)
        env.reset()
        buf = torch.zeros(n, dtype=torch.uint8, device="cuda")
        replay = env.capture_step(buf)
        gen = torch.Generator(device="cuda").manual_seed(9)
        digests = []
        for i in range(STEPS):
            buf.copy_(torch.randint(0, 4, (n,), generator=gen, device="cuda", dtype=torch.uint8))
            replay()
            if i % 13 == 0:
                digests.append(torch.cat([digest(env.obs), env.reward.view(torch.int32).long(), env.done.long()]))
        digests.append(env.get_state().long().flatten())
        outs.append(torch.cat(digests))
        env.close()
        del env, replay
    assert torch.equal(outs[0], outs[1])


def test_step_host_reads_compressible_obs(lmz):
    n = 1 << 14
    outs = []
    for plain in (False, True):
        env = lmz.LmazeVecCuda(n, "v0", seed=6)
        if plain:
            make_plain(lmz, env)
        env.reset()
        r = torch.empty(n, dtype=torch.float32).pin_memory()
        d = torch.empty(n, dtype=torch.uint8).pin_memory()
        o = torch.empty(env.obs.shape, dtype=torch.float32).pin_memory()
        gen = torch.Generator().manual_seed(2)
        for _ in range(STEPS):
            env.step_host(torch.randint(0, 4, (n,), generator=gen, dtype=torch.uint8), r, d, obs_host=o)
        outs.append((o.clone(), r.clone(), d.clone(), env.obs.cpu()))
        env.close()
    for x, y in zip(*outs):
        assert torch.equal(x.view(torch.uint8), y.view(torch.uint8))
    assert torch.equal(outs[0][0], outs[0][3])          # the D2H copy is what the device holds


def test_obs_outlives_the_handle_and_is_freed_with_its_last_reference(lmz, supported):
    n = 1 << 20
    gc.collect()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    env = lmz.LmazeVecCuda(n, "v0", seed=1)
    env.reset()
    obs = env.obs
    nbytes = obs.numel() * obs.element_size()
    assert free0 - torch.cuda.mem_get_info()[0] >= nbytes
    expect = digest(obs)
    env.close()
    del env
    gc.collect()
    assert torch.equal(digest(obs), expect)              # still readable, still what the last render wrote
    view = obs[7:9]
    del obs, expect
    torch.cuda.empty_cache()
    assert free0 - torch.cuda.mem_get_info()[0] >= nbytes   # a view keeps the whole allocation
    del view
    torch.cuda.empty_cache()
    # the memory is back at once (compression metadata included); slack for the allocator's own blocks
    assert torch.cuda.mem_get_info()[0] >= free0 - (256 << 20)


def test_plain_request_gives_plain_memory_and_the_same_outputs(lmz):
    from gym_lmaze_b200 import _abi
    n = 1 << 14
    outs = []
    for compressible in (True, False):
        env = lmz.LmazeVecCuda(n, "v0", seed=4)
        env.obs = None
        env.obs, compressed_bytes = _abi.obs_empty((n, 4, 84, 84), torch.float32, env.device, compressible)
        if not compressible:
            assert compressed_bytes == 0
        env._bind()
        env.reset()
        gen = torch.Generator(device="cuda").manual_seed(8)
        for _ in range(STEPS):
            env.step(torch.randint(0, 4, (n,), generator=gen, device="cuda", dtype=torch.uint8))
        outs.append((env.obs.clone(), env.reward.clone(), env.done.clone(), env.get_state()))
        env.close()
    for x, y in zip(*outs):
        assert torch.equal(x, y)
