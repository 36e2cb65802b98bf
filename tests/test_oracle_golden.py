"""CPU tier: the C restatement (oracle/) against the golden fixtures that
tests/golden/gen_golden.py produced from the UNMODIFIED reference."""
import hashlib
import os

import numpy as np
import pytest

from golden_io import Traces, f64, fov_image, loc_image, pack_v2_spawn, reward_f32_bits, unpack


def test_layouts_match_reference(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "layouts.npz"))
    for name, variant in (("v0", oracle_mod.V0), ("v3", oracle_mod.V3)):
        rows = oracle_mod.layout(variant)
        assert rows == [str(r) for r in z[name]]
        assert hashlib.md5("/".join(rows).encode()).hexdigest() == str(z[name + "_md5"])
    # SURVEY.md section 8a (a2): md5 of the v0 rows
    assert str(z["v0_md5"]).startswith("b2b870fa")


def test_v0_transition_table_exhaustive(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v0_table.npz"))
    tab = np.concatenate([z["table"], z["edge"]])
    assert z["table"].shape == (72 * 5 * 4, 11)
    o = oracle_mod.OracleVec(oracle_mod.V0, 1, autoreset=False)
    for (x, y, a, prb, sb, nx, ny, rb, d, gd, sa) in tab:
        o.force(0, int(x), int(y), step_count=int(sb), reward=float(f64(prb)), goal_count=3)
        dd, _ = o.step_one(0, int(a))
        pos, sc, gc, rw = o.export()
        assert (pos[0, 0], pos[0, 1]) == (nx, ny)
        assert rw.view(np.int64)[0] == rb          # f64 bit pattern, incl. -0.0 (Q2) and stale reward (Q1)
        assert dd == d and sc[0] == sa and gc[0] - 3 == gd


def test_v0_renders_all_positions(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v0_table.npz"))
    o = oracle_mod.OracleVec(oracle_mod.V0, 1, autoreset=False)
    for (x, y), bits in zip(z["positions"], z["renders"]):
        o.force(0, int(x), int(y))
        got = o.render_one(0)
        assert got.dtype == np.float32 and got.shape == (4, 84, 84)
        assert np.array_equal(got, unpack(bits, (4, 84, 84)))
    # channel sums quoted in SURVEY.md T0
    assert got.sum(axis=(1, 2)).tolist() == [49.0, 3528.0, 49.0, 3430.0]


def test_v0_reset_semantics(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v0_table.npz"))
    bx, by, rbits, sc, gc, gx, gy = z["reset_info"]
    o = oracle_mod.OracleVec(oracle_mod.V0, 1, autoreset=False)
    o.force(0, 4, 4, step_count=55, reward=-1.0, goal_count=5)
    obs = o.reset(spawn=[[bx, by, -1, -1]])
    pos, s, g, rw = o.export()
    assert tuple(pos[0]) == (bx, by, gx, gy) and s[0] == sc and g[0] == gc
    assert rw.view(np.int64)[0] == rbits and rbits == np.float64(-0.0).view(np.int64)
    assert np.array_equal(obs[0], unpack(z["reset_obs"], (4, 84, 84)))
    # the reference rejected (2,2) [wall] and (5,5) [goal] before accepting (10,10)
    assert tuple(z["reject_info"][:2]) == (10, 10)
    L = oracle_mod.lib()
    e = o._env(0)
    assert L.lmzo_reset(e, 2, 2, -1, -1) == -1 and L.lmzo_reset(e, 5, 5, -1, -1) == -1
    assert L.lmzo_reset(e, 10, 10, -1, -1) == 0


@pytest.mark.parametrize("variant_name", ["v0", "v3"])
def test_traces(oracle_mod, golden_dir, variant_name):
    variant = oracle_mod.V0 if variant_name == "v0" else oracle_mod.V3
    shape = oracle_mod.OBS_SHAPE[variant]
    tr = Traces(golden_dir, variant_name)
    o = oracle_mod.OracleVec(variant, tr.n_envs, autoreset=True)
    sp0 = tr.per_env("spawn0")
    if variant == oracle_mod.V0:
        sp0 = np.concatenate([sp0, -np.ones_like(sp0)], axis=1)
    o.reset(spawn=sp0)
    acts, spawns, dones_ref = tr.per_step("actions"), tr.per_step("spawn"), tr.per_step("done")
    want_r, obs_bits = reward_f32_bits(tr.per_step("reward_bits")), tr.per_step("obs")
    pos_ref, sc_ref = tr.per_step("pos"), tr.per_step("step_count")
    for t in range(tr.T):
        spawn = spawns[t]
        if variant == oracle_mod.V0:
            spawn = np.concatenate([spawn, -np.ones_like(spawn)], axis=1)
        spawn = np.where(dones_ref[t][:, None] > 0, spawn, 1)      # unused rows: any value
        # pre-reset positions are checked through a non-resetting twin below; here: outputs
        obs, rew, done = o.step(acts[t], spawn=spawn)
        assert np.array_equal(rew.view(np.uint32), want_r[t]), t
        assert np.array_equal(done, dones_ref[t]), t
        assert np.array_equal(obs, unpack(obs_bits[t], shape)), t
        pos, sc = o.export()[:2]
        live = done == 0
        assert np.array_equal(pos[live, :pos_ref.shape[2]], pos_ref[t][live]), t
        assert np.array_equal(sc[live], sc_ref[t][live]), t
    assert o.stats[1] == int(dones_ref.sum())
    assert o.stats[1] >= 2 * tr.n_envs       # every env finished at least two episodes


def test_v0_real_mt_trace(oracle_mod, golden_dir):
    """BASELINE config-1-style run: spawns came from the reference's own MT19937 stream."""
    z = np.load(os.path.join(golden_dir, "v0_traces.npz"))
    o = oracle_mod.OracleVec(oracle_mod.V0, 1, autoreset=True)
    o.reset(spawn=[[z["mt_spawn0"][0], z["mt_spawn0"][1], -1, -1]])
    goal_bits = np.float32(100.0).view(np.uint32)
    for t in range(len(z["mt_actions"])):
        sp = z["mt_spawn"][t]
        spawn = [[sp[0], sp[1], -1, -1]] if z["mt_done"][t] else [[1, 1, -1, -1]]
        _, rew, done = o.step([z["mt_actions"][t]], spawn=spawn, want_obs=False)
        assert rew.view(np.uint32)[0] == reward_f32_bits(z["mt_reward_bits"][t])
        assert done[0] == z["mt_done"][t]
        if not done[0]:
            assert tuple(o.export()[0][0][:2]) == tuple(z["mt_pos"][t])
        elif rew.view(np.uint32)[0] == goal_bits:
            pass
    assert z["mt_done"].sum() >= 5


def test_v3_transition_table(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v3_table.npz"))
    tab = np.concatenate([z["table"], z["edge"]])
    assert len(z["table"]) == 6 * 73 * 5
    o = oracle_mod.OracleVec(oracle_mod.V3, 1, autoreset=False)
    for (bx, by, gx, gy, a, sb, nx, ny, rb, d, sa) in tab:
        o.force(0, int(bx), int(by), int(gx), int(gy), step_count=int(sb))
        dd, _ = o.step_one(0, int(a))
        pos, sc, _, rw = o.export()
        assert tuple(pos[0]) == (nx, ny, gx, gy)
        assert rw.view(np.int64)[0] == rb
        assert dd == d and sc[0] == sa


def test_v3_renders(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v3_table.npz"))
    o = oracle_mod.OracleVec(oracle_mod.V3, 1, autoreset=False)
    for (bx, by, gx, gy), bits in zip(z["render_keys"], z["renders"]):
        o.force(0, int(bx), int(by), int(gx), int(gy))
        assert np.array_equal(o.render_one(0), unpack(bits, (3, 72, 72)))
    bx, by, gx, gy, sc = z["reset_info"]
    obs = o.reset(spawn=[[bx, by, gx, gy]])
    assert np.array_equal(obs[0], unpack(z["reset_obs"], (3, 72, 72)))
    assert tuple(z["test_info"]) == (7, 8, 8, 8)       # reset(mode="test") cells
    o.force(0, 7, 8, 8, 8)
    assert np.array_equal(o.render_one(0), unpack(z["test_obs"], (3, 72, 72)))


def test_philox_known_answers(oracle_mod):
    # Random123 known-answer vectors for philox4x32-10
    assert [hex(v) for v in oracle_mod.philox([0] * 4, [0] * 2)] == \
        ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    assert [hex(v) for v in oracle_mod.philox([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2)] == \
        ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    assert [hex(v) for v in oracle_mod.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344],
                                              [0xa4093822, 0x299f31d0])] == \
        ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_rng_spawn_distribution(oracle_mod):
    rows = oracle_mod.layout(oracle_mod.V0)
    counts = {}
    for i in range(7100):
        sx, sy, gx, gy = oracle_mod.rng_spawn(oracle_mod.V0, 99, i, 0)
        assert rows[sx][sy] in "BS"
        counts[(sx, sy)] = counts.get((sx, sy), 0) + 1
    assert len(counts) == 71 and min(counts.values()) > 50 and max(counts.values()) < 160
    rows3 = oracle_mod.layout(oracle_mod.V3)
    for i in range(500):
        sx, sy, gx, gy = oracle_mod.rng_spawn(oracle_mod.V3, 5, i, 2)
        assert rows3[sx][sy] != "W" and rows3[gx][gy] != "W" and (sx, sy) != (gx, gy)
    acts = [oracle_mod.rng_action(1, 2, t) for t in range(4000)]
    assert sorted(set(acts)) == [0, 1, 2, 3] and min(np.bincount(acts)) > 850


def test_pyloop_matches_c_oracle(oracle_mod):
    """The interpreted restatement bench.py times for context agrees with the C oracle."""
    from oracle.pyloop import PyLoopV0
    env = PyLoopV0(oracle_mod.layout(oracle_mod.V0), (3, 5))
    o = oracle_mod.OracleVec(oracle_mod.V0, 1, autoreset=False)
    o.reset(spawn=[[3, 5, -1, -1]])
    for a in (1, 1, 0, 7, 3, 2):
        obs, r, d, _ = env.step(a)
        o_ref, r_ref, d_ref = o.step([a])
        assert np.array_equal(obs, o_ref[0]) and np.float32(r).view(np.uint32) == r_ref.view(np.uint32)[0]
        assert bool(d) == bool(d_ref[0])


def test_live_reference_random_walk(oracle_mod):
    """Where the reference checkout is present (build container), step it live beside the oracle."""
    from oracle import ref_loader
    if not ref_loader.reference_available():
        pytest.skip("reference checkout not present (GPU box): golden fixtures cover this")
    env, scripted, _ = ref_loader.make_reference_env("v0", first_draws=(4, 4))
    o = oracle_mod.OracleVec(oracle_mod.V0, 1, autoreset=False)
    o.reset(spawn=[[4, 4, -1, -1]])
    rng = np.random.RandomState(5)
    for t in range(25):
        a = int(rng.randint(0, 5))
        obs, r, d, info = env.step(a)
        o_ref, r_ref, d_ref = o.step([a])
        assert np.array_equal(obs, o_ref[0]) and np.float32(r).view(np.uint32) == r_ref.view(np.uint32)[0]
        assert bool(d) == bool(d_ref[0]) and info == a


# ---------------------------------------------------------------- v2 (multi-layout foveal env)
def test_v2_layouts(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v2_layouts.npz"))
    md5s = []
    for k in range(5):
        rows = oracle_mod.layout_v2(k + 1)
        assert rows == [str(r) for r in z["layouts"][k]]
        md5s.append(hashlib.md5("/".join(rows).encode()).hexdigest()[:8])
    assert md5s == ["670a2974", "c7ab0302", "0f7e0ab0", "d82dd8d9", "19d9c0c4"]      # SURVEY.md section 8f


def test_v2_transition_table(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v2_table.npz"))
    o = oracle_mod.OracleVec(oracle_mod.V2, 1, autoreset=False)
    for row, bits in zip(z["table"], z["obs"]):
        L, bx, by, gx, gy, px, py, a, sb, nx, ny, rb, d, sa = (int(v) for v in row)
        o.force_v2(0, L, bx, by, gx, gy, px, py, step_count=sb)
        dd, _ = o.step_one(0, a)
        pos, sc, _, rw = o.export()
        assert tuple(pos[0]) == (nx, ny, gx, gy) and rw.view(np.int64)[0] == rb and dd == d and sc[0] == sa
        assert np.array_equal(o.render_one(0), unpack(bits, (5, 35, 35)))
    rw = np.int64(z["table"][:, 11]).view(np.float64)
    assert set(rw.tolist()) == {-1.0, -0.01, 100.0, 0.0}
    assert np.signbit(rw[rw == 0.0]).all() and (rw == 0.0).sum() >= 20      # X-but-not-goal cells return -0.0


def test_v2_traces(oracle_mod, golden_dir):
    tr = Traces(golden_dir, "v2")
    o = oracle_mod.OracleVec(oracle_mod.V2, tr.n_envs, autoreset=True)
    init = tr.per_env("init")                                      # bx, by, gx, gy, layout, layout-before
    for e in range(tr.n_envs):                                     # the maze the constructor rolled
        oracle_mod.lib().lmzo_layout_v2(int(init[e, 5]), ctypes_grid(o, e))
    obs = o.reset(spawn=pack_v2_spawn(init))
    assert np.array_equal(obs, unpack(tr.per_env("first_obs"), (5, 35, 35)))
    acts, s5, dref = tr.per_step("actions"), tr.per_step("spawn"), tr.per_step("done")
    want_r, obs_bits = reward_f32_bits(tr.per_step("reward_bits")), tr.per_step("obs")
    for t in range(tr.T):
        spawn = np.where(dref[t][:, None] > 0, pack_v2_spawn(s5[t]), 0)
        obs, rew, done = o.step(acts[t], spawn=spawn)
        assert np.array_equal(rew.view(np.uint32), want_r[t]), t
        assert np.array_equal(done, dref[t]), t
        assert np.array_equal(obs, unpack(obs_bits[t], (5, 35, 35))), t
    assert o.stats[1] == int(dref.sum()) >= 16


def ctypes_grid(o, i):
    """char* to env i's grid (offset of lmzo_env.grid = 7 ints)."""
    import ctypes
    return ctypes.cast(o._env(i) + 7 * 4, ctypes.c_char_p)


# ---------------------------------------------------------------- v4 (v2 + float visit layer)
def test_v4_transition_table(oracle_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "v4_table.npz"))
    o = oracle_mod.OracleVec(oracle_mod.V4, 1, autoreset=False)
    for k, row in enumerate(z["table"]):
        L, bx, by, gx, gy, a, sb, nx, ny, rb, d, sa = (int(v) for v in row)
        o.force_v2(0, L, bx, by, gx, gy, bx, by, step_count=sb)
        o.set_visit(0, z["pre_visit"][k])
        dd, _ = o.step_one(0, a)
        pos, sc, _, rw = o.export()
        assert tuple(pos[0]) == (nx, ny, gx, gy) and rw.view(np.int64)[0] == rb and dd == d and sc[0] == sa
        assert np.array_equal(o.export_visit()[0].view(np.uint32), z["post_visit"][k].view(np.uint32))   # bit-exact f32
        got = o.render_one(0)
        assert np.array_equal(got.view(np.uint32), fov_image(z["obs_bits"][k], z["obs_visit"][k]).view(np.uint32))


def test_v4_traces(oracle_mod, golden_dir):
    tr = Traces(golden_dir, "v4")
    o = oracle_mod.OracleVec(oracle_mod.V4, tr.n_envs, autoreset=True)
    obs = o.reset(spawn=pack_v2_spawn(tr.per_env("init")))          # bx, by, gx, gy, layout
    assert np.array_equal(obs, fov_image(tr.per_env("first_bits"), tr.per_env("first_visit")))
    acts, s5, dref = tr.per_step("actions"), tr.per_step("spawn"), tr.per_step("done")
    want_r, visit_sum = reward_f32_bits(tr.per_step("reward_bits")), tr.per_step("visit_sum")
    obs_bits, obs_visit = tr.per_step("obs_bits"), tr.per_step("obs_visit")
    for t in range(tr.T):
        spawn = np.where(dref[t][:, None] > 0, pack_v2_spawn(s5[t]), 0)
        obs, rew, done = o.step(acts[t], spawn=spawn)
        vis = o.export_visit()
        assert np.array_equal(rew.view(np.uint32), want_r[t]), t
        assert np.array_equal(done, dref[t]), t
        assert np.array_equal(obs.view(np.uint32), fov_image(obs_bits[t], obs_visit[t]).view(np.uint32)), t
        assert np.array_equal([float(v.astype(np.float64).sum()) for v in vis], visit_sum[t]), t
    assert np.array_equal(vis.view(np.uint32), tr.per_env("final_visit").view(np.uint32))


# ---------------------------------------------------------------- v5 / v6 (planner / actor protocol)
@pytest.mark.parametrize("variant", ["v5", "v6", "v5_edge"])
def test_v5_traces(oracle_mod, golden_dir, variant):
    """Every value the reference returned from reset / plannerStep / step over 4 x ~730 events; "v5_edge": 21 scripted
    envs on the paths random traces never take (steps before any plannerStep, stepping on past globalDone, goal
    next to the ball, every planner cell, the 50-planner-step timeout) -- tests/golden/gen_golden_v5_edge.py."""
    tr = Traces(golden_dir, variant)
    n_events = 0
    for e in range(tr.n_envs):
        o = oracle_mod.OracleHier(1)
        z = tr.env(e)
        for k, row in enumerate(z["events"]):
            kind, arg, grb, orb, gd, ld, bx, by = (int(v) for v in row[:8])
            if kind == 0:
                fov = o.reset(spawn=[pack_v2_spawn(row[8:13])])
                assert np.array_equal(fov[0].view(np.uint32), fov_image(z["fov_bits"][k], z["fov_visit"][k]).view(np.uint32)), (e, k)
            elif kind == 1:
                loc, err = o.planner_step([arg])
                assert not err[0] and np.array_equal(loc[0], loc_image(z["loc_bits"][k])), (e, k)
            else:
                fov, loc, gr, lr, gdo, ldo, err = o.step([arg])
                assert not err[0]
                assert gr.view(np.uint32)[0] == reward_f32_bits(grb), (e, k)
                assert lr.view(np.uint32)[0] == reward_f32_bits(orb), (e, k)
                assert (gdo[0], ldo[0]) == (gd, ld), (e, k)
                assert np.array_equal(fov[0].view(np.uint32), fov_image(z["fov_bits"][k], z["fov_visit"][k]).view(np.uint32)), (e, k)
                assert np.array_equal(loc[0], loc_image(z["loc_bits"][k])), (e, k)
            st = o.export()[0]
            assert (st[0], st[1]) == (bx, by), (e, k)
            assert float(o.export_visit()[0].astype(np.float64).sum()) == z["visit_sum"][k], (e, k)
            n_events += 1
    assert n_events > (400 if variant == "v5_edge" else 2500)
    if variant == "v6":       # safeFovealGoal(): re-draw until the window cell is not a wall (lmaze_env_v6.py:505-523)
        o = oracle_mod.OracleHier(1)
        rows = [str(r) for r in tr["safe_layout"]]
        k = [i for i in range(1, 6) if oracle_mod.layout_v2(i) == rows][0]
        draws, pos = tr["safe_draws"], 0
        for bx, by, want, used in tr["safe_results"]:
            o.reset(spawn=[[4, 4, 8, 8 | (k << 5)]], want_obs=False)
            oracle_mod.lib().lmzo_env_force_v2(o._env(0), k, int(bx), int(by), 8, 8, int(bx), int(by), 0)
            got, n_used = o.safe_goal(0, draws[pos:pos + 40])
            assert (got, n_used) == (want, used)
            pos += used
