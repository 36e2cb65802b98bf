"""The four lmz_config.tune knobs of the v0 / v3 full render, and lmz_create's refusal of CTA sizes no kernel is built for.

tune[0] picks the instantiation of lmz_env_tma_kernel (1, 2, 4 or 8 issuing warps) or lmz_env_st_kernel (256, 512 or
1024 threads), tune[1] the L2 hint of the bulk copies (4: the unhinted instruction), tune[2] the CTAs per SM and
tune[3] the largest piece a blob segment is cut into.  A knob point that wrote wrong bytes, or fewer of them, would
look like a speed-up in the launch sweeps (tools/sweep_render.py, v3_sweep.py, st128_sweep.py), so every point here
runs in lockstep with a default-configured handle and is compared with it byte for byte after every call, and with
the CPU oracle on a set_state that puts the ball (v3: ball and goal) on every cell, which produces every segment
layout the variant has.

Sizing: N = 3 x SMs x 8 x 32 + 21, so that at the widest TMA CTA (8 issuing warps) every warp grabs about three
32-env tiles; the tile count is odd and the last tile partial.  Each observation buffer has one guard row before and
after the rows the handle writes, filled with a sentinel: a copy past the last row hits a guard row, and a copy into a
neighbouring row shows after a masked reset, which does not rewrite that neighbour."""
import ctypes

import numpy as np
import pytest
import torch

from gpu_helpers import lmz, need_free, same_bytes, sms

PATTERN = 0x3C5AA5C3                           # sentinel word of the guard rows and of unwritten rows
SEED, ID0, T = 5, 3, 120
ROWS = 1 << 14                                 # rows per chunk of the oracle comparisons
GROUP = 7                                      # tuned handles beside one default handle
BAND = {"v0": 2352, "v3": 1152}                # bytes of one ball band (V::BAND_BYTES)
ROW_BYTES = {"v0": 4 * 84 * 84 * 4, "v3": 3 * 72 * 72 * 4}


def _points(variant):
    """(render_mode, tune) of every knob point of one variant, one knob varied at a time."""
    band = BAND[variant]
    tma = [(t0, 0, 0, 0) for t0 in (32, 64, 128, 256)] + [(0, t1, 0, 0) for t1 in (1, 2, 3, 4)]
    tma += [(0, 0, t2, 0) for t2 in (1, 2)]
    tma += [(0, 0, 0, t3) for t3 in (48, band, band + 16, 4080, 4096, 4704, 16384, 37632, 1 << 20)]
    tma += [(256, 4, 2, 4080)]
    st = [(t0, 0, t2, 0) for t0 in (256, 512) for t2 in (0, 1)] + [(1024, 0, 0, 0), (1024, 4, 1, 4080)]
    incr = [(0, 4, 0, 4080), (0, 1, 0, band)]
    return [("tma", t) for t in tma] + [("st128", t) for t in st] + [("incremental", t) for t in incr]


GRAPH_POINT = ("tma", (256, 4, 2, 4080))       # replays a captured step (8 warps re-arm the work counter)
N_GROUPS = (len(_points("v0")) + GROUP - 1) // GROUP
assert N_GROUPS == (len(_points("v3")) + GROUP - 1) // GROUP


def _words(t):
    return t.view(torch.int32).reshape(-1)


class Guarded(object):
    """`rows` observation rows between two guard rows, every word set to PATTERN."""

    def __init__(self, rows, row_shape):
        self.buf = torch.empty((rows + 2,) + tuple(row_shape), dtype=torch.float32, device="cuda")
        self.rows = self.buf[1:rows + 1]
        self.fill()

    def fill(self):
        _words(self.buf).fill_(PATTERN)

    def guards_intact(self):
        return bool((_words(self.buf[0]) == PATTERN).all()) and bool((_words(self.buf[-1]) == PATTERN).all())


class Handle(object):
    """One env whose observation rows are a Guarded buffer of its own; `win` is the Guarded buffer of its render
    window (N - 100 rows, possibly shared with other handles that use it one at a time)."""

    def __init__(self, lmz, variant, n, render_mode, tune, win):
        from gym_lmaze_b200 import _abi
        self.abi, self.point = _abi, (render_mode, tune)
        self.env = lmz.LmazeVecCuda(n, variant, seed=SEED, env_id0=ID0, autoreset=True, with_obs=False,
                                    render_mode=render_mode, tune=tune)
        self.full, self.win, self.cur = Guarded(n, self.env.obs_shape), win, None
        self.abi.call(self.env._lib.lmz_bind_dl, self.env._h, self.full.rows, self.env.reward, self.env._done_u8)
        self.window(None)

    def window(self, env_lo):
        """Render window [env_lo, env_lo + N - 100) into `win`, or the whole batch (None) into `full`."""
        self.cur = self.full if env_lo is None else self.win
        self.abi.call(self.env._lib.lmz_set_window_dl, self.env._h, self.cur.rows, 0 if env_lo is None else env_lo)
        self.env.obs = self.cur.rows

    def close(self):
        self.env.close()


def _compare(ref, h, what):
    """h's observation buffer (guard rows included), reward and done against the default handle's."""
    assert h.cur.guards_intact(), ("guard row overwritten",) + what
    assert same_bytes(h.cur.buf, ref.cur.buf), ("obs",) + what
    assert torch.equal(_words(h.env.reward), _words(ref.env.reward)), ("reward",) + what
    assert torch.equal(h.env._done_u8, ref.env._done_u8), ("done",) + what


def _lockstep(ref, tuned, call, what, refill=False):
    """call(handle) on the default handle, then on each tuned one, each compared right after its call.  refill: the
    full-render handles share one window buffer, reset to the sentinel before each of them writes it (the incremental
    render patches its previous render, so those handles keep a window buffer of their own)."""
    call(ref)
    assert ref.cur.guards_intact(), ("default handle: guard row overwritten",) + what
    for h in tuned:
        if refill and h.point[0] != "incremental":
            h.cur.fill()
        call(h)
        _compare(ref, h, (h.point,) + what)


def _cells(O, variant):
    rows = O.layout(O.V0 if variant == "v0" else O.V3)
    G = len(rows)
    return [(x, y) for x in range(1, G - 1) for y in range(1, G - 1) if rows[x][y] != "W"]


def _states(O, variant):
    """Every (ball) / (ball, goal) placement the oracle accepts, with its oracle render on the device."""
    cells = _cells(O, variant)
    if variant == "v0":
        cand = [(x, y, 5, 5) for x, y in cells]
    else:
        cand = [(bx, by, gx, gy) for bx, by in cells for gx, gy in cells]
    ora = O.OracleVec(O.V0 if variant == "v0" else O.V3, len(cand), autoreset=False)
    keep = []
    for s in cand:
        try:
            ora.force(len(keep), s[0], s[1], -1 if variant == "v0" else s[2], -1 if variant == "v0" else s[3])
        except ValueError:
            continue
        keep.append(s)
    renders = torch.from_numpy(np.stack([ora.render_one(i) for i in range(len(keep))])).cuda()
    keep = np.array(keep, dtype=np.int32)
    rows = {x for x, _ in cells}
    assert set(keep[:, 0].tolist()) == rows                                      # every ball row
    if variant == "v3":
        assert len(keep) >= 4096 and set(keep[:, 2].tolist()) == rows            # every goal row
    return keep, renders


def _oracle_check(h, renders, n_states):
    """Row i of the whole-batch buffer is the oracle's render of state i % n_states."""
    obs = h.full.rows
    for lo in range(0, obs.shape[0], ROWS):
        idx = torch.arange(lo, min(lo + ROWS, obs.shape[0]), device="cuda") % n_states
        assert torch.equal(_words(obs[lo:lo + ROWS]), _words(renders[idx])), (h.point, lo)


def _sequence(ref, tuned, states, renders, n, graph=None, steps=T):
    """reset, exhaustive set_state + render (oracle), set_state + step, T steps (uint8 actions 0..4, one int64 step,
    a rollout), a masked reset of every third env, a render window at an odd env_lo (render + step), back to the whole
    batch; then the final state and counters.  graph: a tuned handle that then replays a captured step."""
    everyone = [ref] + tuned
    _lockstep(ref, tuned, lambda h: h.env.reset(), ("reset",))
    st = ref.env.get_state()
    k = torch.arange(n, device="cuda") % len(states)
    sv = torch.as_tensor(states, device="cuda")[k]
    st[:, 0:4] = sv
    st[:, 4] = torch.arange(n, device="cuda", dtype=torch.int32) % 101       # time-outs spread over the steps
    _lockstep(ref, tuned, lambda h: h.env.set_state(st), ("set_state",))
    _lockstep(ref, tuned, lambda h: h.env.render_obs(), ("render",))
    for h in everyone:
        _oracle_check(h, renders, len(states))
    for h in everyone:
        assert h.env.stats()["steps"] == 0          # every set_state row is a state the env can be in

    gen = torch.Generator(device="cuda").manual_seed(SEED)

    def actions():
        return torch.randint(0, 5, (n,), generator=gen, device="cuda", dtype=torch.uint8)    # 4: unmatched branch
    # a set_state (and, below, a rollout) leaves the incremental tensor out of sync: the next step re-renders it all
    st2 = st.roll(1, 0)
    _lockstep(ref, tuned, lambda h: h.env.set_state(st2), ("set_state 2",))
    a = actions()
    _lockstep(ref, tuned, lambda h: h.env.step(a), ("step after set_state",))
    for t in range(steps):
        a = actions()
        if t == 7:
            a = a.to(torch.int64)
        if t == 40:
            _lockstep(ref, tuned, lambda h: h.env.rollout(5), ("rollout", t))
        _lockstep(ref, tuned, lambda h: h.env.step(a), ("step", t))
    assert ref.env.stats(check_errors=False)["timeouts"] > n // 10      # auto-reset renders happened

    mask = (torch.arange(n, device="cuda") % 3 == 0).to(torch.uint8)
    _lockstep(ref, tuned, lambda h: h.env.reset(mask=mask), ("masked reset",))
    a = actions()
    _lockstep(ref, tuned, lambda h: h.env.step(a), ("step after masked reset",))

    lo = 37                                        # odd, so that the window starts inside a tile
    for h in everyone:
        h.window(lo)
    _lockstep(ref, tuned, lambda h: h.env.render_obs(), ("window render",), refill=True)
    a = actions()
    _lockstep(ref, tuned, lambda h: h.env.step(a), ("window step",), refill=True)
    for h in everyone:
        assert h.full.guards_intact() and same_bytes(h.full.buf, ref.full.buf), (h.point, "whole batch while windowed")
        h.window(None)
    a = actions()
    _lockstep(ref, tuned, lambda h: h.env.step(a), ("step after window",))
    _lockstep(ref, tuned, lambda h: h.env.render_obs(), ("render after window",))

    def finish(h):
        assert torch.equal(h.env.get_state(), ref.env.get_state()), h.point
        assert h.env.stats(check_errors=False) == ref.env.stats(check_errors=False), h.point
    for h in tuned:
        finish(h)
    if graph is not None:
        abuf = torch.zeros(n, dtype=torch.uint8, device="cuda")
        replay = graph.env.capture_step(abuf)         # renders once before capturing
        ref.env.render_obs()
        _compare(ref, graph, ("graph capture",))
        for r in range(4):
            a = actions()
            ref.env.step(a)
            abuf.copy_(a)
            replay()
            _compare(ref, graph, ("graph replay", r))
        finish(graph)


def _run(lmz, oracle_mod, variant, points, n, graph_point=None, steps=T):
    row_shape = (4, 84, 84) if variant == "v0" else (3, 72, 72)
    n_incr = sum(mode == "incremental" for mode, _ in points)
    need_free((len(points) + n_incr + 3) * (n + 2) * ROW_BYTES[variant] + (8 << 30))
    states, renders = _states(oracle_mod, variant)
    ref = Handle(lmz, variant, n, "tma", None, Guarded(n - 100, row_shape))
    win = Guarded(n - 100, row_shape)
    tuned = [Handle(lmz, variant, n, mode, tune, Guarded(n - 100, row_shape) if mode == "incremental" else win)
             for mode, tune in points]
    graph = next((h for h in tuned if h.point == graph_point), None)
    try:
        _sequence(ref, tuned, states, renders, n, graph, steps)
    finally:
        for h in [ref] + tuned:
            h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("group", range(N_GROUPS))
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_full_render_knobs_lockstep(lmz, oracle_mod, variant, group):
    """Every TMA, ST128 and incremental knob point of _points(variant), GROUP at a time beside one default handle."""
    pts = _points(variant)[group * GROUP:(group + 1) * GROUP]
    _run(lmz, oracle_mod, variant, pts, 3 * sms() * 8 * 32 + 21, GRAPH_POINT if GRAPH_POINT in pts else None)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["v0", "v3"])
def test_bulk_split_16_bytes(lmz, oracle_mod, variant):
    """tune[3] = 16, the smallest piece the ABI accepts (every segment cut into 16-byte copies), on a batch of about
    two tiles per issuing warp, and the same with 8 issuing warps per CTA."""
    n = 2 * sms() * 32 + 5
    _run(lmz, oracle_mod, variant, [("tma", (0, 0, 0, 16)), ("tma", (256, 4, 0, 16))], n, steps=30)


# ---------------------------------------------------------------- lmz_create refuses CTA sizes no kernel is built for
REFUSAL_PATHS = [
    # (variant, obs_mode, render_mode, accepted tune[0], refused examples)
    ("v0", "full", "tma", (0, 32, 64, 128, 256), (96, 512)),
    ("v3", "full", "tma", (0, 32, 64, 128, 256), (96, 512)),
    ("v0", "full", "st128", (0, 256, 512, 1024), (128,)),
    ("v3", "full", "st128", (0, 256, 512, 1024), (128,)),
    ("v0", "full", "incremental", (0,), (32,)),
    ("v3", "full", "incremental", (0,), (32,)),
    ("v0", "compact", "tma", (0,), (32, 128)),
    ("v3", "bits", "tma", (0,), (32, 128)),
    ("v2", "full", "tma", (0, 128, 160, 192, 224, 256, 512, 1024), (96,)),
    ("v4", "full", "tma", (0, 128, 160, 192, 224, 256, 512, 1024), (96,)),
    ("v5", "full", "tma", (0, 128, 160, 192, 224, 256, 512, 1024), (96,)),
    ("v2", "compact", "tma", (0, 64, 128, 256), (512,)),
    ("v4", "compact", "tma", (0, 64, 128, 256), (512,)),
    ("v5", "compact", "tma", (0, 64, 128, 256), (512,)),
]


@pytest.mark.parametrize("variant,obs_mode,render_mode,accepted,refused", REFUSAL_PATHS,
                         ids=["-".join(p[:3]) for p in REFUSAL_PATHS])
def test_create_refuses_cta_sizes_without_a_kernel(variant, obs_mode, render_mode, accepted, refused):
    """lmz_create validates tune[0] against the kernel that renders the configured observation before it looks for a
    device: an accepted size gets past validation (a handle on a GPU machine, LMZ_ERR_CUDA "no CUDA device"
    without one), any other size is LMZ_ERR_INVALID with a message naming the sizes that kernel is built for."""
    from gym_lmaze_b200 import build, _abi
    build.build()
    L = _abi.load()
    has_cuda = torch.cuda.is_available()
    cfg = _abi.LmzConfig()
    L.lmz_default_config(ctypes.byref(cfg))
    cfg.variant = {"v0": _abi.LMZ_V0, "v2": _abi.LMZ_V2, "v3": _abi.LMZ_V3, "v4": _abi.LMZ_V4, "v5": _abi.LMZ_V5}[variant]
    cfg.num_envs = 64
    cfg.obs_mode = {"full": _abi.OBS_FULL, "compact": _abi.OBS_COMPACT, "bits": _abi.OBS_BITS}[obs_mode]
    cfg.render_mode = {"tma": _abi.RENDER_TMA, "st128": _abi.RENDER_ST128, "incremental": _abi.RENDER_INCREMENTAL}[render_mode]
    listed = ("{%s}" % ", ".join(str(t) for t in accepted)).encode()
    for t in accepted + refused:
        cfg.tune[0] = t
        h = ctypes.c_void_p()
        rc = L.lmz_create(ctypes.byref(cfg), ctypes.byref(h))
        if t in refused:
            assert rc == -1 and not h.value, t
            msg = L.lmz_last_error()
            assert (b"tune[0] = %d" % t) in msg and listed in msg, msg
        elif has_cuda:
            assert rc == 0 and h.value, (t, L.lmz_last_error())
            assert L.lmz_destroy(h) == 0
        else:
            assert rc == -2 and b"no CPU path" in L.lmz_last_error(), t
