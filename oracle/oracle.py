"""ctypes wrapper around oracle/liblmaze_oracle.so (test infrastructure only).

Importers: tests/, __graft_entry__.smoke(), bench.py's cpu_baseline / --impl
reference legs.  The product package never imports this module.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liblmaze_oracle.so")

V0, V2, V3, V4, V5 = 0, 2, 3, 4, 5
NUM_STATS = 8
STAT_NAMES = ("steps", "episodes", "goals", "timeouts", "wall_bumps", "moves", "stale", "eplen_sum")
OBS_SHAPE = {V0: (4, 84, 84), V2: (5, 35, 35), V3: (3, 72, 72), V4: (7, 35, 35), V5: (7, 35, 35)}
# f32 bit patterns of the only rewards the reference can emit (SURVEY.md Q8)
REWARD_BITS = {"neg_zero": 0x80000000, "wall": 0xBF800000, "move": 0xBC23D70A, "goal": 0x42C80000}


def build(force=False):
    """Compile the oracle with the system gcc (no-op if the .so is newer than its sources)."""
    srcs = [os.path.join(_HERE, f) for f in ("lmaze_oracle.c", "lmaze_oracle.h")]
    if (not force and os.path.isfile(_LIB_PATH)
            and os.path.getmtime(_LIB_PATH) >= max(os.path.getmtime(s) for s in srcs)):
        return _LIB_PATH
    subprocess.check_call(["make", "-s", "-B", "-C", _HERE, "CC=gcc"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(_LIB_PATH):
        build()
    L = ctypes.CDLL(_LIB_PATH)
    vp, i32, i64, u32, u64, dbl = (ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64,
                                   ctypes.c_uint32, ctypes.c_uint64, ctypes.c_double)
    ip = ctypes.POINTER(ctypes.c_int)
    L.lmzo_abi_version.restype = ctypes.c_int
    L.lmzo_layout.argtypes = [ctypes.c_int, ctypes.c_char_p]
    L.lmzo_layout.restype = ctypes.c_int
    L.lmzo_obs_floats.argtypes = [ctypes.c_int]
    L.lmzo_obs_floats.restype = i64
    L.lmzo_init.argtypes = [vp, ctypes.c_int]
    L.lmzo_reset.argtypes = [vp] + [ctypes.c_int] * 4
    L.lmzo_reset.restype = ctypes.c_int
    L.lmzo_step.argtypes = [vp, i64, ip]
    L.lmzo_step.restype = ctypes.c_int
    L.lmzo_done.argtypes = [vp]
    L.lmzo_done.restype = ctypes.c_int
    L.lmzo_render.argtypes = [vp, vp]
    L.lmzo_render.restype = None
    L.lmzo_philox4x32_10.argtypes = [vp, vp, vp]
    L.lmzo_philox4x32_10.restype = None
    L.lmzo_rng_spawn.argtypes = [ctypes.c_int, u64, u64, u32, ip, ip, ip, ip]
    L.lmzo_rng_spawn.restype = None
    L.lmzo_rng_action.argtypes = [u64, u64, u64]
    L.lmzo_rng_action.restype = ctypes.c_int
    L.lmzo_rng_action25.argtypes = [u64, u64, u64]
    L.lmzo_rng_action25.restype = ctypes.c_int
    L.lmzo_rng_hier.argtypes = [u64, u64, u64, ip, ip]
    L.lmzo_rng_hier.restype = None
    L.lmzo_vec_step.argtypes = [vp, i64, vp, vp, u64, u64, vp, ctypes.c_int, vp, vp, vp, vp, ctypes.c_int]
    L.lmzo_vec_step.restype = None
    L.lmzo_vec_reset.argtypes = [vp, i64, ctypes.c_int, vp, u64, u64, vp, vp, ctypes.c_int]
    L.lmzo_vec_reset.restype = None
    L.lmzo_sizeof_env.restype = i64
    L.lmzo_env_at.argtypes = [vp, i64]
    L.lmzo_env_at.restype = vp
    L.lmzo_env_set_flags.argtypes = [vp, ctypes.c_int, ctypes.c_int]
    L.lmzo_env_set_flags.restype = None
    L.lmzo_vec_export.argtypes = [vp, i64, vp, vp, vp, vp]
    L.lmzo_vec_export.restype = None
    L.lmzo_env_force.argtypes = [vp, ctypes.c_int] + [ctypes.c_int] * 4 + [i64, dbl, i64]
    L.lmzo_env_force.restype = ctypes.c_int
    L.lmzo_env_force_v2.argtypes = [vp] + [ctypes.c_int] * 7 + [i64]
    L.lmzo_env_force_v2.restype = ctypes.c_int
    L.lmzo_vec_export_aux.argtypes = [vp, i64, vp]
    L.lmzo_vec_export_aux.restype = None
    L.lmzo_vec_export_visit.argtypes = [vp, i64, vp]
    L.lmzo_vec_export_visit.restype = None
    L.lmzo_env_set_visit.argtypes = [vp, vp]
    L.lmzo_env_set_visit.restype = None
    u8p = vp
    L.lmzo_vec_reset_v5.argtypes = [vp, i64, u8p, vp, u64, u64, vp, vp]
    L.lmzo_vec_reset_v5.restype = None
    L.lmzo_vec_planner_v5.argtypes = [vp, i64, vp, u8p, vp, vp]
    L.lmzo_vec_planner_v5.restype = None
    L.lmzo_vec_step_v5.argtypes = [vp, i64, vp, u8p] + [vp] * 7
    L.lmzo_vec_step_v5.restype = None
    L.lmzo_vec_render_v5.argtypes = [vp, i64, u8p, vp, vp, vp]
    L.lmzo_vec_render_v5.restype = None
    L.lmzo_vec_export_v5.argtypes = [vp, i64, vp]
    L.lmzo_vec_export_v5.restype = None
    L.lmzo_safe_goal_v6.argtypes = [vp, vp, ctypes.c_int, ip]
    L.lmzo_safe_goal_v6.restype = ctypes.c_int
    L.lmzo_layout_v2.argtypes = [ctypes.c_int, ctypes.c_char_p]
    L.lmzo_layout_v2.restype = ctypes.c_int
    L.lmzo_rng_spawn_v2.argtypes = [u64, u64, u32, ctypes.c_int] + [ip] * 6
    L.lmzo_rng_spawn_v2.restype = None
    _lib = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def layout(variant):
    """Rows of the maze as a list of strings."""
    L = lib()
    G = L.lmzo_layout(variant, None)
    buf = ctypes.create_string_buffer(G * G)
    L.lmzo_layout(variant, buf)
    cells = buf.raw.decode("ascii")
    return [cells[i * G:(i + 1) * G] for i in range(G)]


def layout_v2(k):
    """Rows of v2 maze k (1..5)."""
    buf = ctypes.create_string_buffer(18 * 18)
    if lib().lmzo_layout_v2(k, buf) < 0:
        raise ValueError(k)
    cells = buf.raw.decode("ascii")
    return [cells[i * 18:(i + 1) * 18] for i in range(18)]


def philox(ctr, key):
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().lmzo_philox4x32_10(_ptr(c), _ptr(k), _ptr(out))
    return out


def rng_spawn(variant, seed, env_id, episode):
    v = [ctypes.c_int() for _ in range(4)]
    lib().lmzo_rng_spawn(variant, seed, env_id, episode, *[ctypes.byref(x) for x in v])
    return tuple(x.value for x in v)  # sx, sy, gx, gy


def rng_action(seed, env_id, t):
    return lib().lmzo_rng_action(seed, env_id, t)


def rng_action25(seed, env_id, t):
    return lib().lmzo_rng_action25(seed, env_id, t)


def rng_hier(seed, env_id, t):
    g, a = ctypes.c_int(), ctypes.c_int()
    lib().lmzo_rng_hier(seed, env_id, t, ctypes.byref(g), ctypes.byref(a))
    return g.value, a.value


class OracleVec(object):
    """N independent oracle envs with the framework's batched semantics.

    step(): per env -- reference step; record f32 reward + done; if done and
    autoreset, reference reset at the injected (or Philox-spec) cells; then the
    reference render.  Mirrors gym_lmaze_b200.envs.LmazeVecCuda so parity tests can
    drive both with the same calls.
    """

    def __init__(self, variant, n, seed=0, env_id0=0, autoreset=True, threads=1, random_ball=True, random_goal=True,
                 lazy_init=False):
        """lazy_init: leave the envs zeroed for the first reset() to initialise (on all threads): for large batches,
        whose env-by-env initialisation from Python takes seconds.  Call reset() before anything else then."""
        self.L = lib()
        self.variant, self.n, self.seed, self.env_id0 = variant, int(n), int(seed), int(env_id0)
        self.autoreset, self.threads = bool(autoreset), int(threads)
        self.env_bytes = self.L.lmzo_sizeof_env()
        self._mem = np.zeros(self.n * self.env_bytes, dtype=np.uint8)  # zero => lazily lmzo_init'ed
        assert not lazy_init or (random_ball and random_goal)
        for i in range(0 if lazy_init else self.n):
            self.L.lmzo_init(self._env(i), variant)
            if not (random_ball and random_goal):
                self.L.lmzo_env_set_flags(self._env(i), int(random_ball), int(random_goal))
        self.episode = np.zeros(self.n, dtype=np.uint32)
        self.stats = np.zeros(NUM_STATS, dtype=np.int64)
        self.obs_shape = OBS_SHAPE[variant]

    def _env(self, i):
        return self._mem.ctypes.data + i * self.env_bytes

    @staticmethod
    def _spawn_arr(spawn, n):
        if spawn is None:
            return None
        s = np.ascontiguousarray(spawn, dtype=np.int32)
        assert s.shape == (n, 4), s.shape
        return s

    def reset(self, spawn=None, want_obs=True):
        s = self._spawn_arr(spawn, self.n)
        obs = np.empty((self.n,) + self.obs_shape, dtype=np.float32) if want_obs else None
        self.L.lmzo_vec_reset(_ptr(self._mem), self.n, self.variant, _ptr(s), self.seed, self.env_id0,
                              _ptr(self.episode), _ptr(obs), self.threads)
        return obs

    def step(self, actions, spawn=None, want_obs=True, obs_out=None):
        a = np.ascontiguousarray(actions, dtype=np.int64)
        assert a.shape == (self.n,)
        s = self._spawn_arr(spawn, self.n)
        obs = obs_out if obs_out is not None else (
            np.empty((self.n,) + self.obs_shape, dtype=np.float32) if want_obs else None)
        reward = np.empty(self.n, dtype=np.float32)
        done = np.empty(self.n, dtype=np.uint8)
        self.L.lmzo_vec_step(_ptr(self._mem), self.n, _ptr(a), _ptr(s), self.seed, self.env_id0,
                             _ptr(self.episode), int(self.autoreset), _ptr(obs), _ptr(reward), _ptr(done),
                             _ptr(self.stats), self.threads)
        return obs, reward, done

    def export(self):
        pos = np.empty((self.n, 4), dtype=np.int32)
        sc = np.empty(self.n, dtype=np.int64)
        gc = np.empty(self.n, dtype=np.int64)
        rw = np.empty(self.n, dtype=np.float64)
        self.L.lmzo_vec_export(_ptr(self._mem), self.n, _ptr(pos), _ptr(sc), _ptr(gc), _ptr(rw))
        return pos, sc, gc, rw

    def force(self, i, sx, sy, gx=-1, gy=-1, step_count=0, reward=-0.0, goal_count=0):
        rc = self.L.lmzo_env_force(self._env(i), self.variant, sx, sy, gx, gy, step_count, reward, goal_count)
        if rc != 0:
            raise ValueError("oracle rejected forced state %r" % ((i, sx, sy, gx, gy),))

    def force_v2(self, i, layout, sx, sy, gx, gy, px, py, step_count=0):
        rc = self.L.lmzo_env_force_v2(self._env(i), layout, sx, sy, gx, gy, px, py, step_count)
        if rc != 0:
            raise ValueError("oracle rejected forced v2 state")

    def reset_masked(self, mask):
        """Device-RNG reset of the envs where mask is true (lmz_reset with a mask and no spawn cells)."""
        for i in np.nonzero(np.asarray(mask))[0]:
            i = int(i)
            self.L.lmzo_vec_reset(self._env(i), 1, self.variant, None, self.seed, self.env_id0 + i,
                                  self.episode.ctypes.data + 4 * i, None, 1)

    def export_visit(self):
        """v4 visit layer state[2] of every env, float32 [N, 18, 18]."""
        out = np.empty((self.n, 18, 18), dtype=np.float32)
        self.L.lmzo_vec_export_visit(_ptr(self._mem), self.n, _ptr(out))
        return out

    def set_visit(self, i, visit):
        v = np.ascontiguousarray(visit, dtype=np.float32)
        assert v.size == 324
        self.L.lmzo_env_set_visit(self._env(i), _ptr(v))

    def export_aux(self):
        """int32 [N,4]: layout, prev_x, prev_y, bad_actions (v2)."""
        aux = np.empty((self.n, 4), dtype=np.int32)
        self.L.lmzo_vec_export_aux(_ptr(self._mem), self.n, _ptr(aux))
        return aux

    # single-env access for table tests
    def step_one(self, i, action):
        cls = ctypes.c_int()
        d = self.L.lmzo_step(self._env(i), int(action), ctypes.byref(cls))
        return d, cls.value

    def render_one(self, i):
        obs = np.empty(self.obs_shape, dtype=np.float32)
        self.L.lmzo_render(self._env(i), _ptr(obs))
        return obs


class OracleHier(object):
    """N oracle envs of the planner/actor variant (lmaze-v5 / v6), batched like LmazeHierCuda."""

    def __init__(self, n, seed=0, env_id0=0, random_ball=True, random_goal=True):
        self.L = lib()
        self.n, self.seed, self.env_id0 = int(n), int(seed), int(env_id0)
        self.env_bytes = self.L.lmzo_sizeof_env()
        self._mem = np.zeros(self.n * self.env_bytes, dtype=np.uint8)
        for i in range(self.n):
            self.L.lmzo_init(self._env(i), V5)
            if not (random_ball and random_goal):
                self.L.lmzo_env_set_flags(self._env(i), int(random_ball), int(random_goal))
        self.episode = np.zeros(self.n, dtype=np.uint32)

    def _env(self, i):
        return self._mem.ctypes.data + i * self.env_bytes

    @staticmethod
    def _mask(mask, n):
        return None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8).reshape(n)

    def reset(self, spawn=None, mask=None, want_obs=True):
        s = None if spawn is None else np.ascontiguousarray(spawn, dtype=np.int32).reshape(self.n, 4)
        fov = np.zeros((self.n, 7, 35, 35), dtype=np.float32) if want_obs else None
        self.L.lmzo_vec_reset_v5(_ptr(self._mem), self.n, _ptr(self._mask(mask, self.n)), _ptr(s), self.seed,
                                 self.env_id0, _ptr(self.episode), _ptr(fov))
        return fov

    def planner_step(self, goals, mask=None):
        g = np.ascontiguousarray(goals, dtype=np.int64).reshape(self.n)
        loc = np.zeros((self.n, 4, 35, 35), dtype=np.float32)
        err = np.zeros(self.n, dtype=np.uint8)
        self.L.lmzo_vec_planner_v5(_ptr(self._mem), self.n, _ptr(g), _ptr(self._mask(mask, self.n)), _ptr(loc), _ptr(err))
        return loc, err

    def step(self, actions, mask=None):
        a = np.ascontiguousarray(actions, dtype=np.int64).reshape(self.n)
        fov = np.zeros((self.n, 7, 35, 35), dtype=np.float32)
        loc = np.zeros((self.n, 4, 35, 35), dtype=np.float32)
        gr = np.zeros(self.n, np.float32); lr = np.zeros(self.n, np.float32)
        gd = np.zeros(self.n, np.uint8); ld = np.zeros(self.n, np.uint8); err = np.zeros(self.n, np.uint8)
        self.L.lmzo_vec_step_v5(_ptr(self._mem), self.n, _ptr(a), _ptr(self._mask(mask, self.n)), _ptr(fov), _ptr(loc),
                                _ptr(gr), _ptr(lr), _ptr(gd), _ptr(ld), _ptr(err))
        return fov, loc, gr, lr, gd, ld, err

    def render(self, mask=None, fov=None, loc=None):
        """Both observations of the current state (rows where mask is false are left as passed in / zero)."""
        fov = np.zeros((self.n, 7, 35, 35), dtype=np.float32) if fov is None else fov
        loc = np.zeros((self.n, 4, 35, 35), dtype=np.float32) if loc is None else loc
        err = np.zeros(self.n, dtype=np.uint8)
        self.L.lmzo_vec_render_v5(_ptr(self._mem), self.n, _ptr(self._mask(mask, self.n)), _ptr(fov), _ptr(loc), _ptr(err))
        return fov, loc, err

    def export(self):
        out = np.zeros((self.n, 16), dtype=np.int32)
        self.L.lmzo_vec_export_v5(_ptr(self._mem), self.n, _ptr(out))
        return out

    def export_visit(self):
        out = np.empty((self.n, 18, 18), dtype=np.float32)
        self.L.lmzo_vec_export_visit(_ptr(self._mem), self.n, _ptr(out))
        return out

    def safe_goal(self, i, draws):
        d = np.ascontiguousarray(draws, dtype=np.int64)
        used = ctypes.c_int()
        return self.L.lmzo_safe_goal_v6(self._env(i), _ptr(d), len(d), ctypes.byref(used)), used.value
