"""LmazeVecCuda -- the reference's gym Env surface over N mazes on one B200.

Host-side mirror of the reference classes for the hot path:
  variant "v0" <-> LmazeEnv     (reference gym_lmaze/envs/lmaze_env.py:11-256)
  variant "v3" <-> LmazeEnv_v3  (reference gym_lmaze/envs/lmaze_env_v3.py:17-402)
  variant "v2" <-> LmazeEnv_v2  (reference gym_lmaze/envs/lmaze_env_v2.py:17-405; Discrete(25), obs (5,35,35))
  variant "v4" <-> LmazeEnv_v4  (reference gym_lmaze/envs/lmaze_env_v4.py:17-482; v2 + float visit layer, obs (7,35,35))

Same method names and argument meaning -- `reset()` returns the observation,
`step(action)` returns `(obs, reward, done, info)` (old-gym 4-tuple,
lmaze_env.py:237), `action_space` / `observation_space` are the reference's
(`Discrete(4)`, `Box(0, 1, (4, 84, 84))`, lmaze_env.py:16,20) -- but every value is
a batch: obs `float32 [N, C, H, W]`, reward `float32 [N]`, done `bool [N]` CUDA
tensors.  This module only owns tensors and forwards to the C ABI
(include/lmaze_b200.h) through ctypes with tensors exchanged as DLPack capsules;
all env arithmetic happens in the CUDA kernels.  There is no CPU path.
"""
import ctypes

import torch

from .. import _abi
from ..spaces import make_spaces

# every accepted variant spelling -> (name, ABI id, batched class).  v6 is v5 plus safeFovealGoal: one ABI variant.
_VARIANTS = {spelling: (name, abi_id, batched)
             for name, abi_id, batched in (("v0", _abi.LMZ_V0, "LmazeVecCuda"), ("v2", _abi.LMZ_V2, "LmazeVecCuda"),
                                           ("v3", _abi.LMZ_V3, "LmazeVecCuda"), ("v4", _abi.LMZ_V4, "LmazeVecCuda"),
                                           ("v5", _abi.LMZ_V5, "LmazeHierCuda"), ("v6", _abi.LMZ_V5, "LmazeHierCuda"))
             for spelling in (name, int(name[1:]), "lmaze-" + name)}
_RENDER = {"tma": _abi.RENDER_TMA, "st128": _abi.RENDER_ST128, "incremental": _abi.RENDER_INCREMENTAL}
_OBS_MODE = {"full": _abi.OBS_FULL, "compact": _abi.OBS_COMPACT, "bits": _abi.OBS_BITS}
# lmaze_env_v3.py:236-247 -- the strings v3's step() accepts; anything else is its unmatched branch
_V3_WORDS = {"left": 0, "0": 0, "right": 1, "1": 1, "up": 2, "2": 2, "down": 3, "3": 3}
INVALID_ACTION = 255
_ACTION_DTYPES = (torch.uint8, torch.int32, torch.int64)


def shard_range(total_envs, rank, world_size):
    """Contiguous global-id range [lo, hi) owned by `rank` (SURVEY.md section 8e)."""
    total_envs, rank, world_size = int(total_envs), int(rank), int(world_size)
    if not (0 <= rank < world_size):
        raise ValueError("rank %d outside world of %d" % (rank, world_size))
    lo = total_envs * rank // world_size
    hi = total_envs * (rank + 1) // world_size
    return lo, hi


class _ReferenceSurface(object):
    """The reference's display hooks (lmaze_env.py:12,55-59,251-256).  cv2 display is out of scope: they only set
    the flags."""
    metadata = {"render.modes": ["human"]}

    def render(self, mode="human", close=False):
        self.VISUALIZE = (mode == "human")

    def rendering(self, msg):
        self.VISUALIZE = msg

    def writing(self, msg):
        self.SAVEFRAME = msg


class LmazeVecCuda(_ReferenceSurface):
    _batched = "LmazeVecCuda"            # the batched class _VARIANTS names for the variants this class runs

    def __init__(self, num_envs=1, variant="v0", device=None, seed=0, autoreset=True, render_mode="tma",
                 env_id0=0, random_ball=True, random_goal=True, with_obs=True, tune=None, obs_mode="full",
                 obs_window=None):
        if variant not in _VARIANTS:
            raise ValueError("unknown variant %r (built: v0, v2, v3, v4; v5/v6 through LmazeHierCuda)" % (variant,))
        if _VARIANTS[variant][2] != self._batched:
            raise ValueError("lmaze-v5/v6 is the planner/actor env: construct LmazeHierCuda")
        if render_mode not in _RENDER:
            raise ValueError("render_mode must be 'tma', 'st128' or 'incremental'")
        if obs_mode not in _OBS_MODE:
            raise ValueError("obs_mode must be 'full', 'compact' or 'bits'")
        self._lib = _abi.load()          # raises if the CUDA extension is missing: no fallback
        if not torch.cuda.is_available():
            raise RuntimeError("LmazeVecCuda needs a CUDA device; gym_lmaze_b200 has no CPU path")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.variant = _VARIANTS[variant][1]
        self.num_envs = int(num_envs)
        self.autoreset = bool(autoreset)
        self.env_id0 = int(env_id0)
        self.seed = int(seed)
        self.render_mode = render_mode
        # incremental render: True while `obs` may not hold a full render of the current state (mirrors the
        # handle's own flag); a captured graph of the incremental kernel must not be replayed then
        self._obs_desync = True

        shape = (ctypes.c_int64 * 3)()
        _abi.check(self._lib.lmz_obs_shape(self.variant, ctypes.byref(shape)))
        self.full_obs_shape = tuple(shape)               # the reference's observation_space shape
        self.obs_mode = obs_mode
        _abi.check(self._lib.lmz_obs_desc(self.variant, _OBS_MODE[obs_mode], ctypes.byref(shape), None))
        self.obs_shape = tuple(shape)                    # shape of one row of `self.obs` in this obs_mode
        if obs_mode == "bits":                           # u8 [N, R]: one bit per cell of the compact layers
            self.obs_shape = (int(shape[0]),)
        foveal = self.variant in (_abi.LMZ_V2, _abi.LMZ_V4, _abi.LMZ_V5)
        # compact observations: u8 [C,G,G] layers for the full-view variants, f32 [C,5,5] crops for the foveal ones
        self.obs_dtype = torch.float32 if (obs_mode == "full" or foveal) else torch.uint8
        self.grid_size = self._lib.lmz_grid_size(self.variant)
        self.expansion = self.full_obs_shape[1] // (5 if foveal else self.grid_size)      # the reference's expansionRatio
        self.num_actions = self._lib.lmz_num_actions(self.variant)      # Discrete(4) / Discrete(25)
        self.num_layouts = self._lib.lmz_num_layouts(self.variant)
        self._state_cols = self._lib.lmz_state_cols(self.variant)      # get_state() columns
        self.single_action_space, self.single_observation_space = make_spaces(self.num_actions, self.full_obs_shape)
        self.action_space, self.observation_space = self.single_action_space, self.single_observation_space
        self.VISUALIZE = False           # lmaze_env.py:26; cv2 display is out of scope

        cfg = _abi.LmzConfig()
        self._lib.lmz_default_config(ctypes.byref(cfg))
        cfg.variant, cfg.num_envs, cfg.env_id0 = self.variant, self.num_envs, self.env_id0
        cfg.seed, cfg.device = self.seed & 0xFFFFFFFFFFFFFFFF, self.device.index
        cfg.autoreset, cfg.random_ball, cfg.random_goal = int(autoreset), int(random_ball), int(random_goal)
        cfg.render_mode = _RENDER[render_mode]
        cfg.obs_mode = _OBS_MODE[obs_mode]
        for i, v in enumerate(tune or ()):
            cfg.tune[i] = int(v)
        handle = ctypes.c_void_p()
        _abi.check(self._lib.lmz_create(ctypes.byref(cfg), ctypes.byref(handle)))
        self._h = handle

        # caller-owned (PyTorch) output tensors, bound once; the kernels write them in place
        n = self.num_envs
        self.obs_window = n if obs_window is None else int(obs_window)
        if not (1 <= self.obs_window <= n):
            raise ValueError("obs_window must be in [1, num_envs]")
        self.window_lo = 0
        self._obs_compressed = False
        self.obs = self._obs_tensor((self.obs_window,) + self.obs_shape, self.obs_dtype) if with_obs else None
        self.reward = torch.zeros(n, dtype=torch.float32, device=self.device)
        self._done_u8 = torch.zeros(n, dtype=torch.uint8, device=self.device)
        self.done = self._done_u8.view(torch.bool)
        self._bind()

    # ------------------------------------------------------------------ plumbing
    def _obs_tensor(self, shape, dtype):
        """An uninitialised observation tensor: compressible device memory for the modes whose kernels write it
        faster there (DESIGN.md §2, observation memory), torch.empty for the others."""
        if not self._compressible_obs():
            return torch.empty(shape, dtype=dtype, device=self.device)
        t, compressed_bytes = _abi.obs_empty(shape, dtype, self.device, True)
        self._obs_compressed = compressed_bytes > 0
        return t

    def _compressible_obs(self):
        # full renders write whole rows, about half of whose 128 B lines are all zeros: +12.5 % on the v0 step, +2 to
        # +17 % on the other full renders.  The incremental kernel patches parts of lines, which compressed memory
        # turns into read-modify-writes (-73 %); compact modes stay plain until each of their kernels is measured
        return self.obs_mode == "full" and self.render_mode != "incremental"

    @property
    def obs_compressed(self):
        """True when the observation tensors this env allocated are in compressible memory (the device and driver
        granted it for this mode); a tensor bound by the caller is whatever the caller made it."""
        return self._obs_compressed

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _bind(self):
        windowed = self.obs is not None and self.obs_window < self.num_envs
        _abi.call(self._lib.lmz_bind_dl, self._h, None if windowed else self.obs, self.reward, self._done_u8)
        if windowed:
            self.set_window(0)

    def set_window(self, env_lo):
        """Point the obs buffer at envs [env_lo, env_lo + obs_window): later steps / render_obs()
        write only those rows (every env still steps).  For batches whose full observation
        tensor does not fit in HBM."""
        env_lo = int(env_lo)
        _abi.call(self._lib.lmz_set_window_dl, self._h, self.obs, env_lo)
        self._obs_desync = True
        self.window_lo = env_lo

    def render_window(self, env_lo):
        """set_window(env_lo) + render the current state of that window into `obs`."""
        self.set_window(env_lo)
        return self.render_obs()

    def expand(self, obs=None):
        """Compact u8 [n,C,G,G] (foveal variants: f32 [n,C,5,5]) or bit-packed u8 [n,R] -> the reference's f32
        [n,C,G*E,G*E] image (torch plumbing; exact, because the reference upsample is a pure xE replication,
        lmaze_env.py:219-234, and every value of the un-expanded layers is 0.0 or 1.0)."""
        obs = self.obs if obs is None else obs
        if self.obs_mode == "bits" and obs.dim() == 2:
            obs = self.unpack_bits(obs)
        if obs.shape[-1] == self.full_obs_shape[-1]:
            return obs
        e = self.expansion
        return obs.to(torch.float32).repeat_interleave(e, dim=2).repeat_interleave(e, dim=3)

    def unpack_bits(self, bits):
        """Bit-packed rows u8 [n,R] -> the compact layers u8 [n,C,G,G] (bit k%8 of byte k/8 = cell k)."""
        C, G = self.full_obs_shape[0], self.grid_size
        shifts = torch.arange(8, dtype=torch.uint8, device=bits.device)
        cells = (bits.unsqueeze(-1) >> shifts) & 1
        return cells.reshape(bits.shape[0], -1)[:, :C * G * G].reshape(bits.shape[0], C, G, G)

    def initState(self):
        """Reference initState() (lmaze_env.py:243-244): the un-expanded state layers, last reward,
        done flag and {'newState': True} -- batched: f32 [N, C*G*G].  Needs obs_mode='compact'."""
        if self.obs_mode != "compact" or self.obs_window != self.num_envs:
            raise RuntimeError("initState() needs obs_mode='compact' over the whole batch")
        state = self.render_obs().to(torch.float32).reshape(self.num_envs, -1)
        return state, self.reward, self.done, {"newState": True}

    def _as_actions(self, actions):
        """Anything the reference's `int(msg)` (lmaze_env.py:148) accepts, batched."""
        if isinstance(actions, (list, tuple)) and actions and isinstance(actions[0], str):
            actions = [_V3_WORDS.get(a, INVALID_ACTION) for a in actions]
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(actions)
        if actions.is_floating_point():
            actions = actions.to(torch.int64)            # int() truncates toward zero
        elif actions.dtype == torch.bool:
            actions = actions.to(torch.uint8)
        elif actions.dtype not in _ACTION_DTYPES:
            actions = actions.to(torch.int64)
        if actions.device != self.device:
            actions = actions.to(self.device, non_blocking=True)
        return actions.contiguous()

    def _as_spawn(self, spawn):
        if spawn is None:
            return None
        spawn = torch.as_tensor(spawn)
        if spawn.dim() == 2 and spawn.shape[1] == 2:      # v0 convenience: (x, y) only
            spawn = torch.cat([spawn, torch.full_like(spawn, -1)], dim=1)
        if spawn.dim() == 2 and spawn.shape[1] == 5:      # v2: (ball_x, ball_y, goal_x, goal_y, new_layout)
            spawn = torch.cat([spawn[:, :3], (spawn[:, 3:4] | (spawn[:, 4:5] << 5))], dim=1)
        return spawn.to(device=self.device, dtype=torch.int32).contiguous()

    # ------------------------------------------------------------------ gym surface
    def reset(self, spawn=None, mask=None, mode="train"):
        """Start new episodes (all envs, or those where `mask` is true) and return obs.

        mode="test" is the v3 reference's fixed evaluation start (lmaze_env_v3.py:145-146,154-155):
        goal (8,8), ball (7,8).

        spawn: optional int [N, 4] (ball_x, ball_y, goal_x, goal_y) -- the cells the
        reference's rejection sampling (lmaze_env.py:70-78) would have drawn; default is
        the device RNG.
        """
        if mode == "test":
            if self.variant != _abi.LMZ_V3:
                raise ValueError("reset(mode='test') exists only in lmaze-v3")
            # goal_x carries LMZ_SPAWN_FORCE: test mode beats RANDOM_BALL / RANDOM_GOAL = False (lmaze_env_v3.py:145-155)
            spawn = torch.tensor([[7, 8, 8 + _abi.SPAWN_FORCE, 8]], dtype=torch.int32).expand(self.num_envs, 4)
        spawn = self._as_spawn(spawn)
        if mask is not None:
            mask = torch.as_tensor(mask).to(device=self.device).to(torch.uint8).contiguous()
        _abi.call(self._lib.lmz_reset_dl, self._h, mask, spawn, self._stream())
        if mask is None:
            self._obs_desync = False
        return self.obs

    def step(self, actions, spawn=None):
        """One fused kernel: transition + reward + done (+ auto-reset) + obs render.

        Returns (obs, reward, done, info); `info["action"]` echoes the actions, the
        batched form of the reference returning `msg` as its 4th element
        (lmaze_env.py:237).  With autoreset the obs rows of finished envs already
        show the next episode's first observation.
        """
        actions = self._step(actions, spawn)
        return self.obs, self.reward, self.done, {"action": actions}

    def _step(self, actions, spawn):
        """Launch the fused step; returns the actions as the kernel read them."""
        actions = self._as_actions(actions)
        _abi.call(self._lib.lmz_step_dl, self._h, actions, self._as_spawn(spawn), self._stream())
        self._obs_desync = False         # a step always leaves the window fully rendered (full render when out of sync)
        return actions

    def capture_step(self, actions_buf, spawn_buf=None):
        """Capture one fused step into a CUDA graph and return `replay()`.

        `actions_buf` (and `spawn_buf`) are static device tensors: write the next actions into
        them (e.g. `actions_buf.copy_(a)`) and call `replay()`; obs / reward / done are the env's
        bound tensors.  For small batches the step is launch-bound (a 4,096-env step is ~65 us of
        GPU work), and a graph replay skips the Python + ctypes + validation cost.  The kernels
        re-arm their own work counters, so a captured launch replays correctly any number of times.

        render_mode="incremental": the captured launch is the patch kernel, which is only correct while `obs`
        holds a full render of the current state.  After set_state / rollout / set_window call render_obs()
        (or step() / reset()) before the next replay; replay() raises RuntimeError otherwise.
        """
        actions_buf = self._as_actions(actions_buf)
        spawn_buf = self._as_spawn(spawn_buf)
        if self.obs is not None:
            self.render_obs()            # warm the launch path (function attributes) without changing state
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._step(actions_buf, spawn_buf)
        self._graphs = getattr(self, "_graphs", []) + [(graph, actions_buf, spawn_buf)]
        if self.render_mode != "incremental":
            return graph.replay

        def replay():
            if self._obs_desync:
                raise RuntimeError("incremental render: obs is out of sync with the env state (set_state / rollout / "
                                   "set_window since the last render); call render_obs() before replaying the graph")
            graph.replay()
        return replay

    def step_host(self, actions_host, reward_host, done_host, obs_host=None):
        """End-to-end step with HOST buffers (pinned CPU tensors): H2D actions, fused
        step, D2H reward/done (and obs if given), stream synchronised on return."""
        ad = self._host_buffer("actions_host", actions_host, _ACTION_DTYPES)
        self._host_buffer("reward_host", reward_host, (torch.float32,))
        self._host_buffer("done_host", done_host, (torch.uint8, torch.bool))
        if obs_host is not None and (obs_host.dtype != self.obs_dtype or not obs_host.is_contiguous()
                                     or obs_host.numel() != self.obs.numel()):
            raise ValueError("obs_host must be a contiguous tensor with obs's dtype and size")
        _abi.check(self._lib.lmz_step_host(
            self._h, actions_host.data_ptr(), ad, reward_host.data_ptr(), done_host.data_ptr(),
            None if obs_host is None else obs_host.data_ptr(), self._stream()))
        self._obs_desync = False
        return reward_host, done_host

    def _host_buffer(self, name, t, dtypes=None):
        """Check one buffer of the host-step calls: a contiguous CPU tensor of num_envs elements and, unless dtypes
        is None, of one of `dtypes`.  Returns the index of its dtype there: for _ACTION_DTYPES, the ABI dtype code."""
        if t.device.type != "cpu" or not t.is_contiguous() or t.numel() != self.num_envs:
            raise ValueError("%s must be a contiguous CPU tensor of num_envs elements" % name)
        if dtypes is None:
            return None
        if t.dtype not in dtypes:
            raise ValueError("%s dtype must be %s" % (name, "/".join(str(d)[len("torch."):] for d in dtypes)))
        return dtypes.index(t.dtype)

    # f32 value of each reward code (lmaze_env.py:21-23,109): REWARD_TABLE[codes] is the reward tensor, bit for bit
    REWARD_BITS = (0x80000000, 0xBF800000, 0xBC23D70A, 0x42C80000)

    @classmethod
    def reward_table(cls, device=None):
        return torch.tensor([b - (1 << 32) if b >= (1 << 31) else b for b in cls.REWARD_BITS],
                            dtype=torch.int32, device=device).view(torch.float32)

    def rollout(self, T, actions=None, rewards=None, dones=None, reward_codes=None):
        """T fused steps, no per-step obs.  actions None => device-side random actions.
        Returns (rewards f32 [T, N], dones bool [T, N]); with reward_codes=True (or a u8 [T, N] tensor) the first
        element is the 1-byte reward code instead (0: -0.0, 1: -1.0, 2: -0.01, 3: 100.0; `reward_table()[codes]`)."""
        T = int(T)
        if actions is not None:
            actions = self._as_actions(actions)
        if dones is None:
            dones = torch.empty((T, self.num_envs), dtype=torch.uint8, device=self.device)
        dones_u8 = dones.view(torch.uint8) if dones.dtype == torch.bool else dones
        if reward_codes is not None and reward_codes is not False:
            if reward_codes is True:
                reward_codes = torch.empty((T, self.num_envs), dtype=torch.uint8, device=self.device)
            _abi.call(self._lib.lmz_rollout_codes_dl, self._h, T, actions, reward_codes, dones_u8, self._stream())
            rewards = reward_codes
        else:
            if rewards is None:
                rewards = torch.empty((T, self.num_envs), dtype=torch.float32, device=self.device)
            _abi.call(self._lib.lmz_rollout_dl, self._h, T, actions, rewards, dones_u8, self._stream())
        self._obs_desync = True          # every env moved, nothing was rendered
        return rewards, dones_u8.view(torch.bool)

    def host_pipeline(self, with_obs=True):
        """Double-buffered end-to-end stepping for a HOST consumer (lmz_step_host_async / lmz_step_host_wait)."""
        return HostPipeline(self, with_obs)

    def render_obs(self):
        """Re-render the current state into `obs` without stepping."""
        _abi.check(self._lib.lmz_render(self._h, self._stream()))
        self._obs_desync = False
        return self.obs

    # ------------------------------------------------------------------ state / stats
    def get_state(self):
        """int32 [N, 8]: _abi.STATE_COLS (x, y, goal_x, goal_y, step_count, reward_code, goal_count, episode);
        for v5/v6 int32 [N, 17]: _abi.STATE_COLS_HIER."""
        out = torch.empty((self.num_envs, self._state_cols), dtype=torch.int32, device=self.device)
        _abi.call(self._lib.lmz_get_state_dl, self._h, out, self._stream())
        return out

    def set_state(self, state):
        state = torch.as_tensor(state).to(device=self.device, dtype=torch.int32).contiguous()
        _abi.call(self._lib.lmz_set_state_dl, self._h, state, self._stream())
        self._obs_desync = True

    def get_visit(self):
        """v4: the float visit layer state[2] of every env, f32 [N, 18, 18]."""
        out = torch.empty((self.num_envs, 18, 18), dtype=torch.float32, device=self.device)
        _abi.call(self._lib.lmz_get_visit_dl, self._h, out, self._stream())
        return out

    def set_visit(self, visit):
        visit = torch.as_tensor(visit).to(device=self.device, dtype=torch.float32).contiguous()
        _abi.call(self._lib.lmz_set_visit_dl, self._h, visit, self._stream())

    def stats(self, check_errors=True):
        out = (ctypes.c_int64 * _abi.NUM_STATS)()
        err = ctypes.c_int64()
        _abi.check(self._lib.lmz_stats(self._h, ctypes.byref(out), ctypes.byref(err), self._stream()))
        if check_errors and err.value:
            raise ValueError("%d injected spawn cells were rejected (wall/goal/out of range), actions were out of "
                             "range, or set_state rows were not reachable states" % err.value)
        return dict(zip(_abi.STAT_NAMES, (int(v) for v in out)))

    def stats_reset(self):
        _abi.check(self._lib.lmz_stats_reset(self._h, self._stream()))

    def stats_allreduce(self, group=None, check_errors=True):
        """Sum of the integer episode counters over all ranks (never on the step path)."""
        import torch.distributed as dist
        local = self.stats(check_errors=check_errors)
        return allreduce_stats(local, self.device, group) if dist.is_available() and dist.is_initialized() else local

    @property
    def launch_count(self):
        return int(self._lib.lmz_launch_count(self._h))

    def layout(self, index=1):
        buf = ctypes.create_string_buffer(self.grid_size * self.grid_size)
        _abi.check(self._lib.lmz_layout_ex(self.variant, int(index), buf))
        s = buf.raw.decode("ascii")
        return [s[i * self.grid_size:(i + 1) * self.grid_size] for i in range(self.grid_size)]

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.lmz_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostStep(object):
    """Pinned host buffers one pipelined step lands in."""
    __slots__ = ("obs", "reward", "done")

    def __init__(self, obs, reward, done):
        self.obs, self.reward, self.done = obs, reward, done


class HostPipeline(object):
    """Pipeline depth 2 over lmz_step_host_async / lmz_step_host_wait: `submit(actions_host)` enqueues step k (H2D
    actions, fused step, D2H of reward / done / obs into this pipeline's pinned buffers on the handle's copy stream)
    and then waits for step k-1, whose HostStep it returns (None on the first call); `drain()` waits for the last
    one.  Step k's D2H overlaps step k+1's H2D + kernel.  obs needs obs_mode 'compact' or 'bits'; the buffers of a
    returned HostStep are overwritten by the second submit after it."""

    def __init__(self, env, with_obs=True):
        if with_obs and (env.obs is None or env.obs_mode == "full"):
            raise ValueError("a host pipeline carries compact or bit-packed observations (obs_mode='compact' / 'bits'); "
                             "use with_obs=False to keep the f32 observation on the device")
        self.env = env
        n = env.num_envs
        self.slots = [HostStep(torch.empty((n,) + env.obs_shape, dtype=env.obs_dtype).pin_memory() if with_obs else None,
                               torch.empty(n, dtype=torch.float32).pin_memory(),
                               torch.empty(n, dtype=torch.uint8).pin_memory()) for _ in range(2)]
        self._pending = None            # ticket of the step in flight
        self._keep = None
        self._k = 0                     # steps submitted (one pipeline per env handle)

    def submit(self, actions_host):
        env = self.env
        ad = env._host_buffer("actions_host", actions_host, _ACTION_DTYPES)
        ticket = ctypes.c_int32(-1)
        slot = self.slots[self._k & 1]                       # the handle alternates its two device slots the same way
        self._k += 1
        _abi.check(env._lib.lmz_step_host_async(
            env._h, actions_host.data_ptr(), ad, slot.reward.data_ptr(),
            slot.done.data_ptr(), None if slot.obs is None else slot.obs.data_ptr(), env._stream(), ctypes.byref(ticket)))
        assert self.slots[ticket.value] is slot
        prev, self._pending = self._pending, ticket.value
        keep, self._keep = self._keep, actions_host          # actions must outlive their H2D copy
        if prev is None:
            return None
        _abi.check(env._lib.lmz_step_host_wait(env._h, prev))
        del keep
        return self.slots[prev]

    def drain(self):
        if self._pending is None:
            return None
        prev, self._pending = self._pending, None
        _abi.check(self.env._lib.lmz_step_host_wait(self.env._h, prev))
        self._keep = None
        return self.slots[prev]


def allreduce_stats(local, device, group=None):
    """All-reduce a stats dict as one int64[8] message (NCCL on GPU, gloo on CPU)."""
    import torch.distributed as dist
    backend = dist.get_backend(group)
    dev = device if backend == "nccl" else torch.device("cpu")
    t = torch.tensor([local[k] for k in _abi.STAT_NAMES], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return dict(zip(_abi.STAT_NAMES, (int(v) for v in t.tolist())))
