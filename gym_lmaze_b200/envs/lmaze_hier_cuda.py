"""LmazeHierCuda -- the reference's two-level planner / actor env over N mazes on one B200.

Host-side mirror of LmazeEnv_v5 (reference gym_lmaze/envs/lmaze_env_v5.py:17-712) and LmazeEnv_v6
(lmaze_env_v6.py, = v5 + safeFovealGoal, :505-523).  Same protocol and method names, batched:

    fov = env.reset()                      # foveal obs  f32 [N, 7, 35, 35]          (lmaze_env_v5.py:102-153)
    loc = env.plannerStep(goals, mask)     # local obs   f32 [N, 4, 35, 35]          (:158-182)
    fov, loc, globalReward, originalReward, globalDone, localDone, fovealGoal, action = env.step(actions)   (:187-292)

`plannerStep` acts on the envs where `mask` is true (None = all): the caller passes the envs whose local
episode just ended (`localDone | globalDone` with autoreset).  `step` advances every env.  All arithmetic
runs in the CUDA kernel behind the C ABI (include/lmaze_b200.h); this class only owns tensors.
"""
import ctypes

import torch

from .. import _abi
from .lmaze_vec_cuda import LmazeVecCuda, _ACTION_DTYPES, _VARIANTS


class LmazeHierCuda(LmazeVecCuda):
    _batched = "LmazeHierCuda"

    def __init__(self, num_envs=1, variant="v5", device=None, seed=0, autoreset=True, env_id0=0, random_ball=True,
                 random_goal=True, tune=None, obs_mode="full"):
        if variant not in _VARIANTS or _VARIANTS[variant][2] != self._batched:
            raise ValueError("LmazeHierCuda is the planner/actor env: variant must be 'v5' or 'v6'")
        self.variant_name = _VARIANTS[variant][0]
        super().__init__(num_envs, variant, device=device, seed=seed, autoreset=autoreset, env_id0=env_id0,
                         random_ball=random_ball, random_goal=random_goal, tune=tune, obs_mode=obs_mode)
        shape = (ctypes.c_int64 * 3)()
        _abi.check(self._lib.lmz_local_obs_shape(self.variant, ctypes.byref(shape)))
        self.full_local_obs_shape = tuple(shape)
        # obs_mode="compact": both observations are the 5x5 crops before the x7 upsample (f32 [N,7,5,5] / [N,4,5,5])
        self.local_obs_shape = tuple(shape) if obs_mode == "full" else (shape[0], 5, 5)
        n, dev = self.num_envs, self.device
        self.loc_obs = self._obs_tensor((n,) + self.local_obs_shape, torch.float32).zero_()
        self.local_reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self._ldone_u8 = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.local_done = self._ldone_u8.view(torch.bool)
        self._loc_err_u8 = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.loc_err = self._loc_err_u8.view(torch.bool)
        self.foveal_goal = torch.full((n,), 12, dtype=torch.uint8, device=dev)      # hot cell of fovealGoal
        _abi.call(self._lib.lmz_bind_local_dl, self._h, self.loc_obs, self.local_reward, self._ldone_u8,
                  self._loc_err_u8, self.foveal_goal)
        self.global_reward, self.global_done, self.fov_obs = self.reward, self.done, self.obs
        self.step_limit, self.foveal_step_limit = 10, 50                           # lmaze_env_v5.py:47-48

    # ------------------------------------------------------------------ protocol
    def plannerStep(self, goals, mask=None):
        """Reference plannerStep (lmaze_env_v5.py:158-182) for the envs where mask is true; returns the local obs.
        mask="auto": the envs that are waiting for their planner (localDone set, or no plannerStep since their
        last reset) -- decided on the device, no host round trip."""
        goals = self._as_actions(goals)
        if isinstance(mask, str):
            if mask != "auto":
                raise ValueError("mask must be a tensor, None or 'auto'")
            _abi.call(self._lib.lmz_planner_step_auto_dl, self._h, goals, self._stream())
            return self.loc_obs
        if mask is not None:
            mask = torch.as_tensor(mask).to(device=self.device).to(torch.uint8).contiguous()
        _abi.call(self._lib.lmz_planner_step_dl, self._h, goals, mask, self._stream())
        return self.loc_obs

    planner_step = plannerStep

    def expand_local(self, loc=None):
        """Compact local obs f32 [n,4,5,5] -> the reference's [n,4,35,35] image (exact x7 replication)."""
        loc = self.loc_obs if loc is None else loc
        if loc.shape[-1] == self.full_local_obs_shape[-1]:
            return loc
        return loc.repeat_interleave(7, dim=2).repeat_interleave(7, dim=3)

    def goal_plane(self):
        """fovealGoal as the reference returns it: f32 [N, 1, 5, 5] one-hot (lmaze_env_v5.py:165-168)."""
        return torch.nn.functional.one_hot(self.foveal_goal.long(), 25).to(torch.float32).view(-1, 1, 5, 5)

    def step(self, actions, spawn=None, goal_plane=True):
        """Reference step (lmaze_env_v5.py:187-292), batched 8-tuple.  `loc_err` marks the envs where the
        reference's buildLocalObservation would raise IndexError (their local rows are zeros)."""
        actions = self._step(actions, spawn)
        return (self.obs, self.loc_obs, self.reward, self.local_reward, self.done, self.local_done,
                self.goal_plane() if goal_plane else self.foveal_goal, actions)

    def safeFovealGoal(self, draws=None):
        """lmaze-v6 safeFovealGoal (lmaze_env_v6.py:505-523): per env a goal 0..24 whose window cell is not a
        wall.  draws: optional int64 [N, K] = the values np.random.randint(0, 25) would return, consumed until
        a non-wall cell comes up; then returns (goals, used).  Default: device RNG, returns goals u8 [N]."""
        goals = torch.empty(self.num_envs, dtype=torch.uint8, device=self.device)
        if draws is None:
            _abi.call(self._lib.lmz_safe_goal_dl, self._h, None, goals, None, self._stream())
            return goals
        draws = torch.as_tensor(draws).to(device=self.device, dtype=torch.int64).contiguous()
        used = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        _abi.call(self._lib.lmz_safe_goal_dl, self._h, draws, goals, used, self._stream())
        return goals, used

    safe_foveal_goal = safeFovealGoal

    def step_host(self, goals_host, actions_host, greward_host, lreward_host, gdone_host, ldone_host):
        """End-to-end planner + actor step with HOST buffers (pinned CPU tensors): H2D goals and actions,
        plannerStep(mask="auto") + step, D2H both rewards and both done flags, stream synchronised on return."""
        ad = self._host_buffer("actions_host", actions_host, _ACTION_DTYPES)
        if self._host_buffer("goals_host", goals_host, _ACTION_DTYPES) != ad:
            raise ValueError("goals_host must have actions_host's dtype")
        self._host_buffer("greward_host", greward_host, (torch.float32,))
        self._host_buffer("lreward_host", lreward_host, (torch.float32,))
        self._host_buffer("gdone_host", gdone_host)
        self._host_buffer("ldone_host", ldone_host)
        _abi.check(self._lib.lmz_hier_step_host(
            self._h, goals_host.data_ptr(), actions_host.data_ptr(), ad, greward_host.data_ptr(),
            lreward_host.data_ptr(), gdone_host.data_ptr(), ldone_host.data_ptr(), self._stream()))
        return greward_host, lreward_host, gdone_host, ldone_host

    def rollout(self, T, goals=None, actions=None):
        """T fused planner + actor steps, no per-step observations (lmz_hier_rollout): per step plannerStep(goals[t])
        for the envs waiting for their planner, then step(actions[t]).  goals / actions: [T, N] of one integer dtype,
        or both None for device-side random ones.  Returns (globalReward f32, originalReward f32, globalDone bool,
        localDone bool), each [T, N]."""
        T = int(T)
        if (goals is None) != (actions is None):
            raise ValueError("give both goals and actions, or neither")
        if goals is not None:
            goals, actions = self._as_actions(goals), self._as_actions(actions)
            if goals.dtype != actions.dtype:
                goals = goals.to(actions.dtype)
        n, dev = self.num_envs, self.device
        gr = torch.empty((T, n), dtype=torch.float32, device=dev)
        lr = torch.empty((T, n), dtype=torch.float32, device=dev)
        gd = torch.empty((T, n), dtype=torch.uint8, device=dev)
        ld = torch.empty((T, n), dtype=torch.uint8, device=dev)
        _abi.call(self._lib.lmz_hier_rollout_dl, self._h, T, goals, actions, gr, lr, gd, ld, self._stream())
        return gr, lr, gd.view(torch.bool), ld.view(torch.bool)

    def _unsupported(self, *a, **k):
        raise NotImplementedError("not available for the planner/actor env (lmaze-v5/v6)")

    set_window = render_window = initState = host_pipeline = _unsupported
