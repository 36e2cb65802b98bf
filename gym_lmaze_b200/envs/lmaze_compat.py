"""Single-maze classes with the reference's exact call surface, backed by the CUDA path (N = 1).

    LmazeEnv      <-> reference gym_lmaze/envs/lmaze_env.py:11     ('lmaze-v0')
    LmazeEnv_v2   <-> reference gym_lmaze/envs/lmaze_env_v2.py:17  ('lmaze-v2')
    LmazeEnv_v3   <-> reference gym_lmaze/envs/lmaze_env_v3.py:17  ('lmaze-v3')
    LmazeEnv_v4   <-> reference gym_lmaze/envs/lmaze_env_v4.py:17  ('lmaze-v4')
    LmazeEnv_v5   <-> reference gym_lmaze/envs/lmaze_env_v5.py:17  ('lmaze-v5', planner / actor protocol)
    LmazeEnv_v6   <-> reference gym_lmaze/envs/lmaze_env_v6.py:17  ('lmaze-v6', v5 + safeFovealGoal)

Same returns and types as the reference: `reset()` -> numpy float32 observation, `step(a)` ->
`(obs, reward, done, info)` with reward a Python float (exactly -0.0 / -1.0 / -0.01 / 100.0), done a
bool and info the action that was passed (lmaze_env.py:237).  No auto-reset: the caller resets, and
stepping past `done` is legal, as in the reference.  The env arithmetic still runs in the CUDA
kernels (one env); only the result is copied to the host.  For throughput use LmazeVecCuda.
"""
import numpy as np
import torch

from .lmaze_vec_cuda import LmazeVecCuda, INVALID_ACTION, _ReferenceSurface, _V3_WORDS
from .lmaze_hier_cuda import LmazeHierCuda

# f32 bit pattern -> the reference's Python float (lmaze_env.py:21-23,109): the shortest decimal that reads back as
# that f32, which is the literal the reference wrote (-0.01, not the f32's -0.009999999776...)
_REWARD = {b: float(str(np.uint32(b).view(np.float32))) for b in LmazeVecCuda.REWARD_BITS}


class _OneMaze(_ReferenceSurface):
    """One env of a batched class (no auto-reset), read back with the reference's Python types."""
    _vec_class = LmazeVecCuda

    def __init__(self, device=None, seed=0, **kwargs):
        self._vec = self._vec_class(1, self._variant, device=device, seed=seed, autoreset=False, **kwargs)
        self.VISUALIZE = False
        self.reset()                                   # the reference constructors end with reset()

    def _obs(self):
        return self._vec.obs[0].cpu().numpy()          # a fresh array per call, like the reference's np.zeros

    @staticmethod
    def _reward(t):
        """A one-env f32 reward tensor -> the reference's Python float."""
        return _REWARD[int(t.view(torch.int32).item()) & 0xFFFFFFFF]

    def close(self):
        self._vec.close()

    @property
    def state_vector(self):
        """x, y, goal_x, goal_y, stepCount, ... of the single env (see LmazeVecCuda.get_state)."""
        return self._vec.get_state()[0].tolist()


class _SingleMaze(_OneMaze):
    _variant = "v0"

    def __init__(self, device=None, seed=0, **kwargs):
        super().__init__(device=device, seed=seed, **kwargs)
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space

    def reset(self, spawn=None, **kwargs):
        """spawn: optional (ball_x, ball_y[, goal_x, goal_y[, layout]]) to pin the cells the reference's
        random draws would have produced; default is the device RNG."""
        if spawn is not None:
            spawn = [list(spawn)]
        self._vec.reset(spawn=spawn, **kwargs)
        return self._obs()

    def _code(self, action):
        return int(action)                             # lmaze_env.py:148: msg = int(msg)

    def step(self, action):
        code = self._code(action)
        wire = code if 0 <= code < 255 else INVALID_ACTION     # any unmatched value takes the (0,0) branch
        self._vec.step(torch.tensor([wire], dtype=torch.uint8))
        return self._obs(), self._reward(self._vec.reward), bool(self._vec.done.item()), code      # msg = int(msg)


class LmazeEnv(_SingleMaze):
    _variant = "v0"


class LmazeEnv_v2(_SingleMaze):
    _variant = "v2"

    def step(self, action):
        code = int(action)
        if not 0 <= code <= 24:
            # the reference indexes a 5x5 array with the action (lmaze_env_v2.py:136-137)
            raise IndexError("lmaze-v2 action %d outside Discrete(25)" % code)
        return super().step(code)


class LmazeEnv_v4(LmazeEnv_v2):
    _variant = "v4"


class LmazeEnv_v3(_SingleMaze):
    _variant = "v3"

    def _code(self, action):
        # lmaze_env_v3.py:236-247: step() compares STRINGS; an int never matches and leaves the offset (0,0)
        return _V3_WORDS.get(action, INVALID_ACTION) if isinstance(action, str) else INVALID_ACTION

    def step(self, action):
        obs, r, d, _ = super().step(action)            # _code() maps the string
        return obs, r, d, action

    def reset(self, mode="train", spawn=None):
        if mode == "test":
            self._vec.reset(mode="test")
            return self._obs()
        return super().reset(spawn=spawn)


class LmazeEnv_v5(_OneMaze):
    """Reference LmazeEnv_v5: reset() -> foveal obs; plannerStep(goal) -> local obs; step(a) -> the 8-tuple
    (fovobs, locobs, globalReward, originalReward, globalDone, localDone, fovealGoal, local_action),
    lmaze_env_v5.py:285-292.  The constructor ends with reset(), like the reference's (lmaze_env_v5.py:92)."""
    _vec_class = LmazeHierCuda
    _variant = "v5"

    def __init__(self, device=None, seed=0, **kwargs):
        self.step_limit, self.foveal_step_limit = 10, 50
        super().__init__(device=device, seed=seed, **kwargs)

    def reset(self, spawn=None):
        """spawn: optional (ball_x, ball_y, goal_x, goal_y, layout) pinning the reference's random draws."""
        self._vec.reset(spawn=None if spawn is None else [list(spawn)])
        return self._obs()

    def _loc(self):
        if bool(self._vec.loc_err.item()):
            # lmaze_env_v5.py:365-366: the actor is 3 cells right of / below the planner-time fovea
            raise IndexError("index 5 is out of bounds for axis 1 with size 5")
        return self._vec.loc_obs[0].cpu().numpy()

    def plannerStep(self, goal):
        goal = int(goal)                                   # :165
        if not 0 <= goal <= 24:
            raise IndexError("lmaze-v5 foveal goal %d outside the 5x5 window" % goal)
        self._vec.plannerStep(torch.tensor([goal], dtype=torch.uint8))
        return self._loc()

    def step(self, goal):
        code = int(goal)                                   # :190
        wire = code if 0 <= code < 255 else INVALID_ACTION
        v = self._vec
        v.step(torch.tensor([wire], dtype=torch.uint8), goal_plane=False)
        return (self._obs(), self._loc(), self._reward(v.reward), self._reward(v.local_reward), bool(v.done.item()),
                bool(v.local_done.item()), v.goal_plane()[0].cpu().numpy(), code)


class LmazeEnv_v6(LmazeEnv_v5):
    _variant = "v6"

    def safeFovealGoal(self, draws=None):
        """lmaze_env_v6.py:505-523.  draws: optional list of the np.random.randint(0, 25) values to consume."""
        if draws is None:
            return int(self._vec.safeFovealGoal().item())
        goals, _ = self._vec.safeFovealGoal([list(draws)])
        return int(goals.item())
