"""ctypes binding of include/lmaze_b200.h + DLPack capsule plumbing.

The shared library is the product: if it cannot be loaded this module raises --
there is no Python or CPU fallback for the env path.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LMAZE_B200_LIB") or os.path.join(_PKG, "liblmaze_b200.so")   # override: tuning builds only

LMZ_V0, LMZ_V2, LMZ_V3, LMZ_V4, LMZ_V5 = 0, 2, 3, 4, 5
RENDER_TMA, RENDER_ST128, RENDER_INCREMENTAL = 0, 1, 2
OBS_FULL, OBS_COMPACT, OBS_BITS = 0, 1, 2
NUM_STATS = 8
SPAWN_FORCE = 64          # LMZ_SPAWN_FORCE
OBS_MEM_COMPRESSIBLE = 1  # LMZ_OBS_MEM_COMPRESSIBLE
STAT_NAMES = ("steps", "episodes", "goals", "timeouts", "wall_bumps", "moves", "stale", "eplen_sum")
STATE_COLS = ("x", "y", "goal_x", "goal_y", "step_count", "reward_code", "goal_count", "episode")
STATE_COLS_HIER = ("x", "y", "prev_x", "prev_y", "fovea_x1", "fovea_y1", "goal_x", "goal_y", "fgoal_x", "fgoal_y",
                   "last_x", "last_y", "fgoal_action", "step_count", "foveal_step_count", "flags", "episode")

class LmzConfig(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_int32),
        ("variant", ctypes.c_int32),
        ("num_envs", ctypes.c_int64),
        ("env_id0", ctypes.c_int64),
        ("seed", ctypes.c_uint64),
        ("device", ctypes.c_int32),
        ("autoreset", ctypes.c_int32),
        ("random_ball", ctypes.c_int32),
        ("random_goal", ctypes.c_int32),
        ("render_mode", ctypes.c_int32),
        ("tune", ctypes.c_int32 * 4),
        ("obs_mode", ctypes.c_int32),
        ("reserved", ctypes.c_int32 * 2),
    ]


class LmzError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("lmaze_b200 error %d: %s" % (code, message))
        self.code = code


_vp, _i32, _i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
_SHAPE = ctypes.POINTER(_i64 * 3)

# export -> argtypes, or (argtypes, restype) where it does not return int: every symbol include/lmaze_b200.h declares
# (tests/test_abi_cpu.py checks the header against EXPORTS)
_PROTOTYPES = {
    "lmz_abi_version": [],
    "lmz_last_error": ([], ctypes.c_char_p),
    "lmz_default_config": ([ctypes.POINTER(LmzConfig)], None),
    "lmz_obs_shape": [_i32, _SHAPE],
    "lmz_grid_size": [_i32],
    "lmz_obs_desc": [_i32, _i32, _SHAPE, ctypes.POINTER(_i32)],
    "lmz_layout": [_i32, ctypes.c_char_p],
    "lmz_num_layouts": [_i32],
    "lmz_layout_ex": [_i32, _i32, ctypes.c_char_p],
    "lmz_num_actions": [_i32],
    "lmz_set_window": [_vp, _vp, _i64, _i64],
    "lmz_set_window_dl": [_vp, _vp, _i64],
    "lmz_create": [ctypes.POINTER(LmzConfig), ctypes.POINTER(_vp)],
    "lmz_destroy": [_vp],
    "lmz_alloc_obs": [_i32, _i64, _i32, ctypes.POINTER(_vp), ctypes.POINTER(_i64)],
    "lmz_free_obs": [_vp],
    "lmz_bind": [_vp, _vp, _vp, _vp],
    "lmz_bind_dl": [_vp, _vp, _vp, _vp],
    "lmz_reset": [_vp, _vp, _vp, _vp],
    "lmz_reset_dl": [_vp, _vp, _vp, _vp],
    "lmz_step": [_vp, _vp, _i32, _vp, _vp],
    "lmz_step_dl": [_vp, _vp, _vp, _vp],
    "lmz_step_host": [_vp, _vp, _i32, _vp, _vp, _vp, _vp],
    "lmz_step_host_async": [_vp, _vp, _i32, _vp, _vp, _vp, _vp, ctypes.POINTER(_i32)],
    "lmz_step_host_wait": [_vp, _i32],
    "lmz_render": [_vp, _vp],
    "lmz_rollout": [_vp, _i32, _vp, _i32, _vp, _vp, _vp],
    "lmz_rollout_dl": [_vp, _i32, _vp, _vp, _vp, _vp],
    "lmz_rollout_codes": [_vp, _i32, _vp, _i32, _vp, _vp, _vp],
    "lmz_rollout_codes_dl": [_vp, _i32, _vp, _vp, _vp, _vp],
    "lmz_get_state": [_vp, _vp, _vp],
    "lmz_set_state": [_vp, _vp, _vp],
    "lmz_get_state_dl": [_vp, _vp, _vp],
    "lmz_set_state_dl": [_vp, _vp, _vp],
    "lmz_get_visit": [_vp, _vp, _vp],
    "lmz_set_visit": [_vp, _vp, _vp],
    "lmz_get_visit_dl": [_vp, _vp, _vp],
    "lmz_set_visit_dl": [_vp, _vp, _vp],
    "lmz_stats": [_vp, ctypes.POINTER(_i64 * NUM_STATS), ctypes.POINTER(_i64), _vp],
    "lmz_stats_reset": [_vp, _vp],
    "lmz_launch_count": ([_vp], _i64),
    "lmz_state_cols": [_i32],
    "lmz_local_obs_shape": [_i32, _SHAPE],
    "lmz_bind_local": [_vp] * 6,
    "lmz_bind_local_dl": [_vp] * 6,
    "lmz_planner_step": [_vp, _vp, _i32, _vp, _vp],
    "lmz_planner_step_dl": [_vp, _vp, _vp, _vp],
    "lmz_safe_goal": [_vp, _vp, _i32, _vp, _vp, _vp],
    "lmz_safe_goal_dl": [_vp, _vp, _vp, _vp, _vp],
    "lmz_planner_step_auto": [_vp, _vp, _i32, _vp],
    "lmz_planner_step_auto_dl": [_vp, _vp, _vp],
    "lmz_hier_step_host": [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp],
    "lmz_hier_rollout": [_vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp],
    "lmz_hier_rollout_dl": [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
}
EXPORTS = tuple(_PROTOTYPES)


_lib = None


def load():
    """dlopen the in-tree CUDA library and declare its prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `python -m gym_lmaze_b200.build` (needs nvcc, sm_100a). "
            "gym_lmaze_b200 has no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    for name, proto in _PROTOTYPES.items():
        fn = getattr(L, name)
        fn.argtypes, fn.restype = proto if isinstance(proto, tuple) else (proto, ctypes.c_int)
    if L.lmz_abi_version() != 1:
        raise ImportError("liblmaze_b200.so ABI version %d, binding expects 1" % L.lmz_abi_version())
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise LmzError(rc, (load().lmz_last_error() or b"").decode("utf-8", "replace"))


# ---- DLPack: borrow the DLManagedTensor* out of a "dltensor" capsule -------------
_PyCapsule_GetPointer = ctypes.pythonapi.PyCapsule_GetPointer
_PyCapsule_GetPointer.restype = ctypes.c_void_p
_PyCapsule_GetPointer.argtypes = [ctypes.py_object, ctypes.c_char_p]


def dl(tensor):
    """(pointer-or-None, capsule) for an optional tensor argument: the pointer is valid while the capsule lives.

    The capsule is never renamed to "used_dltensor", so when it is collected
    PyTorch's capsule destructor calls the DLManagedTensor deleter itself -- the
    shim never takes ownership (include/lmaze_b200.h conventions).
    """
    if tensor is None:
        return None, None
    capsule = tensor.__dlpack__()
    return _PyCapsule_GetPointer(capsule, b"dltensor"), capsule


_TYPESTR = {"torch.float32": "<f4", "torch.uint8": "|u1"}     # the observation dtypes


class _ObsMemory(object):
    """One lmz_alloc_obs allocation, shown to torch through __cuda_array_interface__.  torch holds this object for as
    long as any tensor or view of the memory lives; dropping the last one returns the memory at once (lmz_free_obs),
    whatever became of the env handle it was bound to."""

    def __init__(self, lib, device, shape, dtype, compressible):
        nbytes = dtype.itemsize
        for d in shape:
            nbytes *= int(d)
        ptr, granted = ctypes.c_void_p(), ctypes.c_int64()
        check(lib.lmz_alloc_obs(device, nbytes, OBS_MEM_COMPRESSIBLE if compressible else 0, ctypes.byref(ptr),
                                ctypes.byref(granted)))
        self._free, self.ptr, self.compressed_bytes = lib.lmz_free_obs, ptr.value, granted.value
        self.__cuda_array_interface__ = {"shape": tuple(int(d) for d in shape), "typestr": _TYPESTR[str(dtype)],
                                         "data": (ptr.value, False), "version": 2}

    def __del__(self):
        self._free(self.ptr)


def obs_empty(shape, dtype, device, compressible):
    """(tensor, compressed bytes): an uninitialised tensor like torch.empty(shape, dtype=dtype, device=device) in
    memory from lmz_alloc_obs, compressible where the device and driver grant it."""
    import torch
    device = torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    mem = _ObsMemory(load(), device.index, shape, dtype, compressible)
    return torch.as_tensor(mem, device=device), mem.compressed_bytes


def call(fn, *args):
    """fn(*args) for an lmz_*_dl export, raising LmzError if it fails.  Each tensor argument goes in as a borrowed
    DLPack capsule that stays alive until fn returns; None and the other arguments are passed as they are."""
    borrowed = [dl(a) if hasattr(a, "__dlpack__") else (a, None) for a in args]
    check(fn(*[p for p, _ in borrowed]))
