"""gym_lmaze_b200 -- B200-native batched LMaze step/reset (drop-in for the hot path of gkm2708/gym-lmaze).

Keeps the reference's registration ids (reference gym_lmaze/__init__.py:3-38) for the
variants that are built and adds vectorised ids.  `make(id, num_envs=...)` works without
gym; when gym or gymnasium is importable the ids are registered there as well.
"""
from .envs import LmazeVecCuda, shard_range, allreduce_stats, INVALID_ACTION  # noqa: F401
from .envs import LmazeEnv, LmazeEnv_v2, LmazeEnv_v3, LmazeEnv_v4, LmazeEnv_v5, LmazeEnv_v6  # noqa: F401
from .envs import LmazeHierCuda  # noqa: F401
from .envs.lmaze_vec_cuda import _VARIANTS

__version__ = "0.1.0"

# id -> (variant, default kwargs).  'lmaze-vK' are the reference's ids; 'lmaze-vec-vK' the batched ones.
_REGISTRY = {}


def register(id, variant, **defaults):
    _REGISTRY[id] = (variant, defaults)


_SINGLE = {"v0": LmazeEnv, "v2": LmazeEnv_v2, "v3": LmazeEnv_v3, "v4": LmazeEnv_v4, "v5": LmazeEnv_v5, "v6": LmazeEnv_v6}


def make(id, **kwargs):
    """'lmaze-vK' -> the reference's single-maze surface (numpy obs, float reward, bool done, action);
    'lmaze-vec-vK' (or num_envs=...) -> the batched LmazeVecCuda."""
    if id not in _REGISTRY:
        raise KeyError("unknown env id %r; built ids: %s" % (id, ", ".join(sorted(_REGISTRY))))
    variant, defaults = _REGISTRY[id]
    kw = dict(defaults)
    kw.update(kwargs)
    if "-vec-" not in id and "num_envs" not in kwargs:
        kw.pop("num_envs", None)
        return _SINGLE[variant](**kw)
    return globals()[_VARIANTS[variant][2]](variant=variant, **kw)      # the class gym_entry_point(id) names


def registered_ids():
    return sorted(_REGISTRY)


register("lmaze-v0", "v0", num_envs=1)
register("lmaze-v2", "v2", num_envs=1)
register("lmaze-v3", "v3", num_envs=1)
register("lmaze-v4", "v4", num_envs=1)
register("lmaze-v5", "v5", num_envs=1)
register("lmaze-v6", "v6", num_envs=1)
register("lmaze-vec-v5", "v5", num_envs=4096)
register("lmaze-vec-v6", "v6", num_envs=4096)
register("lmaze-vec-v0", "v0", num_envs=4096)
register("lmaze-vec-v2", "v2", num_envs=4096)
register("lmaze-vec-v3", "v3", num_envs=4096)
register("lmaze-vec-v4", "v4", num_envs=4096)


def gym_entry_point(env_id):
    """(entry_point, kwargs) registered with gym for `env_id`.  The reference's ids 'lmaze-vK' point at the
    reference-typed single-maze classes (reference gym_lmaze/__init__.py:3-38: 'gym_lmaze.envs:LmazeEnv', ...),
    so gym.make('lmaze-v0') and gym_lmaze_b200.make('lmaze-v0') return the same kind of object; only the
    'lmaze-vec-vK' ids construct the batched classes."""
    variant, defaults = _REGISTRY[env_id]
    if "-vec-" in env_id:
        return "gym_lmaze_b200:" + _VARIANTS[variant][2], dict(defaults, variant=variant)
    return "gym_lmaze_b200:" + _SINGLE[variant].__name__, {}


def register_with(register_fn):
    """Register every built id through `register_fn(id=..., entry_point=..., kwargs=...)` (gym's or gymnasium's
    `register`).  A failing id (e.g. a clash with an installed reference package) is reported, not hidden."""
    import warnings
    done = []
    for env_id in sorted(_REGISTRY):
        entry_point, kwargs = gym_entry_point(env_id)
        try:
            register_fn(id=env_id, entry_point=entry_point, kwargs=kwargs)
            done.append(env_id)
        except Exception as exc:
            warnings.warn("gym_lmaze_b200: could not register %r with gym: %r" % (env_id, exc), RuntimeWarning)
    return done


def _register_with_gym():
    import importlib
    for modname in ("gymnasium", "gym"):
        try:
            mod = importlib.import_module(modname + ".envs.registration")
        except ImportError:
            continue                     # that package is not installed: nothing to register with
        register_with(mod.register)


_register_with_gym()
