"""CPU tier: the C-ABI library loads without a GPU, exports every symbol the header
declares, validates arguments, and refuses to run without a CUDA device (no fallback)."""
import ctypes
import os
import sys
import re

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module")
def abi():
    from gym_lmaze_b200 import build, _abi
    build.build()
    return _abi


def header_symbols():
    src = open(os.path.join(ROOT, "include", "lmaze_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lmz_[a-z_0-9]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(abi):
    L = abi.load()
    syms = header_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(L, s), "header declares %s but the library does not export it" % s
    assert sorted(abi.EXPORTS) == syms            # the binding covers the whole header
    assert L.lmz_abi_version() == 1


def test_library_is_self_contained(abi):
    """No torch / python / oracle linkage: only libc-level dependencies."""
    import subprocess
    out = subprocess.run(["ldd", abi.LIB_PATH], stdout=subprocess.PIPE, text=True).stdout
    assert "torch" not in out and "python" not in out and "oracle" not in out and "libcudart" not in out


def test_static_queries_and_layouts(abi, golden_dir):
    L = abi.load()
    shape = (ctypes.c_int64 * 3)()
    assert L.lmz_obs_shape(abi.LMZ_V0, ctypes.byref(shape)) == 0 and tuple(shape) == (4, 84, 84)
    assert L.lmz_obs_shape(abi.LMZ_V3, ctypes.byref(shape)) == 0 and tuple(shape) == (3, 72, 72)
    assert L.lmz_obs_shape(abi.LMZ_V5, ctypes.byref(shape)) == 0 and tuple(shape) == (7, 35, 35)
    assert L.lmz_local_obs_shape(abi.LMZ_V5, ctypes.byref(shape)) == 0 and tuple(shape) == (4, 35, 35)
    assert L.lmz_state_cols(abi.LMZ_V5) == 17 and L.lmz_state_cols(abi.LMZ_V0) == 8 and L.lmz_num_actions(abi.LMZ_V5) == 4
    assert L.lmz_obs_shape(7, ctypes.byref(shape)) < 0 and b"unknown variant" in L.lmz_last_error()
    z = np.load(os.path.join(golden_dir, "layouts.npz"))
    for name, variant, G in (("v0", abi.LMZ_V0, 12), ("v3", abi.LMZ_V3, 18)):
        assert L.lmz_grid_size(variant) == G
        buf = ctypes.create_string_buffer(G * G)
        assert L.lmz_layout(variant, buf) == 0
        cells = buf.raw.decode()
        assert [cells[i * G:(i + 1) * G] for i in range(G)] == [str(r) for r in z[name]]


def test_config_validation_and_no_cpu_fallback(abi):
    import torch
    L = abi.load()
    cfg = abi.LmzConfig()
    L.lmz_default_config(ctypes.byref(cfg))
    assert cfg.struct_size == ctypes.sizeof(abi.LmzConfig) and cfg.autoreset == 1 and cfg.random_ball == 1
    h = ctypes.c_void_p()
    bad = abi.LmzConfig.from_buffer_copy(cfg); bad.struct_size = 8
    assert L.lmz_create(ctypes.byref(bad), ctypes.byref(h)) == -1 and b"struct_size" in L.lmz_last_error()
    bad = abi.LmzConfig.from_buffer_copy(cfg); bad.variant = 7
    assert L.lmz_create(ctypes.byref(bad), ctypes.byref(h)) == -4
    bad = abi.LmzConfig.from_buffer_copy(cfg); bad.num_envs = 0
    assert L.lmz_create(ctypes.byref(bad), ctypes.byref(h)) == -1
    assert L.lmz_step(None, None, 0, None, None) == -1 and b"NULL" in L.lmz_last_error()
    if not torch.cuda.is_available():
        # the product path must fail loudly without a device -- never fall back to a CPU env
        assert L.lmz_create(ctypes.byref(cfg), ctypes.byref(h)) == -2
        assert b"no CPU path" in L.lmz_last_error()
        import gym_lmaze_b200 as g
        with pytest.raises(RuntimeError, match="no CPU path"):
            g.make("lmaze-v0")


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the product package may import, load or link it."""
    bad = re.compile(r"(^\s*(from|import)\s+oracle\b)|liblmaze_oracle|lmzo_|oracle\.oracle|ref_loader", re.M)
    for dirpath, _, files in os.walk(os.path.join(ROOT, "gym_lmaze_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                assert not bad.search(open(os.path.join(dirpath, f)).read()), f


def test_registry_and_spaces():
    import gym_lmaze_b200 as g
    from gym_lmaze_b200.spaces import make_spaces
    assert {"lmaze-v0", "lmaze-v3", "lmaze-vec-v0", "lmaze-vec-v3"} <= set(g.registered_ids())
    assert "lmaze-v7" not in g.registered_ids()      # the reference registers a class that does not exist
    a, o = make_spaces(4, (4, 84, 84))
    assert a.n == 4 and tuple(o.shape) == (4, 84, 84) and o.dtype == np.float32
    assert float(np.min(o.low)) == 0.0 and float(np.max(o.high)) == 1.0


def test_gym_registration_entry_points(monkeypatch):
    """The reference ids resolve to the reference-typed single-maze classes -- the class names of reference
    gym_lmaze/__init__.py:3-38 -- and only the 'lmaze-vec-*' ids to the batched classes (VERDICT r1 N3)."""
    import importlib
    import warnings
    import gym_lmaze_b200 as g
    monkeypatch.syspath_prepend(os.path.join(os.path.dirname(__file__), "_gymstub"))
    for m in [k for k in sys.modules if k == "gym" or k.startswith("gym.")]:
        monkeypatch.delitem(sys.modules, m)
    reg = importlib.import_module("gym.envs.registration")
    reg.registry.clear()
    done = g.register_with(reg.register)
    assert set(done) == set(g.registered_ids()) == set(reg.registry)
    ref_names = {"lmaze-v0": "LmazeEnv", "lmaze-v2": "LmazeEnv_v2", "lmaze-v3": "LmazeEnv_v3", "lmaze-v4": "LmazeEnv_v4",
                 "lmaze-v5": "LmazeEnv_v5", "lmaze-v6": "LmazeEnv_v6"}
    for env_id, name in ref_names.items():
        rec = reg.registry[env_id]
        assert rec["entry_point"] == "gym_lmaze_b200:" + name and rec["kwargs"] == {}
        assert getattr(g, name) is g._SINGLE[env_id[-2:]]          # what make(env_id) constructs too
    for k in ("0", "2", "3", "4"):
        rec = reg.registry["lmaze-vec-v" + k]
        assert rec["entry_point"] == "gym_lmaze_b200:LmazeVecCuda" and rec["kwargs"]["variant"] == "v" + k
    for k in ("5", "6"):
        assert reg.registry["lmaze-vec-v" + k]["entry_point"] == "gym_lmaze_b200:LmazeHierCuda"
    # a failing registration is reported, not swallowed
    def boom(**kw):
        raise RuntimeError("id clash")
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        assert g.register_with(boom) == []
    assert len(w) == len(g.registered_ids()) and "id clash" in str(w[0].message)


def test_missing_extension_fails_loudly(abi, monkeypatch):
    """No .so -> ImportError naming the build command; never a silent fallback."""
    monkeypatch.setattr(abi, "_lib", None)
    monkeypatch.setattr(abi, "LIB_PATH", os.path.join(ROOT, "gym_lmaze_b200", "does_not_exist.so"))
    with pytest.raises(ImportError, match="no CPU fallback"):
        abi.load()


def test_shard_range_partitions_the_batch():
    """Contiguous global-id shards (SURVEY 8e): disjoint, ordered, covering, sizes differ by at most one."""
    from hypothesis import example, given, settings, strategies as st
    from gym_lmaze_b200 import shard_range

    @settings(max_examples=200, deadline=None)
    @given(st.integers(0, 1 << 40), st.integers(1, 64))
    def check(total, world):
        edges = [shard_range(total, r, world) for r in range(world)]
        assert edges[0][0] == 0 and edges[-1][1] == total
        for (lo, hi), (lo2, hi2) in zip(edges, edges[1:]):
            assert lo <= hi == lo2 <= hi2
        sizes = [hi - lo for lo, hi in edges]
        assert max(sizes) - min(sizes) <= 1
    for total in (1, 7, 4096, 1_000_000, 16_000_000):      # batch sizes in use, over the world sizes of one node
        for world in (1, 2, 3, 4, 8):
            check = example(total, world)(check)
    check()
    with pytest.raises(ValueError):
        shard_range(10, 3, 3)
