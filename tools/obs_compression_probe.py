#!/usr/bin/env python
"""Does compressible device memory speed up the observation writes?  (GPU box only; Python + ctypes, no library change)

Observation tensors are about half whole lines of zeros (v0 full render: 54.5 % of the aligned 128 B chunks).  Memory
made with cuMemCreate and allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC lets the L2 store such lines
compressed, so fewer bytes reach DRAM.  This probe allocates that memory through libcuda directly, wraps it as a torch
tensor (__cuda_array_interface__), binds it with lmz_bind_dl and times, plain against compressible:
  - what the device and driver grant: the attribute, the granularity, the compression actually granted for one
    2^20-env v0 obs tensor (whole, and in chunks), the device memory it costs;
  - raw write ceilings on 8 GiB: zero_(), fill_(1.0), a copy of real v0 observations tiled over the buffer; obs.sum();
  - the real kernels: one handle per mode whose obs is rebound between a plain and a compressible tensor, alternated;
  - with --sweep: the tune[0..3] launch knobs of the v0 / v3 full render on compressible memory.
    python tools/obs_compression_probe.py OUT.json [--sweep]"""
import ctypes
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import gym_lmaze_b200 as lmz            # noqa: E402
from gym_lmaze_b200 import _abi         # noqa: E402

CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = 107
CU_MEM_ALLOCATION_TYPE_PINNED = 1
CU_MEM_LOCATION_TYPE_DEVICE = 1
CU_MEM_ALLOCATION_COMP_GENERIC = 1
CU_MEM_ACCESS_FLAGS_PROT_READWRITE = 3
CU_MEM_ALLOC_GRANULARITY_RECOMMENDED = 1


class AllocFlags(ctypes.Structure):
    _fields_ = [("compressionType", ctypes.c_ubyte), ("gpuDirectRDMACapable", ctypes.c_ubyte),
                ("usage", ctypes.c_ushort), ("reserved", ctypes.c_ubyte * 4)]


class Location(ctypes.Structure):
    _fields_ = [("type", ctypes.c_int), ("id", ctypes.c_int)]


class AllocProp(ctypes.Structure):
    _fields_ = [("type", ctypes.c_int), ("requestedHandleTypes", ctypes.c_int), ("location", Location),
                ("win32HandleMetaData", ctypes.c_void_p), ("allocFlags", AllocFlags)]


class AccessDesc(ctypes.Structure):
    _fields_ = [("location", Location), ("flags", ctypes.c_int)]


cu = ctypes.CDLL("libcuda.so.1")
CHUNK = None              # physical chunk size of the compressible buffers: the one that got compression granted
_u64 = ctypes.c_uint64


def ck(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed: CUresult %d" % (what, rc))


def prop_for(dev, compress):
    p = AllocProp()
    p.type, p.location.type, p.location.id = CU_MEM_ALLOCATION_TYPE_PINNED, CU_MEM_LOCATION_TYPE_DEVICE, dev
    p.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC if compress else 0
    return p


def granularity(dev, compress):
    g = ctypes.c_size_t()
    ck(cu.cuMemGetAllocationGranularity(ctypes.byref(g), ctypes.byref(prop_for(dev, compress)),
                                        CU_MEM_ALLOC_GRANULARITY_RECOMMENDED), "cuMemGetAllocationGranularity")
    return g.value


class VmmBuffer(object):
    """nbytes of device memory from cuMemCreate, in physical chunks of at most `chunk` bytes mapped into one VA range.
    `compressed_bytes` counts the chunks whose handle reports compression granted."""

    def __init__(self, dev, nbytes, compress=True, chunk=None):
        gran = granularity(dev, compress)
        self.size = (nbytes + gran - 1) // gran * gran
        chunk = self.size if chunk is None else (chunk + gran - 1) // gran * gran
        self.ptr, self.handles, self.compressed_bytes = _u64(), [], 0
        ck(cu.cuMemAddressReserve(ctypes.byref(self.ptr), ctypes.c_size_t(self.size), ctypes.c_size_t(gran), _u64(0),
                                  _u64(0)), "cuMemAddressReserve")
        prop = prop_for(dev, compress)
        off = 0
        while off < self.size:
            sz = min(chunk, self.size - off)
            h = _u64()
            ck(cu.cuMemCreate(ctypes.byref(h), ctypes.c_size_t(sz), ctypes.byref(prop), _u64(0)), "cuMemCreate")
            self.handles.append((h, sz))
            got = AllocProp()
            ck(cu.cuMemGetAllocationPropertiesFromHandle(ctypes.byref(got), h), "cuMemGetAllocationPropertiesFromHandle")
            if got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC:
                self.compressed_bytes += sz
            ck(cu.cuMemMap(_u64(self.ptr.value + off), ctypes.c_size_t(sz), ctypes.c_size_t(0), h, _u64(0)), "cuMemMap")
            off += sz
        acc = AccessDesc()
        acc.location.type, acc.location.id, acc.flags = CU_MEM_LOCATION_TYPE_DEVICE, dev, CU_MEM_ACCESS_FLAGS_PROT_READWRITE
        ck(cu.cuMemSetAccess(self.ptr, ctypes.c_size_t(self.size), ctypes.byref(acc), ctypes.c_size_t(1)), "cuMemSetAccess")

    def tensor(self, shape, dtype=torch.float32):
        typestr = {torch.float32: "<f4", torch.uint8: "|u1"}[dtype]
        owner = self

        class _View(object):
            __cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (self.ptr.value, False),
                                        "version": 2}
            keep = owner
        return torch.as_tensor(_View(), device="cuda")

    def free(self):
        torch.cuda.synchronize()
        off = 0
        for h, sz in self.handles:
            ck(cu.cuMemUnmap(_u64(self.ptr.value + off), ctypes.c_size_t(sz)), "cuMemUnmap")
            ck(cu.cuMemRelease(h), "cuMemRelease")
            off += sz
        ck(cu.cuMemAddressFree(self.ptr, ctypes.c_size_t(self.size)), "cuMemAddressFree")
        self.handles = []


def free_gb():
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info()[0] / 1e9


def smi(fields):
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + fields, "--format=csv,noheader", "-i", "0"],
                              stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
    except Exception as e:          # noqa: BLE001
        return "n/a (%s)" % e


def timed(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def log(*a):
    print(*a, flush=True)


def raw_ceilings(dev, out):
    """zero_ / fill_(1.0) / tiled copy of real v0 obs / sum over 8 GiB, plain then compressible, alternated twice"""
    src_env = lmz.LmazeVecCuda(512, "v0", seed=3)
    src_env.reset()
    for i in range(20):
        src_env.step(torch.randint(0, 4, (512,), device="cuda", dtype=torch.uint8))
    src = src_env.obs.reshape(-1).clone()             # 57.8 MB: stays in L2 while it is copied
    src_env.close()
    del src_env
    reps = (8 << 30) // (src.numel() * 4)
    numel = reps * src.numel()
    gb = numel * 4 / 1e9
    res = []
    for rnd in range(2):
        for kind in ("plain", "compressible"):
            buf = None
            if kind == "plain":
                t = torch.empty(numel, dtype=torch.float32, device="cuda")
            else:
                buf = VmmBuffer(dev, numel * 4, chunk=CHUNK)
                t = buf.tensor((numel,))
            tv = t.view(reps, -1)
            r = {"round": rnd, "memory": kind, "gb": gb}
            r["zero_ms"] = timed(t.zero_, 100)
            r["fill1_ms"] = timed(lambda: t.fill_(1.0), 100)
            r["copy_v0_obs_ms"] = timed(lambda: tv.copy_(src.expand(reps, -1)), 100)
            r["sum_ms"] = timed(lambda: t.sum(), 100)
            for k in ("zero", "fill1", "copy_v0_obs", "sum"):
                r[k + "_tbs"] = gb / r[k + "_ms"]
            if buf is not None:
                r["compressed_bytes"] = buf.compressed_bytes
            log(json.dumps(r))
            res.append(r)
            del t, tv
            if buf is not None:
                buf.free()
            torch.cuda.empty_cache()
    out["raw_8gib"] = res


def obs_buffers(env, kind, dev):
    """(tensors to bind, owners to free) for env's obs (and v5's local obs)"""
    shapes = [((env.num_envs,) + env.obs_shape, env.obs_dtype)]
    if isinstance(env, lmz.LmazeHierCuda):
        shapes.append(((env.num_envs,) + env.local_obs_shape, torch.float32))
    tensors, owners = [], []
    for shape, dtype in shapes:
        nbytes = int(torch.Size(shape).numel()) * torch.tensor([], dtype=dtype).element_size()
        if kind == "plain":
            tensors.append(torch.empty(shape, dtype=dtype, device="cuda"))
        else:
            b = VmmBuffer(dev, nbytes, chunk=CHUNK)
            owners.append(b)
            tensors.append(b.tensor(shape, dtype))
    return tensors, owners


def rebind(env, tensors):
    env.obs = tensors[0]
    _abi.call(env._lib.lmz_bind_dl, env._h, env.obs, env.reward, env._done_u8)
    if len(tensors) > 1:
        env.loc_obs = tensors[1]
        _abi.call(env._lib.lmz_bind_local_dl, env._h, env.loc_obs, env.local_reward, env._ldone_u8,
                  env._loc_err_u8, env.foveal_goal)


def mode_ab(dev, name, make, n, warm_first, steps, rounds=3, warm=20):
    """one handle, its obs rebound plain <-> compressible `rounds` times; ms per step of each"""
    env = make()
    hier = isinstance(env, lmz.LmazeHierCuda)
    if env.obs is not None:               # the constructor's own tensors are not timed: free them first
        env.obs = None
        if hier:
            env.loc_obs = env.fov_obs = None
        torch.cuda.empty_cache()
    R = 4
    ring = torch.randint(0, env.num_actions, (R, n), device="cuda", dtype=torch.uint8)
    goals = torch.randint(0, 25, (R, n), device="cuda", dtype=torch.uint8) if hier else None

    def step(i):
        if hier:
            env.plannerStep(goals[i % R], mask="auto")
            env.step(ring[i % R], goal_plane=False)
        else:
            env.step(ring[i % R])
    res = {"mode": name, "n": n, "runs": []}
    first = True
    for rnd in range(rounds):
        for kind in ("plain", "compressible"):
            tensors, owners = obs_buffers(env, kind, dev)
            rebind(env, tensors)
            if first:
                env.reset()
            w = warm_first if first else warm
            first = False
            i0 = [0]

            def one():
                step(i0[0])
                i0[0] += 1
            for _ in range(w):
                one()
            ms = timed(one, steps, warm=0)
            r = {"round": rnd, "memory": kind, "ms_per_step": ms, "env_steps_per_s": n / (ms * 1e-3)}
            if owners:
                r["compressed_bytes"] = sum(b.compressed_bytes for b in owners)
                r["bytes"] = sum(b.size for b in owners)
            if not hier and env.obs_mode == "full":
                r["obs_sum_ms"] = timed(lambda: env.obs.sum(), 3, warm=1)
            res["runs"].append(r)
            log(name, json.dumps(r))
            env.obs = None
            if hier:
                env.loc_obs = None
            _abi.call(env._lib.lmz_bind_dl, env._h, None, env.reward, env._done_u8)
            del tensors
            for b in owners:
                b.free()
            torch.cuda.empty_cache()
    env.close()
    del env, ring
    torch.cuda.empty_cache()
    p = [r["ms_per_step"] for r in res["runs"] if r["memory"] == "plain"]
    c = [r["ms_per_step"] for r in res["runs"] if r["memory"] == "compressible"]
    res["gain_per_round"] = [a / b - 1 for a, b in zip(p, c)]
    log(name, "gain per round", res["gain_per_round"])
    return res


def sweep(dev, out):
    """tune[0..3] and the render path of the v0 / v3 full render, on compressible memory (a new handle per point)"""
    n = 1 << 20
    points = [("default", "tma", ()), ("t0=64", "tma", (64,)), ("t0=128", "tma", (128,)), ("t0=256", "tma", (256,)),
              ("t2=2", "tma", (0, 0, 2)), ("t0=64,t2=2", "tma", (64, 0, 2)), ("l2=normal", "tma", (0, 2)),
              ("l2=none", "tma", (0, 4)), ("l2=last", "tma", (0, 3)), ("split=4096", "tma", (0, 0, 0, 4096)),
              ("split=16384", "tma", (0, 0, 0, 16384)), ("default", "tma", ()), ("st128", "st128", ()),
              ("st128,t0=512", "st128", (512,)), ("default", "tma", ())]
    out["sweep"] = []
    for variant in ("v0", "v3"):
        probe_env = lmz.LmazeVecCuda(1, variant, with_obs=False)
        shape = (n,) + probe_env.obs_shape
        probe_env.close()
        buf = VmmBuffer(dev, int(torch.Size(shape).numel()) * 4, chunk=CHUNK)
        obs = buf.tensor(shape)
        ring = torch.randint(0, 4, (4, n), device="cuda", dtype=torch.uint8)
        for label, mode, tune in points:
            try:
                env = lmz.LmazeVecCuda(n, variant, seed=2026, render_mode=mode, tune=tune, with_obs=False)
            except Exception as e:          # noqa: BLE001
                log(variant, label, "rejected:", e)
                continue
            env.obs = obs
            env._bind()
            env.reset()
            i0 = [0]

            def one():
                env.step(ring[i0[0] % 4])
                i0[0] += 1
            ms = timed(one, 100, warm=20)
            r = {"variant": variant, "point": label, "render_mode": mode, "tune": list(tune), "ms_per_step": ms,
                 "env_steps_per_s": n / (ms * 1e-3), "compressed_bytes": buf.compressed_bytes}
            log(json.dumps(r))
            out["sweep"].append(r)
            env.close()
            del env
        del obs, ring
        buf.free()
        torch.cuda.empty_cache()


def main():
    path = sys.argv[1]
    do_sweep = "--sweep" in sys.argv
    out = {"gpu": smi("name,power.limit,clocks.sm,clocks.max.sm,memory.total"), "torch": torch.__version__,
           "device_count": torch.cuda.device_count()}
    torch.cuda.init()
    torch.empty(1, device="cuda")           # makes the primary context current on this thread
    dev = torch.cuda.current_device()
    ck(cu.cuInit(0), "cuInit")
    attr = ctypes.c_int()
    ck(cu.cuDeviceGetAttribute(ctypes.byref(attr), CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev),
       "cuDeviceGetAttribute")
    out["generic_compression_supported"] = attr.value
    out["granularity"] = {"plain": granularity(dev, False), "compressible": granularity(dev, True)}
    log(json.dumps(out))

    def save():
        with open(path, "w") as f:
            json.dump(out, f, indent=1)

    # the 2^20-env v0 obs tensor: whole, then in 1 GiB / 16 GiB chunks -- how much compression is granted, at what cost
    obs_bytes = (1 << 20) * 4 * 84 * 84 * 4
    out["grant"] = []
    for chunk in (None, 16 << 30, 1 << 30):
        f0 = free_gb()
        t0 = time.perf_counter()
        try:
            b = VmmBuffer(dev, obs_bytes, chunk=chunk)
        except RuntimeError as e:
            out["grant"].append({"chunk": chunk, "error": str(e)})
            log(json.dumps(out["grant"][-1]))
            continue
        r = {"chunk": chunk, "bytes": b.size, "compressed_bytes": b.compressed_bytes, "chunks": len(b.handles),
             "alloc_s": time.perf_counter() - t0, "free_gb_drop": f0 - free_gb(), "obs_gb": obs_bytes / 1e9}
        b.free()
        r["free_gb_after_release"] = free_gb()
        out["grant"].append(r)
        log(json.dumps(r))
    global CHUNK
    best = max((g for g in out["grant"] if "error" not in g), key=lambda g: g["compressed_bytes"], default=None)
    CHUNK = best["chunk"] if best else None
    out["chunk_used"] = CHUNK
    save()
    raw_ceilings(dev, out)
    save()

    n = 1 << 20
    runs = [("v0_tma", lambda: lmz.LmazeVecCuda(n, "v0", seed=2026, with_obs=False), n, 20, 200)]
    out["modes"] = [mode_ab(dev, *runs[0])]
    save()
    v0 = out["modes"][0]
    go = all(g >= 0.03 for g in v0["gain_per_round"])
    out["go"] = go
    log("GO" if go else "NO-GO", v0["gain_per_round"])
    more = [("v3_tma", lambda: lmz.LmazeVecCuda(n, "v3", seed=2026, with_obs=False), n, 20, 200),
            ("v0_st128", lambda: lmz.LmazeVecCuda(n, "v0", seed=2026, render_mode="st128", with_obs=False), n, 20, 100),
            ("v0_compact_16m", lambda: lmz.LmazeVecCuda(1 << 24, "v0", seed=2026, obs_mode="compact", with_obs=False),
             1 << 24, 20, 100),
            ("v0_incremental", lambda: lmz.LmazeVecCuda(n, "v0", seed=2026, render_mode="incremental", with_obs=False),
             n, 20, 200),
            ("v2_full", lambda: lmz.LmazeVecCuda(n, "v2", seed=2026, with_obs=False), n, 1000, 100),
            ("v4_full", lambda: lmz.LmazeVecCuda(n, "v4", seed=2026, with_obs=False), n, 1000, 100),
            ("v5_full", lambda: lmz.LmazeHierCuda(n, "v5", seed=2026), n, 1000, 100)]
    for m in more:
        try:
            out["modes"].append(mode_ab(dev, *m))
        except Exception as e:          # noqa: BLE001
            out["modes"].append({"mode": m[0], "error": repr(e)})
            log(m[0], "error", repr(e))
        save()
    if do_sweep and go:
        sweep(dev, out)
    out["gpu_after"] = smi("name,power.limit,clocks.sm,clocks.max.sm")
    save()
    log("done")


if __name__ == "__main__":
    main()
