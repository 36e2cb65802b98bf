#!/usr/bin/env python
"""Headline benchmark: env-steps/s of the fused LMaze step at 1M envs per B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: the fused kernel (action
decode, wall lookup, move, reward, done, auto-reset, full f32 observation render,
statistics) over every env of the rank's shard.  Workload = BASELINE.json
configs[2] ("lmaze_env_v0 1M envs, fused step+auto-reset+obs render on 1xB200"),
N = 2^20 envs PER GPU (weak scaling, one process per GPU, no data-path collective).

Prints ONE JSON line (rank 0).  `value` = device-timed throughput with the action
stream already resident in HBM; `e2e` = the same metric through the host-buffer
C-ABI call lmz_step_host (pinned host actions -> H2D -> fused step -> D2H
reward/done), observations staying in HBM where the policy consumes them (DLPack).
`--impl reference` times the CPU oracle port (the reference's algorithm in C,
oracle/) on all host threads; where the unmodified reference is importable
(/root/reference here, baseline/_ref on the GPU box) its own Python step() loop is
timed beside it on every host core (`cpu_baseline.reference_python`).

`extras` (every world size, barrier + max over ranks like `value`): the T=64 rollout
at 2^21 envs per GPU (BASELINE configs[4]), lmaze-v3 full render at 2^20 envs per GPU
(configs[3]), v0 compact and incremental observations, host-consumer e2e lines, and
`checks`: NCCL-summed step counters against launches x envs, and shard invariance
on the real GPUs (rank r's first rows replayed by rank 0 with the same global ids).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V0_OBS_BYTES = 4 * 84 * 84 * 4
# algorithmic bytes per env-step of the fused v0 step (SURVEY.md section 8d / DESIGN.md):
# obs write + u8 action read + packed state read + write + f32 reward write + u8 done write
V0_STEP_BYTES = V0_OBS_BYTES + 1 + 4 + 4 + 4 + 1
V3_OBS_BYTES = 3 * 72 * 72 * 4
V3_STEP_BYTES = V3_OBS_BYTES + 1 + 4 + 4 + 4 + 1
FALLBACK_HBM_GBS = 6650.0      # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
# --dump-outputs keeps at most 256 observation rows (v0: 28.9 MB) and 2^20 values of each per-env output, which holds
# every variant's dump under 64 MB
DUMP_OBS_ROWS = 256
DUMP_ENV_VALUES = 1 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=None,
                    help="untimed steps before the timed region (default 5; 1000 for the foveal variants v2 / v4 / v5, "
                         "whose episodes need that long to de-synchronise: in steady state half the warps of a step "
                         "hold a resetting env, and a v4 / v5 warp folds visit histories of up to ~50 entries)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--variant", default="v0", choices=["v0", "v2", "v3", "v4", "v5"])
    ap.add_argument("--render-mode", default="tma", choices=["tma", "st128", "incremental"])
    ap.add_argument("--obs-mode", default="full", choices=["full", "compact"])
    ap.add_argument("--window", type=int, default=0,
                    help="obs rows kept in HBM (render window); 0 = all envs.  A step then = fused step over "
                         "every env + a render pass per remaining window, so every env's obs is still produced")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the rollout / obs-to-host side measurements")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU-oracle timing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to its caller as DIR/<name>.npy (float32; per-env "
                         "values of up to %d envs and %d observation rows, larger batches as a fixed seeded sample "
                         "whose env indices are written beside them), so that two builds can be compared output for "
                         "output"
                         % (DUMP_ENV_VALUES, DUMP_OBS_ROWS))
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    if args.warmup is None:
        args.warmup = 1000 if (args.impl == "ours" and args.variant in ("v2", "v4", "v5")) else 5
    return args


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def recorded_traffic(variant, render_mode, n_envs):
    """dram bytes per launch from the committed `ncu --set full` capture (scaled to this batch size), and whether
    that capture was taken on the kernel sources this build was compiled from (profiles/traffic.json records the
    hash of csrc/ + include/; a capture of other sources is reported as stale and its number withheld)."""
    try:
        from gym_lmaze_b200.build import source_hash
        doc = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        rec = doc.get("%s_%s" % (variant, render_mode))
        fresh = doc.get("csrc_hash") == source_hash()
        src = {"file": "profiles/traffic.json", "csrc_hash": doc.get("csrc_hash"), "matches_build": fresh}
        if not fresh or not isinstance(rec, dict):
            return None, src
        src["capture"] = rec.get("source")
        return rec["bytes"] * n_envs / rec["envs"], src
    except Exception as exc:
        return None, {"error": repr(exc)}


# --------------------------------------------------------------------------- CPU legs (oracle = checker / baseline only)
def cpu_oracle_throughput_v5(n_envs, threads, budget_s, min_steps=2, warmup=0):
    """lmaze-v5: plannerStep (where the local episode ended) + step + reset on globalDone, both observations
    rendered, on `threads` host threads (one OracleHier slice per thread; ctypes releases the GIL).  The clock
    starts once every thread has built its slice and run `warmup` untimed steps."""
    import numpy as np
    from oracle import oracle as O
    per = max(1, n_envs // threads)
    counts = [0] * threads
    ready = threading.Barrier(threads + 1)

    def worker(k):
        rng = np.random.RandomState(k)

        def step(mask):
            o.planner_step(rng.randint(0, 25, size=per), mask=mask)
            _, _, _, _, gd, ld, _ = o.step(rng.randint(0, 4, size=per))
            if gd.any():
                o.reset(mask=gd, want_obs=False)
            return (gd | ld).astype(np.uint8)
        try:
            o = O.OracleHier(per, seed=1, env_id0=k * per)
            o.reset(want_obs=False)
            mask = np.ones(per, np.uint8)
            for _ in range(warmup):
                mask = step(mask)
        except BaseException:
            ready.abort()          # the main thread's wait raises instead of waiting for this thread forever
            raise
        ready.wait()
        t0 = time.perf_counter()
        while counts[k] < min_steps or time.perf_counter() - t0 < budget_s:
            mask = step(mask)
            counts[k] += 1
    ths = [threading.Thread(target=worker, args=(k,)) for k in range(threads)]
    for t in ths:
        t.start()
    ready.wait()
    t0 = time.perf_counter()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return per * sum(counts) / dt, sum(counts) // threads, dt


def cpu_oracle_throughput(variant, n_envs, threads, budget_s, min_steps=2):
    """Steps/s of the C oracle port (full step + auto-reset + f32 render) on `threads` host threads."""
    if variant == "v5":
        return cpu_oracle_throughput_v5(n_envs, threads, budget_s, min_steps)
    import numpy as np
    from oracle import oracle as O
    ov = {"v0": O.V0, "v2": O.V2, "v3": O.V3, "v4": O.V4}[variant]
    vec = O.OracleVec(ov, n_envs, seed=1, autoreset=True, threads=threads)
    obs = np.empty((n_envs,) + O.OBS_SHAPE[ov], dtype=np.float32)
    vec.reset(want_obs=False)
    rng = np.random.RandomState(1)
    acts = rng.randint(0, 25 if variant in ("v2", "v4") else 4, size=(8, n_envs)).astype(np.int64)
    vec.step(acts[0], obs_out=obs)          # warm (touch pages)
    t0 = time.perf_counter()
    k = 0
    while k < min_steps or time.perf_counter() - t0 < budget_s:
        vec.step(acts[k % 8], obs_out=obs)
        k += 1
    dt = time.perf_counter() - t0
    return n_envs * k / dt, k, dt


def python_loop_throughput(n_steps=40):
    """The reference's implementation STYLE (interpreted per-pixel loop) on this host, 1 core."""
    from oracle import oracle as O
    from oracle.pyloop import PyLoopV0
    import random
    env = PyLoopV0(O.layout(O.V0), (1, 1))
    rng = random.Random(1)
    t0 = time.perf_counter()
    for _ in range(n_steps):
        _, _, d, _ = env.step(rng.randrange(4))
        if d:
            env.reset((1, 1))
    return n_steps / (time.perf_counter() - t0)


def reference_python_throughput(variant, budget_s):
    """The UNMODIFIED reference's own step() loop (BASELINE.md section 4) on every host core for a fixed wall budget:
    P independent processes, each loading gym_lmaze/envs/lmaze_env*.py by path (baseline/_ref on the GPU box,
    /root/reference in the build container) under the test harness's gym stub.  None where it is not present."""
    try:
        from oracle import ref_bench
        return ref_bench.measure(variant, os.cpu_count() or 1, budget_s)
    except Exception as exc:  # pragma: no cover
        return {"error": repr(exc)}


def run_reference(args):
    """`--impl reference`: the CPU arm.  Rank 0 only; other ranks exit 0 without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import oracle as O
    O.build()
    threads = os.cpu_count() or 1
    sample_envs = 32768
    if args.variant == "v5":
        value, k, dt = cpu_oracle_throughput_v5(sample_envs, threads, 0.0, min_steps=args.steps, warmup=args.warmup)
        sample = ("%d-env slice of the %d-env workload per step (plannerStep where due + step + both f32 obs renders), "
                  "C oracle port, %d threads; %d timed steps after %d warm-up steps"
                  % (sample_envs, args.envs, threads, k, args.warmup))
        print(json.dumps({
            "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / max(1, k) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, note="CPU arm: bounded sample per step"),
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return
    ov = {"v0": O.V0, "v2": O.V2, "v3": O.V3, "v4": O.V4}[args.variant]
    import numpy as np
    vec = O.OracleVec(ov, sample_envs, seed=1, autoreset=True, threads=threads)
    obs = np.empty((sample_envs,) + O.OBS_SHAPE[ov], dtype=np.float32)
    vec.reset(want_obs=False)
    acts = np.random.RandomState(1).randint(0, 25 if args.variant in ("v2", "v4") else 4,
                                            size=(8, sample_envs)).astype(np.int64)
    for i in range(args.warmup):
        vec.step(acts[i % 8], obs_out=obs)
    t0 = time.perf_counter()
    for i in range(args.steps):
        vec.step(acts[i % 8], obs_out=obs)
    dt = time.perf_counter() - t0
    value = sample_envs * args.steps / dt
    sample = ("%d-env slice of the %d-env workload per step (full step + auto-reset + f32 obs render), "
              "C oracle port of the reference algorithm, %d pthreads" % (sample_envs, args.envs, threads))
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, note="CPU arm: bounded sample per step"),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample,
                         "reference_python": reference_python_throughput(args.variant, 5.0)},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, note=None):
    G, E, C = {"v0": (12, 7, 4), "v3": (18, 4, 3), "v2": (5, 7, 5), "v4": (5, 7, 7), "v5": (5, 7, 11)}[args.variant]   # v2/v4/v5: 5x5 fovea; v5: (7,35,35) + (4,35,35)
    if args.obs_mode == "compact" and args.variant in ("v2", "v4", "v5"):
        obs, per_env = "f32 (%d,5,5) compact (the 5x5 crops; reference image = x7 replication)" % C, C * 25 * 4
    elif args.obs_mode == "compact":
        obs, per_env = "u8 (%d,%d,%d) compact (un-expanded layers; reference image = x%d replication)" % (C, G, G, E), C * G * G
    else:
        obs, per_env = "f32 (%d,%d,%d) full render" % (C, G * E, G * E), C * G * E * G * E * 4
    W = args.window if 0 < args.window < args.envs else args.envs
    which = ("BASELINE configs[2], HBM roofline run" if args.variant == "v0" and args.obs_mode == "full"
             else "BASELINE configs[3]-style: largest maze variant" if args.variant == "v3" and args.obs_mode == "full"
             else "SURVEY 8f next #1: multi-layout foveal env" if args.variant == "v2"
             else "SURVEY 8f next #3: foveal env + float visit layer" if args.variant == "v4"
             else "SURVEY 8f next #4: planner/actor env, a step = plannerStep(auto mask) + step, two obs tensors"
             if args.variant == "v5" else "compact-observation mode")
    cfg = {
        "workload": "lmaze_env_%s %d envs/GPU, fused step+auto-reset+obs render (%s)" % (args.variant, args.envs, which),
        "variant": args.variant, "envs_per_gpu": args.envs, "obs": obs, "actions": "u8 ring [4,N] resident in HBM",
        "render_mode": args.render_mode, "obs_mode": args.obs_mode, "autoreset": True,
        "obs_window_envs": W,
        "l2": "no flush needed: each step streams %.2f GB of obs, >> 126 MB L2" % (args.envs * per_env / 1e9),
    }
    if W < args.envs:
        cfg["window"] = ("obs tensor holds %d of %d envs; a step = 1 fused step launch + %d render-window launches, "
                         "every env's obs is written once per step" % (W, args.envs, -(-args.envs // W) - 1))
    if args.variant in ("v2", "v4", "v5"):
        cfg["steady_state"] = ("%d warm-up steps before the timed region.  All envs start their first episode together; the "
                               "episodes need about 1,000 steps to de-synchronise (oracle run, random actions, v4: the share "
                               "of warps holding a resetting env settles at 0.50 per step, the visit histories at mean length "
                               "25 with a warp maximum of 50).  Right after a reset a step is up to 30 %% cheaper (no "
                               "divergent resets, short histories): that is not the number to quote" % args.warmup)
    if note:
        cfg["note"] = note
    return cfg


# --------------------------------------------------------------------------- our arm
class Ranks(object):
    """One process per GPU: barrier, max-over-ranks and the device of this rank."""

    def __init__(self, torch, dist):
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize(self.dev)

    def reduce_max(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(self, ok):
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())

    def gather(self, t):
        """[world] list of every rank's copy of `t` (same shape on every rank)."""
        if self.world == 1:
            return [t]
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t.contiguous())
        return out

    def timed_ms(self, fn, reps, warm):
        """`reps` calls of fn(i) after `warm` untimed ones: CUDA events on the launch stream, barrier +
        synchronize on both sides, MAX over ranks.  Returns ms per call."""
        torch = self.torch
        for i in range(warm):
            fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            fn(i)
        e1.record()
        self.barrier()
        return self.reduce_max(e0.elapsed_time(e1)) / reps


def run_ours(args):
    import torch
    import torch.distributed as dist

    rk = Ranks(torch, dist)
    world, rank, dev = rk.world, rk.rank, rk.dev
    barrier, reduce_max = rk.barrier, rk.reduce_max

    import gym_lmaze_b200 as lmz          # raises if the CUDA library is missing: no fallback
    N = args.envs
    W = args.window if 0 < args.window < N else N
    hier = args.variant == "v5"
    SEED = 2026
    if hier:
        env = lmz.LmazeHierCuda(N, "v5", device=dev, seed=SEED, env_id0=rank * N, autoreset=True, obs_mode=args.obs_mode)
    else:
        env = lmz.LmazeVecCuda(N, args.variant, device=dev, seed=SEED, env_id0=rank * N, autoreset=True,
                               render_mode=args.render_mode, obs_mode=args.obs_mode, obs_window=W)
    windows = list(range(0, N, W))
    if windows[-1] + W > N:
        windows[-1] = N - W
    obs_bytes = env.obs[0].numel() * env.obs.element_size()
    # v4: the visit layer is kept as its history (DESIGN.md 3.5): 64 B read + the appended entry (1 B) written per env-step
    step_bytes = obs_bytes + 14 + (VISIT_HIST_BYTES + 1 if args.variant == "v4" else 0)
    if hier:
        step_bytes = 0        # filled in after the timed region from the measured localDone / planner fractions
    if args.render_mode == "incremental":
        # persistent obs tensor: at most the old and the new ExE ball block are rewritten (upper bound)
        E = 7 if args.variant == "v0" else 4
        step_bytes = 2 * E * E * 4 + 14

    def full_step(i):
        """one step = transition of every env + every env's observation written once"""
        actions = ring[i % R]
        if hier:        # plannerStep for the envs waiting for their planner (device-side mask), then the actor step
            env.plannerStep(goal_ring[i % R], mask="auto")
            env.step(actions, goal_plane=False)
            return
        if len(windows) > 1:
            env.set_window(windows[0])
        env.step(actions)
        for lo in windows[1:]:
            env.render_window(lo)
    R = 4

    def action_ring(r):
        """rank r's device-resident action ring (any rank can regenerate it: shard-invariance replay)"""
        gen = torch.Generator(device=dev).manual_seed(1234 + r)
        ring_ = torch.randint(0, env.num_actions, (R, N), generator=gen, device=dev, dtype=torch.uint8)
        goals_ = torch.randint(0, 25, (R, N), generator=gen, device=dev, dtype=torch.uint8) if hier else None
        return ring_, goals_
    ring, goal_ring = action_ring(rank)
    env.reset()

    # ---- device-resident inputs: K launches of the fused kernel, CUDA events on the launch stream
    for i in range(args.warmup):
        full_step(i)
    launches0 = env.launch_count
    sampler = ClockSampler(rk.local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    evs[0].record()
    for i in range(args.steps):
        full_step(i)
        evs[i + 1].record()
    barrier()
    total_ms = reduce_max(evs[0].elapsed_time(evs[-1]))
    gpu_launches = env.launch_count - launches0
    per_step = sorted(evs[i].elapsed_time(evs[i + 1]) / max(1, len(windows)) for i in range(args.steps))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # step() hands its caller the env's own output buffers: read them before anything steps the env again
        outputs = {"obs": env.obs, "reward": env.reward, "done": env.done}
        if hier:
            outputs.update(local_obs=env.loc_obs, local_reward=env.local_reward, local_done=env.local_done,
                           foveal_goal=env.foveal_goal)
        dump_outputs(args.dump_outputs, outputs, windows[-1], "_rank%d" % rank if world > 1 else "")
    value = world * N * args.steps / (total_ms * 1e-3)
    step_ms = total_ms / args.steps
    launches_per_step = max(1, gpu_launches // args.steps)
    kernel_ms = step_ms / launches_per_step      # default config: ONE launch per step, step time == kernel time
    hier_note = None
    if hier:
        ld = float(env._ldone_u8.float().mean())            # share of env-steps whose local episode is over
        st = env.get_state()
        pf = float(((st[:, 15] & 2) != 0).logical_or(st[:, 14] == 0).float().mean())   # share waiting for the planner
        # step launch: foveal + local obs, visit layer read (+ written back where localDone), 3 state words r/w,
        # 2 rewards, 4 flag bytes, action; planner launch: 3 state words read, and for the waiting envs goal +
        # state write + local obs
        fov_b, loc_b = (34300, 19600) if args.obs_mode == "full" else (700, 400)
        step_bytes = int(fov_b + loc_b + VISIT_HIST_BYTES + 1 * ld + 24 + 8 + 4 + 1 + 12 + pf * (loc_b + 12 + 1 + 2))
        hier_note = {"local_done_fraction": ld, "planner_fraction": pf,
                     "bytes": "%d foveal + %d local obs + %d visit history read (+1 x localDone written; the layer is kept "
                              "as its history, DESIGN.md 3.5) + state/rewards/flags/action 37 + planner launch: 12 + "
                              "planner_fraction x (%d local obs + 15)" % (fov_b, loc_b, VISIT_HIST_BYTES, loc_b)}
    achieved = N * step_bytes / (step_ms * 1e-3) / 1e9

    # ---- checks on the real GPUs (SURVEY section 4 T4 / section 8e): counters and shard invariance
    checks = main_workload_checks(rk, lmz, env, args, hier, SEED, N, W, R, action_ring,
                                  steps_done=args.warmup + args.steps)

    # ---- end to end through the host-buffer C-ABI call (pinned host memory)
    hgen = torch.Generator().manual_seed(4321 + rank)
    a_host = torch.randint(0, env.num_actions, (R, N), generator=hgen, dtype=torch.uint8).pin_memory()
    r_host = torch.empty(N, dtype=torch.float32).pin_memory()
    d_host = torch.empty(N, dtype=torch.uint8).pin_memory()
    if hier:
        g_host = torch.randint(0, 25, (R, N), generator=hgen, dtype=torch.uint8).pin_memory()
        r2_host = torch.empty(N, dtype=torch.float32).pin_memory()
        d2_host = torch.empty(N, dtype=torch.uint8).pin_memory()

    def full_step_host(i):
        if hier:
            env.step_host(g_host[i % R], a_host[i % R], r_host, r2_host, d_host, d2_host)
            return
        if len(windows) > 1:
            env.set_window(windows[0])
        env.step_host(a_host[i % R], r_host, d_host)
        for lo in windows[1:]:
            env.render_window(lo)
        if len(windows) > 1:
            torch.cuda.synchronize(dev)

    host_warm = max(3, min(args.warmup, 8))          # (the envs are in steady state already)
    for i in range(host_warm):
        full_step_host(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        full_step_host(i)
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = reduce_max(max(e0.elapsed_time(e1), wall_ms))
    e2e_value = world * N * args.steps / (e2e_ms * 1e-3)
    checksum = float(r_host.sum())               # the host really consumes the result

    stats = env.stats_allreduce(check_errors=not hier) if world > 1 else env.stats(check_errors=not hier)   # v5: random actors hit the reference's IndexError rows
    steps_launched = args.warmup + args.steps + host_warm + args.steps
    env.close()
    del env, ring, goal_ring
    torch.cuda.empty_cache()

    # ---- other operating points, at EVERY world size (each names its own mode; never mixed into `value`)
    extras = {}
    if not args.no_extras:
        sampler2 = ClockSampler(rk.local_rank)              # the extras' timed regions are short: one sampler over all of them
        if rank == 0:
            sampler2.start()
        extras = side_measurements(rk, lmz, args, SEED)
        if rank == 0:
            extras["clocks"] = sampler2.stop()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    traffic, traffic_src = (recorded_traffic(args.variant, args.render_mode, N)
                            if (args.obs_mode == "full" and W == N) else (None, None))
    line = {
        "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": 2 * N if hier else N,
                "d2h_bytes_per_step": 10 * N if hier else 5 * N,
                "ms_per_step": e2e_ms / args.steps,
                "api": "LmazeHierCuda.step_host -> lmz_hier_step_host (C ABI)" if hier
                else "LmazeVecCuda.step_host -> lmz_step_host (C ABI)",
                "obs": "device-resident: this e2e assumes a GPU-resident consumer (the policy reads the obs tensor "
                       "zero-copy via DLPack); actions H2D and reward/done D2H are inside the timed region, the "
                       "observation is NOT copied to the host.  For a HOST consumer see extras.e2e_host_consumer "
                       "(compact / bit-packed obs landing in pinned host memory) and extras.e2e_obs_to_host "
                       "(every f32 obs byte over PCIe).", "reward_checksum": checksum},
        "gpu_launches": gpu_launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "kernel": "lmz_fov_small_kernel<%s>" % args.variant.upper()
                     if (args.variant in ("v2", "v4", "v5") and args.obs_mode == "compact") else
                     "lmz_env_fov_kernel<%s>" % args.variant.upper() if args.variant in ("v2", "v4", "v5") else
                     "lmz_env_incr_kernel<%s>" % args.variant.upper() if args.render_mode == "incremental" else
                     "lmz_env_%s_kernel<%s>" % ("compact" if args.obs_mode == "compact" else
                                                "tma" if args.render_mode == "tma" else "st", args.variant.upper()),
                     "launches_per_step": launches_per_step,
                     "note": "write-only stream; peak is the measured read+write COPY rate, so frac may exceed 1 "
                             "(compare extras.pure_write_fill_gbs)",
                     "bytes_per_env_step": step_bytes, "bytes_per_launch": N * step_bytes // launches_per_step,
                     "kernel_ms_avg": kernel_ms, "kernel_ms_min": per_step[0],
                     "kernel_ms_median": per_step[len(per_step) // 2]},
        "episode_stats": stats,
        "checks": checks,
    }
    checks["nccl_steps_sum"] = {"steps": stats["steps"], "expected": world * N * steps_launched if not hier else None,
                                "what": "sum over ranks of the device step counters (one all_reduce(int64[8])) vs "
                                        "world x envs x step calls of the whole run (%d: warm-up + timed, device and "
                                        "host-buffer loops)" % steps_launched}
    if not hier:
        checks["nccl_steps_sum"]["ok"] = checks["nccl_steps_sum"]["steps"] == checks["nccl_steps_sum"]["expected"]
    if hier_note:
        line["roofline"]["v5"] = hier_note
    if extras:
        line["extras"] = extras
    if not args.no_cpu_baseline and world == 1:
        from oracle import oracle as O
        O.build()
        P = os.cpu_count() or 1
        v_all, k_all, dt_all = cpu_oracle_throughput(args.variant, 16384, P, args.cpu_budget)
        v_one, k_one, dt_one = cpu_oracle_throughput(args.variant, 2048, 1, min(4.0, args.cpu_budget))
        line["cpu_baseline"] = {
            "value": v_all, "unit": "env-steps/s", "cores": P, "kind": "port",
            "sample": "%d steps of a 16384-env slice of the workload (%.1f s), C oracle port, %d pthreads"
                      % (k_all, dt_all, P),
            "single_core": {"value": v_one, "sample": "%d steps x 2048 envs (%.1f s)" % (k_one, dt_one)},
            "reference_python": reference_python_throughput(args.variant, min(8.0, args.cpu_budget)),
            "python_loop": None if hier else {"value": python_loop_throughput(), "cores": 1,
                            "sample": "40 steps of oracle/pyloop.py, a RESTATEMENT of the reference's interpreted "
                                      "per-pixel loop (not the reference: it runs ~2x faster than the real "
                                      "lmaze_env.py, see reference_python / profiles/r1_config0_reference_cpu.json)"},
        }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


VISIT_HIST_BYTES = 64          # one env's visit history (v4 / v5): the window centre of each averaging since the reset


def dump_outputs(out_dir, outputs, obs_env0, suffix=""):
    """--dump-outputs: every output as out_dir/<name><suffix>.npy in float32.  Per-env values are kept for up to
    DUMP_ENV_VALUES envs and observation rows (tensors of more than one dimension) for DUMP_OBS_ROWS envs; a larger
    batch is sampled at indices drawn from a fixed seed, so the same arguments always keep the same envs.  The kept
    env indices (within this rank's batch) are written as env_index / obs_env_index (float64); obs_env0 is the env
    of the observation tensor's first row (the last render window's start)."""
    import numpy as np
    import torch

    def keep(n, k):
        return np.arange(n) if n <= k else np.sort(np.random.RandomState(0).choice(n, k, replace=False))
    env_rows = keep(outputs["reward"].shape[0], DUMP_ENV_VALUES)
    obs_rows = keep(outputs["obs"].shape[0], DUMP_OBS_ROWS)
    arrays = {"env_index": env_rows.astype(np.float64), "obs_env_index": (obs_env0 + obs_rows).astype(np.float64)}
    for name, t in outputs.items():
        rows = torch.from_numpy(obs_rows if t.dim() > 1 else env_rows).to(t.device)
        arrays[name] = t[rows].to(torch.float32).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def main_workload_checks(rk, lmz, env, args, hier, seed, N, W, R, action_ring, steps_done, K=1024, KO=32):
    """Shard invariance ON THE REAL GPUs (SURVEY section 4 T4): rank r's env i has global id r*N + i.  Rank 0 replays,
    for every rank r, the first K envs of r's shard -- a K-env handle with env_id0 = r*N, r's action ring, the same
    number of steps -- and compares reward bits, done flags, packed state rows and the first KO observation rows with
    what rank r computed inside its N-env batch."""
    torch = rk.torch
    if W != N:
        return {"shard_invariance": {"skipped": "render window in use"}}
    K = min(K, N)
    KO = min(KO, K)
    mine = {"reward": env.reward[:K].view(torch.int32).clone(), "done": env._done_u8[:K].clone(),
            "state": env.get_state()[:K].clone(), "obs": env.obs[:KO].clone()}
    if hier:
        mine["reward2"] = env.local_reward[:K].view(torch.int32).clone()
        mine["loc"] = env.loc_obs[:KO].clone()
    gathered = {k: rk.gather(v) for k, v in mine.items()}
    out = {"envs_replayed_per_rank": K, "obs_rows_compared": KO, "steps_replayed": steps_done, "ranks": rk.world,
           "what": "rank 0 re-runs the first %d envs of every rank's shard as a separate %d-env handle with the same "
                   "global ids and compares reward bits / done / state rows / obs rows bit for bit" % (K, K)}
    if rk.rank == 0:
        ok, bad = True, []
        for r in range(rk.world):
            ring_r, goals_r = action_ring(r)
            if hier:
                ref = lmz.LmazeHierCuda(K, "v5", device=rk.dev, seed=seed, env_id0=r * N, autoreset=True, obs_mode=args.obs_mode)
            else:
                ref = lmz.LmazeVecCuda(K, args.variant, device=rk.dev, seed=seed, env_id0=r * N, autoreset=True,
                                       render_mode=args.render_mode, obs_mode=args.obs_mode)
            ref.reset()
            for i in list(range(args.warmup)) + list(range(args.steps)):
                if hier:
                    ref.plannerStep(goals_r[i % R][:K].contiguous(), mask="auto")
                    ref.step(ring_r[i % R][:K].contiguous(), goal_plane=False)
                else:
                    ref.step(ring_r[i % R][:K].contiguous())
            same = (torch.equal(ref.reward.view(torch.int32), gathered["reward"][r])
                    and torch.equal(ref._done_u8, gathered["done"][r])
                    and torch.equal(ref.get_state(), gathered["state"][r])
                    and torch.equal(ref.obs[:KO], gathered["obs"][r]))
            if hier:
                same = same and torch.equal(ref.local_reward.view(torch.int32), gathered["reward2"][r]) \
                    and torch.equal(ref.loc_obs[:KO], gathered["loc"][r])
            if not same:
                ok = False
                bad.append(r)
            ref.close()
            del ring_r, goals_r
        out["ok"], out["mismatching_ranks"] = ok, bad
    return {"shard_invariance": out}


def _free(torch, *envs):
    for e in envs:
        e.close()
    torch.cuda.empty_cache()


def side_measurements(rk, lmz, args, seed):
    """Other operating points, each named with its own mode (never mixed into `value`).  Run on EVERY rank with the
    rank's own global-id shard; every `value` is the whole-job aggregate: world x envs x steps / max-over-ranks time."""
    torch, dev, world, rank = rk.torch, rk.dev, rk.world, rk.rank
    out = {}
    # (0) what a trivial streaming-write kernel gets on this GPU right now (8 GiB torch fill_), rank 0's GPU
    scratch = torch.empty(2 << 30, dtype=torch.float32, device=dev)
    ms = rk.timed_ms(lambda i: scratch.fill_(1.0), 20, 20)
    out["pure_write_fill_gbs"] = {"value": scratch.numel() * 4 / (ms * 1e-3) / 1e9,
                                  "what": "torch.fill_ over 8 GiB on every rank at once (slowest rank): the write-only "
                                          "ceiling; MEASURED_PEAKS hbm_gbs is a read+write copy, so a pure-write kernel "
                                          "can exceed it"}
    del scratch
    torch.cuda.empty_cache()
    if args.variant != "v0" or args.obs_mode != "full" or args.render_mode != "tma":
        return out            # the side measurements belong to the default (headline) run
    try:
        out["rollout_T64"] = rollout_measurement(rk, lmz, seed)
    except Exception as exc:  # pragma: no cover
        out["rollout_T64"] = {"error": repr(exc)}
    for name, fn in (("v3_full_render", lambda: fused_step_measurement(rk, lmz, seed, "v3", 1 << 20, reps=20)),
                     ("v0_compact", lambda: fused_step_measurement(rk, lmz, seed, "v0", 1 << 24, reps=30, obs_mode="compact")),
                     ("v3_compact", lambda: fused_step_measurement(rk, lmz, seed, "v3", 1 << 23, reps=30, obs_mode="compact")),
                     ("incremental_render", lambda: fused_step_measurement(rk, lmz, seed, "v0", 1 << 20, reps=50,
                                                                           render_mode="incremental")),
                     ("e2e_host_consumer", lambda: host_consumer_measurement(rk, lmz, seed))):
        try:
            out[name] = fn()
        except Exception as exc:  # pragma: no cover
            out[name] = {"error": repr(exc)}
        torch.cuda.empty_cache()
    if world > 1 or rank != 0:
        return out
    # ---- single-GPU host-side costs (wall clock; not multi-rank quantities)
    # (1b) BASELINE configs[1]-size batch (4,096 envs): the step is launch-bound (~65 us of GPU work), so what the host
    # side costs per call matters -- plain Python step() vs a CUDA-graph replay of the same fused launch
    try:
        n1 = 4096
        env1 = lmz.LmazeVecCuda(n1, args.variant, device=dev, seed=1, render_mode=args.render_mode)
        env1.reset()
        a1 = torch.randint(0, 4, (n1,), device=dev, dtype=torch.uint8)
        for _ in range(20):
            env1.step(a1)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(2000):
            env1.step(a1)
        torch.cuda.synchronize(dev)
        dt_py = (time.perf_counter() - t0) / 2000
        replay = env1.capture_step(a1)
        for _ in range(20):
            replay()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(2000):
            replay()
        torch.cuda.synchronize(dev)
        dt_g = (time.perf_counter() - t0) / 2000
        out["small_batch_4096"] = {"envs": n1, "python_step_us": dt_py * 1e6, "python_step_env_steps_per_s": n1 / dt_py,
                                   "graph_replay_us": dt_g * 1e6, "graph_replay_env_steps_per_s": n1 / dt_g,
                                   "mode": "BASELINE configs[1] batch size, full f32 render; wall clock over 2000 back-to-back "
                                           "calls (LmazeVecCuda.step through ctypes + DLPack vs capture_step graph replay)"}
        env1.close()
    except Exception as exc:  # pragma: no cover
        out["small_batch_4096"] = {"error": repr(exc)}
    # (2) e2e including the full observation D2H, on a bounded slice (PCIe-bound by construction)
    try:
        n2 = 16384
        env2 = lmz.LmazeVecCuda(n2, args.variant, device=dev, seed=1, render_mode=args.render_mode)
        env2.reset()
        a = torch.randint(0, 4, (n2,), dtype=torch.uint8).pin_memory()
        r = torch.empty(n2, dtype=torch.float32).pin_memory()
        d = torch.empty(n2, dtype=torch.uint8).pin_memory()
        o = torch.empty((n2,) + env2.obs_shape, dtype=torch.float32).pin_memory()
        for _ in range(2):
            env2.step_host(a, r, d, o)
        t0 = time.perf_counter()
        reps = 5
        for _ in range(reps):
            env2.step_host(a, r, d, o)
        dt = (time.perf_counter() - t0) / reps
        out["e2e_obs_to_host"] = {"value": n2 / dt, "unit": "env-steps/s", "envs": n2,
                                  "d2h_bytes_per_step": n2 * (o[0].numel() * 4 + 5),
                                  "d2h_gbs": n2 * o[0].numel() * 4 / dt / 1e9,
                                  "mode": "lmz_step_host with obs_host: every f32 obs byte copied to pinned host memory "
                                          "(PCIe-bound by construction; a host consumer should take the compact or "
                                          "bit-packed observation instead: extras.e2e_host_consumer)"}
        env2.close()
        del o
    except Exception as exc:  # pragma: no cover
        out["e2e_obs_to_host"] = {"error": repr(exc)}
    return out


def rollout_measurement(rk, lmz, seed, n=1 << 21, T=64, K=1024):
    """BASELINE configs[4]: T=64 fused rollout, device-side Philox actions, no per-step obs, 2^21 envs per GPU
    (16 M on 8).  Also the on-hardware checks: NCCL-summed step counter and shard invariance of the rollout."""
    torch, dev, world, rank = rk.torch, rk.dev, rk.world, rk.rank
    env = lmz.LmazeVecCuda(n, "v0", device=dev, seed=seed, env_id0=rank * n, autoreset=True, with_obs=False)
    env.reset()
    rew = torch.empty((T, n), dtype=torch.float32, device=dev)
    don = torch.empty((T, n), dtype=torch.uint8, device=dev)
    env.rollout(T, rewards=rew, dones=don)                      # the first rollout is the one rank 0 replays
    first = rk.gather(torch.cat([rew[:, :K].reshape(-1).view(torch.int32), don[:, :K].reshape(-1).to(torch.int32)]))
    inv = {"envs_replayed_per_rank": K, "steps": T, "ranks": world}
    if rank == 0:
        bad = []
        for r in range(world):
            ref = lmz.LmazeVecCuda(K, "v0", device=dev, seed=seed, env_id0=r * n, autoreset=True, with_obs=False)
            ref.reset()
            rr, dd = ref.rollout(T)
            want = torch.cat([rr.reshape(-1).view(torch.int32), dd.reshape(-1).to(torch.int32)])
            if not torch.equal(want, first[r]):
                bad.append(r)
            ref.close()
        inv["ok"], inv["mismatching_ranks"] = not bad, bad
    reps, warm = 10, 2
    launches0 = env.launch_count
    ms = rk.timed_ms(lambda i: env.rollout(T, rewards=rew, dones=don), reps, warm)
    stats = env.stats_allreduce() if world > 1 else env.stats()
    expected = world * n * T * (1 + reps + warm)
    res = {"value": world * n * T / (ms * 1e-3), "unit": "env-steps/s", "ms_per_rollout": ms, "envs_per_gpu": n,
           "envs_total": world * n, "T": T,
           "mode": "lmz_rollout_kernel<V0>: T fused steps, state in registers, NO per-step obs, device Philox actions, "
                   "reward f32 + done u8 [T,N] written; barrier + max over ranks",
           "bytes_per_env_step": 5.25, "achieved_gbs_per_gpu": n * T * 5.25 / (ms * 1e-3) / 1e9,
           "launches_timed": env.launch_count - launches0 - warm,
           "checks": {"nccl_steps_sum": {"steps": stats["steps"], "expected": expected, "ok": stats["steps"] == expected},
                      "shard_invariance": inv}}
    # same rollout with the 1-byte reward CODE instead of the f32 reward (2 B per env-step instead of 5)
    try:
        codes = torch.empty((T, n), dtype=torch.uint8, device=dev)
        ms2 = rk.timed_ms(lambda i: env.rollout(T, reward_codes=codes, dones=don), reps, warm)
        res["reward_code_u8"] = {"value": world * n * T / (ms2 * 1e-3), "unit": "env-steps/s", "ms_per_rollout": ms2,
                                 "bytes_per_env_step": 2.25,
                                 "mode": "same kernel, rewards written as u8 codes (0: -0.0, 1: -1.0, 2: -0.01, 3: 100.0; "
                                         "LmazeVecCuda.REWARD_TABLE[codes] is the f32 tensor)"}
        del codes
    except Exception as exc:  # pragma: no cover
        res["reward_code_u8"] = {"error": repr(exc)}
    del rew, don
    _free(torch, env)
    return res


def fused_step_measurement(rk, lmz, seed, variant, n, reps, obs_mode="full", render_mode="tma"):
    """One fused step launch per step over `n` envs per GPU in the given mode (its own bytes figure)."""
    torch, dev, world, rank = rk.torch, rk.dev, rk.world, rk.rank
    env = lmz.LmazeVecCuda(n, variant, device=dev, seed=seed, env_id0=rank * n, autoreset=True, obs_mode=obs_mode,
                           render_mode=render_mode)
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    ring = torch.randint(0, env.num_actions, (4, n), generator=gen, device=dev, dtype=torch.uint8)
    env.reset()
    launches0 = env.launch_count
    ms = rk.timed_ms(lambda i: env.step(ring[i % 4]), reps, 5)
    stats = env.stats_allreduce() if world > 1 else env.stats()
    G, E, C = {"v0": (12, 7, 4), "v3": (18, 4, 3)}[variant]
    if render_mode == "incremental":
        b, kern = 2 * E * E * 4 + 14, "lmz_env_incr_kernel"
        mode = ("persistent f32 (%d,%d,%d) obs tensor patched in place (old block erased, new block drawn); tensor content "
                "identical to the full render after every step" % (C, G * E, G * E))
    elif obs_mode == "compact":
        b, kern = C * G * G + 14, "lmz_env_compact_kernel"
        mode = "u8 (%d,%d,%d) compact observation (un-expanded layers; reference image = x%d replication)" % (C, G, G, E)
    else:
        b, kern = C * G * E * G * E * 4 + 14, "lmz_env_tma_kernel"
        mode = "f32 (%d,%d,%d) full render, fused step + auto-reset" % (C, G * E, G * E)
    expected = world * n * (reps + 5)
    res = {"value": world * n / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms, "envs_per_gpu": n,
           "envs_total": world * n, "variant": variant, "kernel": "%s<%s>" % (kern, variant.upper()), "mode": mode,
           "bytes_per_env_step": b, "achieved_gbs_per_gpu": n * b / (ms * 1e-3) / 1e9,
           "launches_timed": env.launch_count - launches0 - 5,
           "nccl_steps_sum": {"steps": stats["steps"], "expected": expected, "ok": stats["steps"] == expected}}
    del ring
    _free(torch, env)
    return res


def host_consumer_measurement(rk, lmz, seed):
    """End to end for a HOST consumer: every output of a step -- observation included -- lands in pinned host
    memory, actions come from pinned host memory, through LmazeVecCuda.step_host_pipelined (lmz_step_host_async /
    lmz_step_host_wait, double buffered: step k's D2H overlaps step k+1's kernel).  Wall clock, max over ranks."""
    torch, dev, world, rank = rk.torch, rk.dev, rk.world, rk.rank
    out = {}
    for name, variant, obs_mode, n in (("v0_compact_u8", "v0", "compact", 1 << 20), ("v0_bits", "v0", "bits", 1 << 22),
                                       ("v3_bits", "v3", "bits", 1 << 22)):
        try:
            env = lmz.LmazeVecCuda(n, variant, device=dev, seed=seed, env_id0=rank * n, autoreset=True, obs_mode=obs_mode)
            env.reset()
            pipe = env.host_pipeline()
            gen = torch.Generator().manual_seed(7 + rank)
            acts = torch.randint(0, 4, (4, n), generator=gen, dtype=torch.uint8).pin_memory()
            reps, warm = 20, 4
            for i in range(warm):
                pipe.submit(acts[i % 4])
            pipe.drain()
            rk.barrier()
            t0 = time.perf_counter()
            csum = 0
            for i in range(reps):
                res = pipe.submit(acts[i % 4])          # returns the PREVIOUS step's host buffers (or None)
                if res is not None:
                    csum += int(res.done[:64].sum())    # the host really touches the result
            last = pipe.drain()
            csum += int(last.done[:64].sum())
            dt = time.perf_counter() - t0
            rk.barrier()
            ms = rk.reduce_max(dt * 1e3) / reps
            per_env = env.obs[0].numel() * env.obs.element_size()
            out[name] = {"value": world * n / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms, "envs_per_gpu": n,
                         "h2d_bytes_per_step": n, "d2h_bytes_per_step": n * (per_env + 5), "obs_bytes_per_env": per_env,
                         "d2h_gbs_per_gpu": n * (per_env + 5) / (ms * 1e-3) / 1e9,
                         "mode": "obs_mode=%s: obs + reward + done ALL copied to pinned host memory every step, actions "
                                 "from pinned host memory, double-buffered (lmz_step_host_async/_wait)" % obs_mode,
                         "done_checksum": csum}
            del pipe, acts
            _free(torch, env)
        except Exception as exc:  # pragma: no cover
            out[name] = {"error": repr(exc)}
    return out


def main():
    args = parse_args()
    # Only the JSON line may reach stdout (NCCL / torchrun banners go to stderr).
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real_stdout, "w")
    import builtins
    _print = builtins.print

    def json_print(*a, **k):
        k.setdefault("file", out)
        _print(*a, **k)
        out.flush()
    globals()["print"] = json_print
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
