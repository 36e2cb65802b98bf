#!/usr/bin/env python
"""Cost of the final-observation pre-pass (lmz_bind_final, lmz_final.cuh) on the configurations bench.py quotes:
    python tools/final_obs_bench.py [--out DIR] [--warmup 1000] [--pairs 3]
writes DIR/r3_final_obs_bench.json and DIR/r3_final_obs_bench.log (DIR defaults to the current directory).

On ONE handle per configuration the final buffer is alternately unbound and bound (`--pairs` pairs), each timed over
K steps with CUDA events on the launch stream, in the steady state (`--warmup` steps first: the episodes start together
after the reset and need about 1,000 steps to de-synchronise, bench.py's foveal warm-up).  Then the worst step: after a
fresh reset() every env times out in the same step (an action that never reaches the goal), so that step writes every
final row; it is timed unbound and bound.  Actions come from a u8 ring [4, N] resident in HBM, as in bench.py."""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# variant, render_mode, obs_mode, envs, timed steps per measurement
CONFIGS = [("v0", "tma", "full", 1 << 20, 30), ("v0", "incremental", "full", 1 << 20, 200),
           ("v0", "tma", "compact", 1 << 24, 100), ("v0", "tma", "bits", 1 << 24, 100),
           ("v3", "tma", "full", 1 << 20, 30),
           ("v2", "tma", "full", 1 << 22, 30), ("v2", "tma", "compact", 1 << 24, 100),
           ("v4", "tma", "full", 1 << 21, 30), ("v4", "tma", "compact", 1 << 23, 100)]
STEP_LIMIT = {"v0": 100, "v3": 101, "v2": 51, "v4": 51}     # the step at which a no-goal episode times out
NO_MOVE = {"v0": 7, "v3": 7, "v2": 12, "v4": 12}             # an action that never reaches the goal


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def run_config(lmz, _abi, variant, render_mode, obs_mode, n, k, warmup, pairs, log):
    import torch
    env = lmz.LmazeVecCuda(n, variant, seed=1, render_mode=render_mode, obs_mode=obs_mode, final_obs=True)
    L, final = env._lib, env.final_obs
    mode = _abi.OBS_BITS if obs_mode == "bits" else _abi.OBS_COMPACT
    stream = torch.cuda.current_stream()

    def bind(on):
        _abi.call(L.lmz_bind_final_dl, env._h, final if on else None, mode)

    gen = torch.Generator(device="cuda").manual_seed(3)
    ring = torch.randint(0, env.num_actions, (4, n), generator=gen, device="cuda", dtype=torch.uint8)
    no_move = torch.full((n,), NO_MOVE[variant], dtype=torch.uint8, device="cuda")

    def timed(steps, actions_of):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            env._step(actions_of(i), None)          # the ABI call alone: lmz_step_dl
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / steps

    env.reset()
    bind(True)
    t0 = time.time()
    for i in range(warmup):
        env._step(ring[i & 3], None)
    torch.cuda.synchronize()
    rec = {"variant": variant, "render_mode": render_mode, "obs_mode": obs_mode, "envs": n, "steps_per_measurement": k,
           "warmup_steps": warmup, "final_row_bytes": final[0].numel() * final.element_size(), "pairs": []}
    for _ in range(pairs):
        pair = {}
        for on in (False, True):
            bind(on)
            timed(3, lambda i: ring[i & 3])
            pair["bound" if on else "unbound"] = timed(k, lambda i: ring[i & 3])
        rec["pairs"].append(pair)
    # the synchronised time-out step right after a reset: every env finishes, every final row is written
    rec["sync_step"] = {}
    for on in (False, True):
        bind(on)
        env.reset()
        for _ in range(STEP_LIMIT[variant] - 1):
            env._step(no_move, None)
        ms = timed(1, lambda i: no_move)
        rec["sync_step"]["bound" if on else "unbound"] = ms
        rec["sync_step"]["done_fraction"] = float(env.done.float().mean())
    unb = sorted(p["unbound"] for p in rec["pairs"])[pairs // 2]
    bnd = sorted(p["bound"] for p in rec["pairs"])[pairs // 2]
    rec["median_ms"] = {"unbound": unb, "bound": bnd}
    rec["overhead_pct"] = 100.0 * (bnd - unb) / unb
    rec["env_steps_per_s"] = {"unbound": n / unb * 1e3, "bound": n / bnd * 1e3}
    s = rec["sync_step"]
    rec["sync_overhead_pct"] = 100.0 * (s["bound"] - s["unbound"]) / s["unbound"]
    log("%-3s %-11s %-7s 2^%-2d  steady: unbound %.4f ms  bound %.4f ms  (%+.2f %%)   sync step: unbound %.4f ms  "
        "bound %.4f ms (%+.1f %%, %.3f of envs done)   [%.0f s]"
        % (variant, render_mode, obs_mode, n.bit_length() - 1, unb, bnd, rec["overhead_pct"], s["unbound"], s["bound"],
           rec["sync_overhead_pct"], s["done_fraction"], time.time() - t0))
    env.close()
    del env, final, ring, no_move
    gc.collect()
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".")
    ap.add_argument("--warmup", type=int, default=1000)
    ap.add_argument("--pairs", type=int, default=3)
    args = ap.parse_args()
    import torch
    import gym_lmaze_b200 as lmz
    from gym_lmaze_b200 import _abi
    if not torch.cuda.is_available():
        raise SystemExit("final_obs_bench.py measures on the GPU: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    lines = []

    def log(msg):
        print(msg, flush=True)
        lines.append(msg)

    info = card()
    log("card: %s | %s" % (info["torch_name"], info["nvidia_smi"]))
    doc = {"what": "ms per lmz_step (CUDA events over K steps) with the final-observation buffer unbound / bound on the "
                   "same handle, alternated; the synchronised time-out step after reset() (every final row written)",
           "card": info, "warmup_steps": args.warmup, "configs": []}
    for variant, render_mode, obs_mode, n, k in CONFIGS:
        doc["configs"].append(run_config(lmz, _abi, variant, render_mode, obs_mode, n, k, args.warmup, args.pairs, log))
    log("card (end of run): %s" % card()["nvidia_smi"])
    with open(os.path.join(args.out, "r3_final_obs_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    with open(os.path.join(args.out, "r3_final_obs_bench.log"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
