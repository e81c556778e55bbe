"""Cost of the next-step auto-reset: us per env-step of API-mode auto-reset stepping, the default same-step reset against
``final_observation=True`` (the step without the reset, then the finish-and-reset pass of dexsim_step_final) and
``autoreset_mode="next_step"`` (dexsim_step_next_reset: one launch, a finished env resets on its next step).  CUDA events
around windows of consecutive steps; the three envs alternate window by window in one process, the order rotating every
repeat; median and min..max over the repeats.  Prints the GPU's name and power limit first.

    python tools/time_next_step.py [repeats]
    python tools/time_next_step.py --profile       # torch.profiler kernel times of each variant, 1 Mi envs, easy15_counts

Workloads (dense reward, random actions from a pool of four HBM-resident tensors; those of tools/time_final_obs.py):
  default_counts   1 Mi envs, config_default's 200-step episodes on the hard curriculum, counts-only; each window starts at a reset and runs
                   400 steps, so it holds two full-batch truncation waves (steps 200 and 400; the next-step env resets them
                   on the step after, 201, inside the window, and 401, in the next window)
  default_track    the same with full episode tracking
  easy15_counts    1 Mi envs, easy curriculum, 15-step episodes (truncations and successes: ~12 % resets per env-step), counts-only, 400 steps
  wide_counts      131,072 envs (the pipeline's wide tile), 200-step episodes, counts-only, 400 steps
"""
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402

PROFILE = "--profile" in sys.argv
args = [a for a in sys.argv[1:] if not a.startswith("--")]
repeats = int(args[0]) if args else 7
CC = dx.CurriculumConfig
STEPS = 400
VARIANTS = {"same_step": {}, "final_obs": dict(final_observation=True), "next_step": dict(autoreset_mode="next_step")}


def gpu_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"GPU: {name}; power limit, max SM clock: {q}"


def make(n, variant, track, cfg, max_steps):
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense", curriculum_config=cfg,
                                    auto_reset=True, respawn=True, loop_max_steps=max_steps, track_episodes=track, seed=42,
                                    **VARIANTS[variant])
    env.reset(seed=42)
    return env


def window(env, pool, from_reset):
    if from_reset:
        env.reset(seed=42)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for t in range(STEPS):
        env.step(pool[t % len(pool)])
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) * 1e3 / STEPS


def run(label, n, track, cfg, max_steps, from_reset):
    g = torch.Generator(device="cuda").manual_seed(0)
    pool = [torch.rand(n, 15, device="cuda", generator=g) * 2 - 1 for _ in range(4)]
    envs = {k: make(n, k, track, cfg, max_steps) for k in VARIANTS}
    for env in envs.values():                   # warm-up: module load, occupancy queries, tensor maps, L2
        window(env, pool, from_reset)
    times = {k: [] for k in envs}
    names = list(envs)
    for r in range(repeats):
        order = names[r % 3:] + names[:r % 3]
        for k in order:
            times[k].append(window(envs[k], pool, from_reset))
    eps = {k: int(e.counters[:, 0].sum()) for k, e in envs.items()}
    resets = eps["same_step"] / ((repeats + 1) * STEPS * n)
    med = {k: statistics.median(v) for k, v in times.items()}
    cols = "  ".join(f"{k} {med[k]:7.2f} us/step [{min(v):7.2f} .. {max(v):7.2f}]" for k, v in times.items())
    rel = lambda k: f"{k} {med[k] - med['same_step']:+6.2f} us ({100 * (med[k] / med['same_step'] - 1):+5.1f} %)"
    print(f"{label:14s} n={n:8d} resets/env-step {100 * resets:5.2f} %:  {cols}  vs same_step: {rel('final_obs')}, "
          f"{rel('next_step')}  episodes {eps}", flush=True)
    del envs
    torch.cuda.empty_cache()


def profile(n=1 << 20, steps=60):
    """Per-kernel device time of each variant over `steps` steps of the easy15_counts workload."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    g = torch.Generator(device="cuda").manual_seed(0)
    pool = [torch.rand(n, 15, device="cuda", generator=g) * 2 - 1 for _ in range(4)]
    for k in VARIANTS:
        env = make(n, k, False, CC.easy(), 15)
        for t in range(2 * steps):             # warm-up into the steady reset rate
            env.step(pool[t % 4])
        torch.cuda.synchronize()
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(steps):
                env.step(pool[t % 4])
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA":
                name = ev.name.split("(")[0].replace("void ", "")
                per.setdefault(name, []).append(ev.device_time)
        print(f"[{k}] kernel device time over {steps} steps, n={n}:", flush=True)
        for name, v in sorted(per.items(), key=lambda kv: -sum(kv[1])):
            print(f"    {sum(v) / steps:8.2f} us/step  {len(v):4d} launches  {name[:110]}", flush=True)
        del env
        torch.cuda.empty_cache()


print(gpu_line(), flush=True)
if PROFILE:
    profile()
    sys.exit(0)
print(f"library: {os.path.basename(dx._lib.LIB_PATH)}; {repeats} repeats of {STEPS}-step windows per variant, rotating", flush=True)
run("default_counts", 1 << 20, False, CC.hard(), 200, True)
run("default_track", 1 << 20, True, CC.hard(), 200, True)
run("easy15_counts", 1 << 20, False, CC.easy(), 15, False)
run("wide_counts", 131072, False, CC.hard(), 200, True)
