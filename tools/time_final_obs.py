"""Cost of final observations: us per env-step of API-mode auto-reset stepping, the default in-kernel reset against
``final_observation=True`` (the step without the reset, then the finish-and-reset pass of dexsim_step_final).  CUDA
events around windows of consecutive steps; the two envs alternate window by window in one process, the order flipping
every repeat; median and min..max over the repeats.  Prints the GPU's name and power limit first.

    python tools/time_final_obs.py [repeats]

Workloads (dense reward, random actions from a pool of four HBM-resident tensors):
  default_counts   1 Mi envs, config_default's 200-step episodes on the hard curriculum, counts-only; each window starts at a reset and runs
                   400 steps, so it holds two full-batch truncation waves (steps 200 and 400)
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

repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 7
CC = dx.CurriculumConfig
STEPS = 400


def gpu_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"GPU: {name}; power limit, max SM clock: {q}"


def make(n, final, track, cfg, max_steps):
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense", curriculum_config=cfg,
                                    auto_reset=True, respawn=True, loop_max_steps=max_steps, track_episodes=track, seed=42,
                                    final_observation=final)
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
    envs = {"auto_reset": make(n, False, track, cfg, max_steps), "final_obs": make(n, True, track, cfg, max_steps)}
    for env in envs.values():                   # warm-up: module load, occupancy queries, tensor maps, L2
        window(env, pool, from_reset)
    times = {k: [] for k in envs}
    for r in range(repeats):
        order = list(envs) if r % 2 == 0 else list(envs)[::-1]
        for k in order:
            times[k].append(window(envs[k], pool, from_reset))
    eps = {k: int(e.counters[:, 0].sum()) for k, e in envs.items()}
    assert eps["auto_reset"] == eps["final_obs"], eps
    resets = eps["auto_reset"] / ((repeats + 1) * STEPS * n)
    med = {k: statistics.median(v) for k, v in times.items()}
    cols = "  ".join(f"{k} {med[k]:7.2f} us/step [{min(v):7.2f} .. {max(v):7.2f}]" for k, v in times.items())
    print(f"{label:14s} n={n:8d} resets/env-step {100 * resets:5.2f} %:  {cols}  "
          f"extra {med['final_obs'] - med['auto_reset']:+6.2f} us ({100 * (med['final_obs'] / med['auto_reset'] - 1):+5.1f} %)",
          flush=True)
    del envs
    torch.cuda.empty_cache()


print(gpu_line(), flush=True)
print(f"library: {os.path.basename(dx._lib.LIB_PATH)}; {repeats} repeats of {STEPS}-step windows per variant, alternating", flush=True)
run("default_counts", 1 << 20, False, CC.hard(), 200, True)
run("default_track", 1 << 20, True, CC.hard(), 200, True)
run("easy15_counts", 1 << 20, False, CC.easy(), 15, False)
run("wide_counts", 131072, False, CC.hard(), 200, True)
