"""Cost of final observations on the host-buffer step: us per step of ``step_host()`` (NumPy-side policies, pinned
host buffers, synchronous calls) for an auto-reset env without and with ``final_observation=True``
(dexsim_step_host vs dexsim_step_host_final).  Every call ends in a stream synchronize, so a host clock around each call
times the whole step: upload, kernels, downloads.  The two envs alternate window by window in one process, the order
flipping every repeat; median and min..max over the repeats of each window's mean.  Prints the GPU's name and power
limit first.

    python tools/time_host_final_obs.py [repeats]

Workloads (dense reward, random actions from a pool of four pinned host arrays; default chunking):
  default_counts   1 Mi envs, 200-step episodes on the hard curriculum, counts-only, copy transport; each window starts
                   at a reset and runs 400 steps.  The two full-batch truncation-wave steps (200 and 400) are reported
                   apart from the other 398 ("steady").
  easy15_counts    1 Mi envs, easy curriculum, 15-step episodes (~12 % resets per env-step), counts-only, 400 steps
  zc_131072        131,072 envs, 200-step episodes, counts-only, zero-copy transport (wide tile), 400 steps from a reset
  zc_32768         32,768 envs, the same
"""
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402

repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 5
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


def make(n, final, cfg, max_steps):
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense", curriculum_config=cfg,
                                    auto_reset=True, respawn=True, loop_max_steps=max_steps, track_episodes=False, seed=42,
                                    final_observation=final)
    env.reset(seed=42)
    return env


def window(env, pool, from_reset, wave_every):
    """Per-step seconds of one window: (steady steps, truncation-wave steps)."""
    if from_reset:
        env.reset(seed=42)
    steady, wave = [], []
    for t in range(STEPS):
        t0 = time.perf_counter()
        env.step_host(pool[t % len(pool)])
        dt = time.perf_counter() - t0
        (wave if wave_every and (t + 1) % wave_every == 0 else steady).append(dt)
    return steady, wave


def run(label, n, cfg, max_steps, from_reset, zero_copy):
    g = torch.Generator().manual_seed(0)
    pool = [(torch.rand(n, 15, generator=g) * 2 - 1).pin_memory() for _ in range(4)]
    envs = {"step_host": make(n, False, cfg, max_steps), "step_host_final": make(n, True, cfg, max_steps)}
    wave_every = max_steps if from_reset else 0
    for env in envs.values():                   # warm-up: module load, occupancy queries, tensor maps, pinned buffers
        window(env, pool, from_reset, wave_every)
    zc0 = dx._lib.lib().dexsim_host_zero_copy_steps()
    steady = {k: [] for k in envs}
    waves = {k: [] for k in envs}
    for r in range(repeats):
        order = list(envs) if r % 2 == 0 else list(envs)[::-1]
        for k in order:
            s, w = window(envs[k], pool, from_reset, wave_every)
            steady[k].append(statistics.fmean(s) * 1e6)
            waves[k] += [x * 1e6 for x in w]
    zc = dx._lib.lib().dexsim_host_zero_copy_steps() - zc0
    assert (zc == 2 * repeats * (STEPS - 1)) if zero_copy else zc == 0, zc   # the first call of a window primes the buffer
    eps = {k: int(e.counters[:, 0].sum()) for k, e in envs.items()}
    assert eps["step_host"] == eps["step_host_final"], eps
    resets = eps["step_host"] / ((repeats + 1) * STEPS * n)
    med = {k: statistics.median(v) for k, v in steady.items()}
    cols = "  ".join(f"{k} {med[k]:8.1f} us/step [{min(v):8.1f} .. {max(v):8.1f}]" for k, v in steady.items())
    print(f"{label:14s} n={n:8d} {'zero-copy' if zero_copy else 'copies   '} resets/env-step {100 * resets:5.2f} %:  "
          f"{'steady ' if wave_every else ''}{cols}  extra {med['step_host_final'] - med['step_host']:+7.1f} us "
          f"({100 * (med['step_host_final'] / med['step_host'] - 1):+5.1f} %)", flush=True)
    if wave_every:
        wm = {k: statistics.median(v) for k, v in waves.items()}
        cols = "  ".join(f"{k} {wm[k]:8.1f} us [{min(v):8.1f} .. {max(v):8.1f}]" for k, v in waves.items())
        print(f"{'':14s} {'':10s} truncation-wave step ({len(waves['step_host'])} per variant):  {cols}  "
              f"extra {wm['step_host_final'] - wm['step_host']:+7.1f} us", flush=True)
    del envs
    torch.cuda.empty_cache()


print(gpu_line(), flush=True)
print(f"library: {os.path.basename(dx._lib.LIB_PATH)}; {repeats} repeats of {STEPS}-step windows per variant, alternating; "
      f"host clock around each synchronous step_host() call", flush=True)
run("default_counts", 1 << 20, CC.hard(), 200, True, False)
run("easy15_counts", 1 << 20, CC.easy(), 15, False, False)
run("zc_131072", 131072, CC.hard(), 200, True, True)
run("zc_32768", 32768, CC.hard(), 200, True, True)
