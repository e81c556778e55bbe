"""Cost of recording the fused rollout's trajectory: ``rollout(50)`` with the in-kernel random policy, plain, with
``enable_trajectory`` (dexsim_rollout_record, 247 bytes written per env-step: observation 180, action 60, reward 4, three
flags 3) and with ``enable_trajectory(final_observation=True)`` (dexsim_rollout_record_final: also the 180-byte terminal
observation of every env-step that ends an episode).  CUDA events around each call; the three envs take turns call by
call in one process, the order rotating every repeat; median and min..max over the repeats.  Prints the GPU's name and
power limit first.

    python tools/time_rollout_trajectory.py [repeats]

Reported per workload and size: us per rollout step (all envs), env-steps/s, and for the recording envs the trajectory
bytes written over the call time against the 6,552 GB/s measured copy peak the bench uses (MEASURED_PEAKS.json).  The
terminal observations count 180 bytes per finished env-step (the useful bytes: a finished lane alone in its warp still
costs 45 sector writes of 32 bytes), at the mean rate of all calls from the episode counters.  The buffers of a 1 Mi-env
recording (13 GB, 22 GB with terminal observations) are far larger than the 126 MB L2, so every row goes to HBM.

Workloads (full episode tracking, rollout()'s requirement, and respawn):
  long:  hard curriculum, dense reward, 200-step episodes -- most episodes end in truncation waves, few resets per step;
  short: easy curriculum, dense reward, 15-step episodes -- a high reset rate, the worst case for the terminal
         observations' scattered stores.
"""
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
repeats = int(args[0]) if args else 9
K = 50
ROW_BYTES = 247
OBS_BYTES = 180
COPY_PEAK_GBS = 6552.0


def gpu_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"GPU: {name}; power limit, max SM clock: {q}"


WORKLOADS = {
    "long": dict(max_episode_steps=200, curriculum_config=dx.CurriculumConfig.hard()),
    "short": dict(max_episode_steps=15, curriculum_config=dx.CurriculumConfig.easy()),
}
VARIANTS = ("plain", "recorded", "final")


def make(n, workload, variant):
    env = dx.BatchedManipulationEnv(n, "cuda", reward_type="dense", track_episodes=True, seed=42, **WORKLOADS[workload])
    env.reset(seed=42)
    if variant != "plain":
        env.enable_trajectory(K, final_observation=variant == "final")
    return env


def call_ms(env):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    env.rollout(K, policy="random")
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end)


def run(n, workload):
    envs = {v: make(n, workload, v) for v in VARIANTS}
    for env in envs.values():                   # warm-up: module load, occupancy query, first touch of the buffers
        call_ms(env)
    times = {k: [] for k in envs}
    for r in range(repeats):
        for j in range(len(VARIANTS)):
            k = VARIANTS[(r + j) % len(VARIANTS)]
            times[k].append(call_ms(envs[k]))
    eps = {k: int(e.counters[:, 0].sum()) for k, e in envs.items()}
    assert len(set(eps.values())) == 1, eps
    fin = eps["final"] / (repeats + 1)                          # finished env-steps per call, the warm-up call included
    print(f"{workload}: n={n}, {fin / (n * K):.4f} finished per env-step", flush=True)
    med = {k: statistics.median(v) for k, v in times.items()}
    for k, v in times.items():
        us_step = med[k] * 1e3 / K
        line = (f"n={n:8d} {workload:5s} {k:8s} {us_step:8.2f} us/step [{min(v) * 1e3 / K:8.2f} .. {max(v) * 1e3 / K:8.2f}]  "
                f"{n * K / (med[k] * 1e-3):.3e} env-steps/s")
        if k != "plain":
            nbytes = ROW_BYTES * n * K + (OBS_BYTES * fin if k == "final" else 0)   # per call, on average
            gbs = nbytes / (med[k] * 1e-3) / 1e9
            line += (f"  trajectory writes {gbs:7.1f} GB/s = {gbs / COPY_PEAK_GBS:5.3f} of the {COPY_PEAK_GBS:,.0f} GB/s copy "
                     f"peak;  {med[k] / med['plain']:5.2f}x the plain call")
            if k == "final":
                line += f", {med[k] / med['recorded']:5.3f}x the recorded call"
        print(line, flush=True)
    del envs
    torch.cuda.empty_cache()


print(gpu_line(), flush=True)
print(f"rollout({K}, policy='random'); {repeats} repeats per variant, rotating", flush=True)
for workload in WORKLOADS:
    run(1 << 20, workload)
    run(131072, workload)
