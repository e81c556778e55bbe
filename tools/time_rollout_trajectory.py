"""Cost of recording the fused rollout's trajectory: ``rollout(50)`` with the in-kernel random policy, without and with
``enable_trajectory`` (dexsim_rollout_record, 247 bytes written per env-step: observation 180, action 60, reward 4, three
flags 3).  CUDA events around each call; the two envs alternate call by call in one process, the order swapping every
repeat; median and min..max over the repeats.  Prints the GPU's name and power limit first.

    python tools/time_rollout_trajectory.py [repeats]

Reported per size: us per rollout step (all envs), env-steps/s, and for the recording env the trajectory bytes written
over the call time against the 6,552 GB/s measured copy peak the bench uses (MEASURED_PEAKS.json).  The buffers of a
1 Mi-env recording (13 GB) are far larger than the 126 MB L2, so every row goes to HBM.

Workload: hard curriculum, dense reward, 200-step episodes, full episode tracking (rollout()'s requirement), respawn.
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
COPY_PEAK_GBS = 6552.0


def gpu_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"GPU: {name}; power limit, max SM clock: {q}"


def make(n, record):
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=200, reward_type="dense",
                                    curriculum_config=dx.CurriculumConfig.hard(), track_episodes=True, seed=42)
    env.reset(seed=42)
    if record:
        env.enable_trajectory(K)
    return env


def call_ms(env):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    env.rollout(K, policy="random")
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end)


def run(n):
    envs = {"plain": make(n, False), "recorded": make(n, True)}
    for env in envs.values():                   # warm-up: module load, occupancy query, first touch of the buffers
        call_ms(env)
    times = {k: [] for k in envs}
    for r in range(repeats):
        for k in (("plain", "recorded") if r % 2 == 0 else ("recorded", "plain")):
            times[k].append(call_ms(envs[k]))
    med = {k: statistics.median(v) for k, v in times.items()}
    for k, v in times.items():
        us_step = med[k] * 1e3 / K
        line = (f"n={n:8d} {k:8s} {us_step:8.2f} us/step [{min(v) * 1e3 / K:8.2f} .. {max(v) * 1e3 / K:8.2f}]  "
                f"{n * K / (med[k] * 1e-3):.3e} env-steps/s")
        if k == "recorded":
            gbs = ROW_BYTES * n * K / (med[k] * 1e-3) / 1e9
            line += (f"  trajectory writes {gbs:7.1f} GB/s = {gbs / COPY_PEAK_GBS:5.3f} of the {COPY_PEAK_GBS:,.0f} GB/s copy "
                     f"peak;  {med[k] / med['plain']:5.2f}x the plain call")
        print(line, flush=True)
    eps = {k: int(e.counters[:, 0].sum()) for k, e in envs.items()}
    assert eps["plain"] == eps["recorded"], eps
    del envs
    torch.cuda.empty_cache()


print(gpu_line(), flush=True)
print(f"rollout({K}, policy='random'); {repeats} repeats per variant, alternating", flush=True)
run(1 << 20)
run(131072)
