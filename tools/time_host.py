"""End-to-end host path timing (experiments): env.step_host with pinned buffers at several chunk counts."""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=200, reward_type="dense", seed=1, auto_reset=True, respawn=True,
                                loop_max_steps=200, track_episodes=False, curriculum_config=dx.CurriculumConfig.easy())
env.reset(seed=1)
pool = [torch.rand(n, 15).mul_(2).sub_(1).pin_memory() for _ in range(2)]
env.host_zero_copy = False                         # the copy transport first
for chunks in (1, 4, 8, 12, 16):
    for t in range(3):
        env.step_host(pool[t % 2], chunks=chunks)
    t0 = time.perf_counter()
    for t in range(20):
        env.step_host(pool[t % 2], chunks=chunks)
    dt = (time.perf_counter() - t0) / 20
    print(f"chunks {chunks:3d}: {dt * 1e3:6.3f} ms/step  {n / dt / 1e6:7.1f} M env-steps/s  D2H {(41 * 4 + 7) * n / dt / 1e9:5.1f} GB/s", flush=True)

for chunks in (8, 16):
    for t in range(3):
        env.step_host(pool[t % 2], chunks=chunks, sync=False, slot=t % 2)
    env.host_sync()
    t0 = time.perf_counter()
    for t in range(20):
        env.step_host(pool[t % 2], chunks=chunks, sync=False, slot=t % 2)
    env.host_sync()
    dt = (time.perf_counter() - t0) / 20
    print(f"async chunks {chunks:3d}: {dt * 1e3:6.3f} ms/step  {n / dt / 1e6:7.1f} M env-steps/s", flush=True)

# zero-copy: actions uploaded by the copy engine, results written to pinned host memory by the kernel itself
env.host_zero_copy = True
from dexterous_rl_manipulation_b200 import _lib  # noqa: E402
L = _lib.lib()
for packed in (False, True):
    for chunks in (1, 2, 4, 8, 16):
        for t in range(3):
            env.step_host(pool[t % 2], chunks=chunks, packed_contacts=packed)
        z0 = int(L.dexsim_host_zero_copy_steps())
        t0 = time.perf_counter()
        for t in range(20):
            env.step_host(pool[t % 2], chunks=chunks, packed_contacts=packed)
        dt = (time.perf_counter() - t0) / 20
        print(f"zero-copy chunks {chunks:3d} packed={int(packed)}: {dt * 1e3:6.3f} ms/step  {n / dt / 1e6:7.1f} M env-steps/s  "
              f"(zero-copy launches {int(L.dexsim_host_zero_copy_steps()) - z0}/20)",
              flush=True)
