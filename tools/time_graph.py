"""API step replayed from a CUDA graph (capture_step, 8 steps per replay) vs eager stepping at mid sizes (experiments)."""
import os
import sys

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402

CC = dx.CurriculumConfig
for n in (int(a) for a in (sys.argv[1:] or ["4096", "65536", "131072", "262144", "1048576"])):
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=200, reward_type="dense", curriculum_config=CC.hard(),
                                    auto_reset=True, respawn=True, loop_max_steps=200, track_episodes=False, seed=42)
    env.reset(seed=42)
    g = torch.Generator(device="cuda").manual_seed(0)
    pool = [torch.rand(n, 15, device="cuda", generator=g) * 2 - 1 for _ in range(8)]
    for t in range(40):
        env.step(pool[t % 8])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(400):
        env.step(pool[t % 8])
    e1.record()
    torch.cuda.synchronize()
    eager = e0.elapsed_time(e1) / 400 * 1e3
    replay = env.capture_step(torch.stack(pool), steps=8)
    for _ in range(10):
        replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(50):
        replay()
    e1.record()
    torch.cuda.synchronize()
    graph = e0.elapsed_time(e1) / 400 * 1e3
    print(f"n={n:8d} eager {eager:7.2f} us/step  graph replay {graph:7.2f} us/step", flush=True)
    del env, replay
