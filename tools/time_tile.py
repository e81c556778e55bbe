"""Pipelined step kernel only, per batch size and variant: CUDA-event time per step.  Run once per tile width, or once per
experiment build (DEXSIM_LIB_PATH=exp/lib....so), to compare tile widths / CTA shapes (experiments only, not a bench
number source).

    python tools/time_tile.py [sizes,comma,separated] [reps] [variants,comma,separated] [auto|narrow|wide]
"""
import os
import sys

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402
from dexterous_rl_manipulation_b200 import _lib  # noqa: E402

CC = dx.CurriculumConfig
sizes = [int(x) for x in sys.argv[1].split(",")] if len(sys.argv) > 1 else [32768, 65536, 131072, 196608, 262144, 524288, 1048576]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 300
variants = sys.argv[3].split(",") if len(sys.argv) > 3 else ["plain", "counts", "track"]
tile = sys.argv[4] if len(sys.argv) > 4 else "auto"
_lib.set_step_impl("tma")
_lib.set_step_tile(tile)
print("lib", os.environ.get("DEXSIM_LIB_PATH", "default"), "tile", tile, flush=True)
for n in sizes:
    g = torch.Generator(device="cuda").manual_seed(0)
    pool = [torch.rand(n, 15, device="cuda", generator=g) * 2 - 1 for _ in range(4)]
    out = []
    for variant in variants:
        kw = dict(max_episode_steps=200, reward_type="dense", curriculum_config=CC.hard(), seed=42)
        if variant != "plain":
            kw.update(auto_reset=True, respawn=True, loop_max_steps=200, track_episodes=variant == "track")
        env = dx.BatchedManipulationEnv(n, "cuda", **kw)
        env.reset(seed=42)
        for t in range(50):
            env.step(pool[t % 4])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for t in range(reps):
            env.step(pool[t % 4])
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / reps * 1e3
        out.append(f"{variant} {us:7.2f} us (frac {410 * n / us / 1e3 / 6552:5.3f})")
        del env
    print(f"n={n:8d}  " + "   ".join(out), flush=True)
