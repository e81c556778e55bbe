"""Short, deterministic launch sequence for ncu (never a source of bench numbers).

    python tools/profile_step.py [num_envs] [variant] [auto|narrow|wide]

variant: api (step kernel, plain), api_counts (auto-reset + counters, the bench path), api_track (auto-reset +
full episode tracking), api_noisy (sigma_obs 0.05 + sigma_dyn 0.1 drawn in-kernel), fused (rollout kernel).
The last argument sets the tile width of the pipelined step kernel (default auto).
8 warm-up launches, then 6 profiled-range launches.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
variant = sys.argv[2] if len(sys.argv) > 2 else "api_track"
_lib.set_step_tile(sys.argv[3] if len(sys.argv) > 3 else "auto")
CC = dx.CurriculumConfig
kw = dict(max_episode_steps=200, reward_type="dense", curriculum_config=CC.hard(), seed=42)
if variant == "api":
    env = dx.BatchedManipulationEnv(n, "cuda", **kw)
elif variant == "api_noisy":
    env = dx.BatchedManipulationEnv(n, "cuda", observation_noise_std=0.05, dynamics_noise_std=0.1, **kw)
elif variant in ("api_track", "api_counts", "api_counts_easy", "api_track_easy"):
    if variant.endswith("_easy"):        # 15-step episodes: ~6.7 % of the envs reset every step
        kw["curriculum_config"] = CC.easy()
    env = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, respawn=True, loop_max_steps=200,
                                    track_episodes=variant.startswith("api_track"), **kw)
else:
    env = dx.BatchedManipulationEnv(n, "cuda", track_episodes=True, **kw)
if os.environ.get("DEXSIM_ALTERNATE", "1") == "0":      # walk the batch in the same direction every step (A/B of the L2 reuse)
    env._alternate_tiles = 0
env.reset(seed=42)
g = torch.Generator(device="cuda").manual_seed(0)
pool = [torch.rand(n, 15, device="cuda", generator=g) * 2 - 1 for _ in range(4)]
for t in range(14 if not variant.endswith('_easy') else 44):
    if variant == "fused":
        env.rollout(20, policy="random")
    else:
        env.step(pool[t % 4])
torch.cuda.synchronize()
print("done", variant, n)
