"""Long-run consistency soak (not a benchmark): the TMA pipeline kernel vs the register kernel over many
thousands of back-to-back launches with auto-reset, counters and ragged tiles; then the chunked host path.

    python tools/soak.py [num_envs] [steps] [full|counts] [auto|narrow|wide]
"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402
from dexterous_rl_manipulation_b200 import _lib  # noqa: E402

CC = dx.CurriculumConfig
n, steps = int(sys.argv[1]) if len(sys.argv) > 1 else 300_007, int(sys.argv[2]) if len(sys.argv) > 2 else 20_000
full = (sys.argv[3] if len(sys.argv) > 3 else "full") == "full"       # "counts": auto-reset + counters only
_lib.set_step_tile(sys.argv[4] if len(sys.argv) > 4 else "auto")       # tile width of the pipelined kernel
kw = dict(max_episode_steps=60, reward_type="dense", auto_reset=True, respawn=True, loop_max_steps=60, track_episodes=full,
          groups=[CC.easy(), CC.medium(), CC.hard()], seed=77)
envs = {impl: dx.BatchedManipulationEnv(n, "cuda", **kw) for impl in ("register", "tma")}
for e in envs.values():
    e.reset(seed=77)
g = torch.Generator(device="cuda").manual_seed(0)
pool = [torch.rand(n, 15, device="cuda", generator=g) * 2.2 - 1.1 for _ in range(7)]
t0 = time.time()
for t in range(steps):
    for impl, e in envs.items():
        _lib.set_step_impl(impl)
        e.step(pool[t % 7])
    if (t + 1) % 5000 == 0:
        a, b = envs["register"], envs["tma"]
        keys = ("_obs", "_op64", "_step_count", "_cmask", "_episode", "counters", "_thr", "_damp") + (("_ep_stats", "_ep_return") if full else ())
        ok = all(torch.equal(getattr(a, k), getattr(b, k)) for k in keys)
        print(f"step {t + 1}: equal={ok} episodes={int(a.counters[:, 0].sum())} ({time.time() - t0:.1f}s)", flush=True)
        assert ok
_lib.set_step_impl("auto")
a, b = envs["register"], envs["tma"]
for t in range(300):
    act = pool[t % 7]
    a.step(act)
    b.step_host(act.cpu().pin_memory(), chunks=1 + t % 8)
assert torch.equal(a._obs, b._obs) and torch.equal(a.counters, b.counters) and (not full or torch.equal(a._ep_return, b._ep_return))
print("host path equal after 300 chunked steps; soak ok")
