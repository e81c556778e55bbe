"""Cost of the in-kernel action fill (dexsim_fill_mlp_actions) and of stepping and evaluating with it.

    python tools/time_policy_actions.py [repeats] [--out PATH]     (writes profiles/r10_policy_actions.txt by default)

1. fill kernel: dexsim_fill_mlp_actions into a preallocated [15, ld] buffer, per launch, [64, 64] ReLU and tanh
   (action_std 0.1), at 131,072 and 1,048,576 envs; CUDA events around 20 back-to-back launches.
2. stepping, per env-step, at the same sizes with the ReLU policy, 50 steps of an auto-reset env per call:
     fill:        50 x step(policy_actions(mlp));
     composition: 50 x step(clip(mlp.mean(obs) + std * fill_normal(stream 4))) -- the three launches the fill replaces,
                  on the observation step() returned;
     rollout:     rollout(50, policy=mlp), the network inside the fused rollout, for scale.
   The three take turns call by call, the order rotating every repeat; median and min..max over the repeats.
3. evaluate_heldout_set_batched, 20 held-out objects x 5,000 episodes (100,000 envs, 200-step episodes, contact history
   on), the ReLU MLP against the heuristic policy; wall clock of the whole call (launch, read-back and
   result dictionaries), two calls after one warm-up call each.
Prints the GPU's name and power limit first.  Workload: hard curriculum, dense reward, tracking on.
"""
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402
from dexterous_rl_manipulation_b200 import _lib  # noqa: E402
from run_baseline_configs import _HeldOut  # noqa: E402

argv = sys.argv[1:]
OUT = os.path.join(ROOT, "profiles", "r10_policy_actions.txt")
if "--out" in argv:
    OUT = argv[argv.index("--out") + 1]
    del argv[argv.index("--out"):argv.index("--out") + 2]
repeats = int(argv[0]) if argv else 7
K, STD, FILLS = 50, 0.1, 20
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


def gpu_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"GPU: {name}; power limit, max SM clock: {q}"


def make_env(n, **kw):
    env = dx.BatchedManipulationEnv(n, "cuda", reward_type="dense", track_episodes=True, seed=42, max_episode_steps=200,
                                    curriculum_config=dx.CurriculumConfig.hard(), **kw)
    env.reset(seed=42)
    return env


def timed(fn):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end)


def policy(act):
    torch.manual_seed(0)
    A = torch.nn.ReLU if act == "relu" else torch.nn.Tanh
    net = torch.nn.Sequential(torch.nn.Linear(45, 64), A(), torch.nn.Linear(64, 64), A(), torch.nn.Linear(64, 15))
    return dx.MlpPolicy.from_torch(net, action_std=STD)


def fill_kernel(n, pols):
    env = make_env(n)
    env._sync_groups()
    out = torch.empty(15, env.ld, device="cuda")

    def launches(pol):
        for _ in range(FILLS):
            _lib.check(env._lib.dexsim_fill_mlp_actions(C.byref(env._state), C.byref(env._params),
                                                        env._ptr(env._groups_dev), env._ptr(env._goe),
                                                        C.byref(pol._struct), out.data_ptr(), env._stream()),
                       "dexsim_fill_mlp_actions")

    for act, pol in pols.items():
        assert torch.equal(env.policy_actions(pol), env.policy_actions(pol))   # warm-up: module load, smem attribute
        ms = [timed(lambda: launches(pol)) for _ in range(repeats)]
        med = statistics.median(ms)
        emit(f"fill   n={n:8d} {act:4s} {med * 1e3 / FILLS:9.2f} us/launch [{min(ms) * 1e3 / FILLS:9.2f} .. "
             f"{max(ms) * 1e3 / FILLS:9.2f}]  {n * FILLS / (med * 1e-3):.3e} actions/s")
    del env


def fill_normal(env, out):
    _lib.check(env._lib.dexsim_fill_normal(C.byref(env._state), C.byref(env._params), 4, 15, C.c_float(1.0),
                                           out.data_ptr(), env._stream()), "dexsim_fill_normal")
    return out[:, :env.num_envs].t()


def stepping(n, pol):
    fill_env = make_env(n, auto_reset=True, loop_max_steps=200)
    comp_env = make_env(n, auto_reset=True, loop_max_steps=200)
    roll_env = make_env(n)
    z = torch.zeros(15, comp_env.ld, device="cuda")
    std = pol.action_std[:15]

    def fill_steps():
        for _ in range(K):
            fill_env.step(fill_env.policy_actions(pol))

    def comp_steps():
        o = comp_env._obs_view
        for _ in range(K):
            a = (pol.mean(o) + std * fill_normal(comp_env, z)).clamp_(-1.0, 1.0)
            o = comp_env.step(a)[0]

    calls = {"fill": fill_steps, "composition": comp_steps, "rollout": lambda: roll_env.rollout(K, policy=pol)}
    for fn in calls.values():
        timed(fn)
    times = {k: [] for k in calls}
    names = list(calls)
    for r in range(repeats):
        for j in range(len(names)):
            k = names[(r + j) % len(names)]
            times[k].append(timed(calls[k]))
    med = {k: statistics.median(v) for k, v in times.items()}
    for k, v in times.items():
        emit(f"step   n={n:8d} {k:12s} {med[k] * 1e3 / K:9.2f} us/step [{min(v) * 1e3 / K:9.2f} .. "
             f"{max(v) * 1e3 / K:9.2f}]  {med[k] / med['fill']:6.2f}x step(policy_actions)")
    del fill_env, comp_env, roll_env


def heldout(pol):
    held = _HeldOut()
    kw = dict(num_episodes_per_object=5000, seed=42, max_episode_steps=200)
    for name, p in (("heuristic", "heuristic"), ("mlp relu", pol)):
        dx.evaluation.evaluate_heldout_set_batched(held, policy=p, **kw)            # warm-up
        secs = []
        for _ in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = dx.evaluation.evaluate_heldout_set_batched(held, policy=p, **kw)
            torch.cuda.synchronize()
            secs.append(time.perf_counter() - t0)
        emit(f"heldout 20 x 5000 {name:9s} {statistics.median(secs):7.3f} s [{min(secs):.3f} .. {max(secs):.3f}]  "
             f"success {res['metrics']['grasp_success_rate']:.3f}  mean length {res['metrics']['mean_episode_length']:.1f}")


emit(gpu_line())
emit(f"[64, 64] policies, action_std {STD}; {repeats} repeats; median [min .. max]")
pols = {"relu": policy("relu"), "tanh": policy("tanh")}
with torch.no_grad():
    for n in (131072, 1 << 20):
        fill_kernel(n, pols)
    for n in (131072, 1 << 20):
        stepping(n, pols["relu"])
    torch.cuda.empty_cache()
    heldout(pols["relu"])
os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
with open(OUT, "w") as fh:
    fh.write("# python tools/time_policy_actions.py\n" + "\n".join(lines) + "\n")
