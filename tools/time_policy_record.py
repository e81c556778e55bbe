"""Cost of the behaviour-policy record and of GAE on the device, and a fixed-seed run of examples/ppo_mlp.py.

    python tools/time_policy_record.py [--repeats R] [--ppo-iters I] [--out FILE]

1. rollout(50) with a [64, 64] ReLU MlpPolicy (action_std 0.1), at 131,072 and 1,048,576 envs:
     recorded:  enable_trajectory(50, final_observation=True)                      (dexsim_rollout_mlp)
     policy:    enable_trajectory(50, final_observation=True, policy_record=True)  (dexsim_rollout_mlp_record)
   CUDA events around each call, the two alternating call by call, median [min .. max] over the repeats.
2. GAE over 1 Mi envs x 50 rows of a real recording: env.gae's kernel (dexsim_gae, called on padded arrays) against the
   torch reverse loop (the same arithmetic, element-wise ops per row).  Bytes the kernel must move: reward 4 + terminated
   1 + finished 1 + values 4 + final_values 4 (read) + advantages 4 + returns 4 (written) per env-row, plus the extra
   values row; compared with the copy peak measured in the same process (a 2 GiB device-to-device copy_, read + write).
3. examples/ppo_mlp.py at 131,072 envs, seed 0, I iterations: seconds and mean episode return per iteration.
Prints the GPU's name and power limit first.  Working sets exceed the 126 MB L2 except the per-call MLP weights.
"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402
from dexterous_rl_manipulation_b200 import _lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--repeats", type=int, default=7)
ap.add_argument("--ppo-iters", type=int, default=30)
ap.add_argument("--out", default=None)
args = ap.parse_args()
K = 50
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


def timed(fn):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end)


def alternate(calls, repeats):
    for fn in calls.values():
        timed(fn)
    times = {k: [] for k in calls}
    names = list(calls)
    for r in range(repeats):
        for j in range(len(names)):
            k = names[(r + j) % len(names)]
            times[k].append(timed(calls[k]))
    return times


def make_env(n):
    env = dx.BatchedManipulationEnv(n, "cuda", reward_type="dense", track_episodes=True, seed=42, max_episode_steps=200,
                                    curriculum_config=dx.CurriculumConfig.hard())
    env.reset(seed=42)
    return env


emit(gpu_line())
torch.manual_seed(0)
net = torch.nn.Sequential(torch.nn.Linear(45, 64), torch.nn.ReLU(), torch.nn.Linear(64, 64), torch.nn.ReLU(),
                          torch.nn.Linear(64, 15)).cuda()
pol = dx.MlpPolicy.from_torch(net, action_std=0.1)

# 1. the record's cost in the rollout
emit(f"1. rollout({K}), [64, 64] ReLU, action_std 0.1; {args.repeats} repeats, alternating; median [min .. max] per step")
for n in (131072, 1 << 20):
    rec, prec = make_env(n), make_env(n)
    rec.enable_trajectory(K, final_observation=True)
    prec.enable_trajectory(K, final_observation=True, policy_record=True)
    with torch.no_grad():
        times = alternate({"recorded": lambda: rec.rollout(K, policy=pol),
                           "policy": lambda: prec.rollout(K, policy=pol)}, args.repeats)
    med = {k: statistics.median(v) for k, v in times.items()}
    for k, v in times.items():
        emit(f"n={n:8d} {k:9s} {med[k] * 1e3 / K:8.2f} us/step [{min(v) * 1e3 / K:8.2f} .. {max(v) * 1e3 / K:8.2f}]  "
             f"{med[k] / med['recorded']:5.3f}x recorded")
    del rec, prec
    torch.cuda.empty_cache()

# 2. GAE: kernel against the torch reverse loop on the same arrays
n = 1 << 20
env = make_env(n)
env.enable_trajectory(K, final_observation=True)
env.rollout(K, policy=pol)
ld = env.ld
g = torch.Generator(device="cuda").manual_seed(1)
values = torch.randn(K + 1, ld, generator=g, device="cuda")
final_values = torch.randn(K, ld, generator=g, device="cuda")
adv, ret = torch.empty(K, ld, device="cuda"), torch.empty(K, ld, device="cuda")
tr = env._traj
traj = _lib.DexsimTrajectory(tr["obs"].data_ptr(), None, tr["reward"].data_ptr(), tr["terminated"].data_ptr(), None,
                             tr["finished"].data_ptr(), K)
L = _lib.lib()
gamma, lam = 0.99, 0.95


def kernel():
    _lib.check(L.dexsim_gae(C.byref(traj), n, ld, K, values.data_ptr(), final_values.data_ptr(), C.c_float(gamma),
                            C.c_float(lam), adv.data_ptr(), ret.data_ptr(), env._stream()), "dexsim_gae")


reward, fin, term = tr["reward"][:K], tr["finished"][:K].bool(), tr["terminated"][:K].bool()
t_adv, t_ret = torch.empty_like(adv), torch.empty_like(ret)
gl = torch.tensor(gamma, dtype=torch.float32) * torch.tensor(lam, dtype=torch.float32)


def torch_loop():
    a_next = torch.zeros(ld, device="cuda")
    for t in range(K - 1, -1, -1):
        nv = torch.where(fin[t], torch.where(term[t], 0.0, final_values[t]), values[t + 1])
        delta = (reward[t] + gamma * nv) - values[t]
        a = torch.where(fin[t], delta, delta + float(gl) * a_next)
        t_adv[t] = a
        t_ret[t] = a + values[t]
        a_next = a


src = torch.empty(1 << 29, device="cuda")            # 2 GiB
dst = torch.empty_like(src)
times = alternate({"dexsim_gae": kernel, "torch_loop": torch_loop, "copy_2GiB": lambda: dst.copy_(src)}, args.repeats)
med = {k: statistics.median(v) for k, v in times.items()}
peak = 2 * src.numel() * 4 / (med["copy_2GiB"] * 1e-3)
moved = n * K * (4 + 1 + 1 + 4 + 4 + 4 + 4) + n * 4
same = torch.equal(adv[:, :n], t_adv[:, :n]) and torch.equal(ret[:, :n], t_ret[:, :n])
emit(f"2. GAE over {n} envs x {K} rows; copy peak {peak / 1e9:.0f} GB/s (2 GiB copy_, read + write); "
     f"kernel and torch loop bit-identical: {same}")
for k in ("dexsim_gae", "torch_loop"):
    v = times[k]
    emit(f"   {k:10s} {med[k] * 1e3:9.1f} us [{min(v) * 1e3:9.1f} .. {max(v) * 1e3:9.1f}]  "
         f"{moved / (med[k] * 1e-3) / 1e9:6.0f} GB/s of the kernel's {moved / 1e6:.0f} MB = "
         f"{moved / (med[k] * 1e-3) / peak:5.2f} of the copy peak")
emit(f"   torch loop / kernel: {med['torch_loop'] / med['dexsim_gae']:.1f}x")
del env, src, dst
torch.cuda.empty_cache()

# 3. the PPO example
import ppo_mlp  # noqa: E402
emit(f"3. examples/ppo_mlp.py --envs 131072 --iters {args.ppo_iters} --seed 0 (steps 50, sigma_obs 0 / 0.02 / 0.05)")
hist = ppo_mlp.train(envs=131072, iters=args.ppo_iters, steps=50, seed=0, log=None)
secs = [h["seconds"] for h in hist[1:]]
emit(f"   {1 / statistics.median(secs):.2f} iterations/s (median over iterations 1..; iteration 0 "
     f"{hist[0]['seconds']:.2f} s); max |log ratio| before the first update {max(h['max_abs_log_ratio0'] for h in hist):.1e}")
emit("   mean episode return per iteration: " + " ".join(f"{h['mean_return']:.2f}" for h in hist))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("# python tools/time_policy_record.py\n" + "\n".join(lines) + "\n")
