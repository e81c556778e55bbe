"""Cost of an observation-conditioned MLP policy inside the fused rollout against the alternatives.

    python tools/time_rollout_mlp.py [repeats]          (writes profiles/r08_rollout_mlp.txt too)

Per size (4,096, 131,072 and 1,048,576 envs), 50 env-steps per env with a [64, 64] ReLU policy (action_std 0.1):
  random:     rollout(50, policy="random") -- the fused rollout without a network, for scale;
  mlp:        rollout(50, policy=MlpPolicy) -- the network evaluated in the rollout kernel (dexsim_rollout_mlp);
  loop:       50 x (torch forward of the same nn.Sequential on step()'s observation, + std * randn, clamp, step()),
              an auto-reset env, eager;
  loop_graph: the same 50 steps captured once in a CUDA graph and replayed.
CUDA events around each call (a call = 50 steps of every env); the four take turns call by call in one process, the
order rotating every repeat; median and min..max over the repeats.  Prints the GPU's name and power limit first.
Before timing, the twin check: MlpPolicy.mean and the torch module on the same observations differ only by torch's
summation order (max |difference| printed).  Workload: hard curriculum, dense reward, 200-step episodes, tracking on.
"""
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import dexterous_rl_manipulation_b200 as dx  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
repeats = int(args[0]) if args else 9
K = 50
STD = 0.1
OUT = os.path.join(ROOT, "profiles", "r08_rollout_mlp.txt")
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


def run(n, net, pol):
    rand_env, mlp_env = make_env(n), make_env(n)
    loop_env = make_env(n, auto_reset=True, loop_max_steps=200)
    graph_env = make_env(n, auto_reset=True, loop_max_steps=200)

    # twin check: the kernel's mean against the torch module on this env's observations
    obs = mlp_env._obs[:, :n].t()
    with torch.no_grad():
        diff = (pol.mean(obs) - net(obs)).abs().max().item()
    emit(f"n={n}: max |MlpPolicy.mean - torch forward| on the reset observations = {diff:.3e}")

    def loop_steps(env):
        o = env._obs_view
        for _ in range(K):
            a = (net(o) + STD * torch.randn(n, 15, device="cuda")).clamp_(-1.0, 1.0)
            o = env.step(a)[0]

    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.no_grad(), torch.cuda.stream(side):
        loop_steps(graph_env)                       # warm-up outside the capture (cuBLAS handles, workspaces)
    torch.cuda.current_stream().wait_stream(side)
    with torch.no_grad(), torch.cuda.graph(graph):
        loop_steps(graph_env)

    calls = {
        "random": lambda: rand_env.rollout(K, policy="random"),
        "mlp": lambda: mlp_env.rollout(K, policy=pol),
        "loop": lambda: loop_steps(loop_env),
        "loop_graph": graph.replay,
    }
    with torch.no_grad():
        for fn in calls.values():                   # warm-up: module load, first touch
            timed(fn)
        times = {k: [] for k in calls}
        names = list(calls)
        for r in range(repeats):
            for j in range(len(names)):
                k = names[(r + j) % len(names)]
                times[k].append(timed(calls[k]))
    med = {k: statistics.median(v) for k, v in times.items()}
    for k, v in times.items():
        emit(f"n={n:8d} {k:10s} {med[k] * 1e3 / K:9.2f} us/step [{min(v) * 1e3 / K:9.2f} .. {max(v) * 1e3 / K:9.2f}]  "
             f"{n * K / (med[k] * 1e-3):.3e} env-steps/s  {med[k] / med['mlp']:6.2f}x the mlp rollout")
    del rand_env, mlp_env, loop_env, graph_env, graph
    torch.cuda.empty_cache()


emit(gpu_line())
emit(f"{K} steps per call, [64, 64] ReLU policy, action_std {STD}; {repeats} repeats per variant, rotating; "
     "median [min .. max] per step of all envs")
torch.manual_seed(0)
net = torch.nn.Sequential(torch.nn.Linear(45, 64), torch.nn.ReLU(), torch.nn.Linear(64, 64), torch.nn.ReLU(),
                          torch.nn.Linear(64, 15)).cuda()
pol = dx.MlpPolicy.from_torch(net, action_std=STD)
for n in (4096, 131072, 1 << 20):
    run(n, net, pol)
if "--no-write" not in sys.argv:
    with open(OUT, "w") as fh:
        fh.write("# python tools/time_rollout_mlp.py\n" + "\n".join(lines) + "\n")
