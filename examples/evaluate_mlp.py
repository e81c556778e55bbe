"""Evaluate a trained MLP policy with the batched evaluation front-ends.

    python examples/ppo_mlp.py --save actor.pt
    python examples/evaluate_mlp.py actor.pt

loads the actor and ``log_std`` that ``examples/ppo_mlp.py --save`` writes (without a file: a freshly initialised actor
of the same shape), then

1. runs the held-out evaluation (``evaluate_heldout_set_batched``) on the 20-object duck-typed held-out set of
   ``examples/run_baseline_configs.py``, and
2. runs a robustness sweep (``run_robustness_sweep_batched``) over observation noise x dynamics noise on one held-out
   object,

and prints the success rate, mean episode length, mean final contacts and failure-type frequencies of every cell, and
how many of a noisy cell's episodes differ from the same episode of the noise-free baseline.
The policy reads the noisy observation, so the observation-noise cells measure what the noise does to it.
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402
from ppo_mlp import mlp  # noqa: E402
from run_baseline_configs import _HeldOut  # noqa: E402


def load_policy(path=None, deterministic=False, device="cuda", seed=0):
    """The ``MlpPolicy`` of a file written by ``ppo_mlp.py --save``, or of a fresh actor when ``path`` is None."""
    torch.manual_seed(seed)
    actor = mlp(15)
    log_std = torch.full((15,), -1.0)
    if path:
        saved = torch.load(path, map_location="cpu")
        actor.load_state_dict(saved["actor"])
        log_std = saved["log_std"]
    return dx.MlpPolicy.from_torch(actor, action_std=None if deterministic else log_std.exp(), device=device)


def cell_line(name, metrics, changed=""):
    freq = {k: round(v["frequency"], 3) for k, v in metrics["failure_type_frequency"].items() if v["count"]}
    return (f"{name:28s} success {metrics['grasp_success_rate']:.3f}  mean length {metrics['mean_episode_length']:6.2f}  "
            f"mean contacts {metrics['mean_contacts']:.3f}{changed}  failures {freq}")


def changed(cell, baseline):
    """Episodes of a sweep cell that differ from the same (replica, episode) of the noise-free baseline: every cell
    uses the same seeds, so a difference is the noise's doing."""
    n = sum(a != b for a, b in zip(cell["episodes"], baseline["episodes"]))
    return f"  {n:5d}/{len(cell['episodes'])} episodes changed"


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("path", nargs="?", help="file written by examples/ppo_mlp.py --save (default: a fresh actor)")
    ap.add_argument("--episodes-per-object", type=int, default=200)
    ap.add_argument("--replicas", type=int, default=256, help="side-by-side copies of every robustness cell")
    ap.add_argument("--episodes", type=int, default=5, help="episodes per replica and robustness cell")
    ap.add_argument("--obs-noise", type=float, nargs="+", default=[0.0, 0.02, 0.05, 0.1])
    ap.add_argument("--dyn-noise", type=float, nargs="+", default=[0.0, 0.05, 0.1])
    ap.add_argument("--deterministic", action="store_true", help="act with the mean (no exploration noise)")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args(argv)
    policy = load_policy(args.path, args.deterministic, seed=args.seed)
    print(f"policy {policy.hidden} {policy.activation}, sha256 {policy.sha256()[:16]}")
    held = _HeldOut()
    res = dx.evaluation.evaluate_heldout_set_batched(held, policy=policy, num_episodes_per_object=args.episodes_per_object,
                                                     seed=42, policy_seed=args.seed)
    print(cell_line(f"held-out ({res['overall_stats']['total_episodes']} episodes)", res["metrics"]))
    sweep = dx.evaluation.run_robustness_sweep_batched(held.get_eval_config(0), args.obs_noise, args.dyn_noise,
                                                       policy=policy, num_episodes=args.episodes, seed=7,
                                                       num_replicas=args.replicas)
    base = sweep["baseline"]
    print(cell_line("baseline", base["metrics"]))
    for key in ("observation_noise", "dynamics_noise"):
        for level, cell in sweep[key].items():
            print(cell_line(f"{key} {level:g}", cell["metrics"], changed(cell, base)))
    for name, cell in sweep["combined_noise"].items():
        print(cell_line(name, cell["metrics"], changed(cell, base)))


if __name__ == "__main__":
    main()
