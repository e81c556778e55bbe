"""PPO on the fused rollout (needs a B200).

    python examples/ppo_mlp.py --envs 131072 --iters 40 --sigma-obs 0.0 0.02 0.05

Each iteration samples with the current actor inside one rollout launch and updates it in torch:

1. ``MlpPolicy.from_torch(actor, std)`` packs the actor and its current standard deviation;
2. ``env.rollout(k, policy=mlp)`` acts with it in the kernel and, after
   ``enable_trajectory(k, final_observation=True, policy_record=True)``, records the behaviour policy's data: the
   network's input ``policy_obs`` (with the observation noise of the env's group), the unclipped action ``raw_action``
   and its ``log_prob``;
3. the critic evaluates the noise-free observations (an asymmetric critic: ``values[k]`` needs no unrecorded input) and
   the terminal observations ``final_observation``;
4. ``env.gae`` turns them into advantages and returns on the device, bootstrapping truncated episodes from the terminal
   observation and never running across an episode boundary;
5. a few epochs of the clipped surrogate objective over ``policy_obs`` / ``raw_action`` / ``log_prob``.

The actor is a tanh MLP [64, 64] with a learned state-independent log-std; the log-probabilities are those of the
unclipped Gaussian sample, the convention of PPO implementations that clip outside the distribution.
"""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402
from dexterous_rl_manipulation_b200 import _lib  # noqa: E402


def mlp(out, hidden=(64, 64)):
    layers, width = [], 45
    for h in hidden:
        layers += [torch.nn.Linear(width, h), torch.nn.Tanh()]
        width = h
    return torch.nn.Sequential(*layers, torch.nn.Linear(width, out))


def train(envs=131072, iters=40, steps=50, sigma_obs=(0.0, 0.02, 0.05), seed=0, epochs=4, minibatches=4, lr=3e-4,
          gamma=0.99, lam=0.95, clip=0.2, max_episode_steps=200, device="cuda", log=print, save=None):
    """Run PPO; returns one dict per iteration: mean episode return, surrogate / value losses of every minibatch,
    ``max_abs_log_ratio0`` (max |log pi(raw_action | policy_obs) - log_prob| over the batch before the first update:
    0 up to float32 rounding, since the torch actor and the kernel evaluate the same network) and wall-clock seconds.
    ``save``: a path to which the trained actor's ``state_dict`` and ``log_std`` are written after the last iteration
    (``torch.save``; ``examples/evaluate_mlp.py`` loads it)."""
    torch.manual_seed(seed)
    groups = [dx.CurriculumConfig.easy()] * len(sigma_obs)
    env = dx.BatchedManipulationEnv(envs, device, reward_type="dense", max_episode_steps=max_episode_steps,
                                    track_episodes=True, groups=groups, group_sigma_obs=tuple(sigma_obs), seed=seed)
    state_obs, _ = env.reset(seed=seed)            # a view of the state: the noise-free observation before each call
    env.enable_trajectory(steps, final_observation=True, policy_record=True)
    actor, critic = mlp(15).to(device), mlp(1).to(device)
    log_std = torch.nn.Parameter(torch.full((15,), -1.0, device=device))
    opt = torch.optim.Adam([*actor.parameters(), *critic.parameters(), log_std], lr=lr)
    value = lambda x: critic(x).squeeze(-1)
    history = []
    for it in range(iters):
        t0 = time.perf_counter()
        obs0 = state_obs.clone()
        policy = dx.MlpPolicy.from_torch(actor, action_std=log_std.detach().exp(), device=device)
        counters, ret_sums = env.rollout(steps, policy=policy, zero_counters=True)
        tr = env.trajectory
        with torch.no_grad():
            obs = torch.cat([obs0[None], tr["obs"]])                           # [k+1, n, 45], noise-free
            values = value(obs)
            final_values = value(tr["final_observation"])
        adv, ret = env.gae(values.contiguous(), final_values.contiguous(), gamma, lam)
        x = tr["policy_obs"].reshape(-1, 45)
        raw = tr["raw_action"].reshape(-1, 15)
        old_lp = tr["log_prob"].reshape(-1)
        v_in = obs[:-1].reshape(-1, 45)
        a = adv.reshape(-1)
        a = (a - a.mean()) / (a.std() + 1e-8)
        r = ret.reshape(-1)
        with torch.no_grad():
            lp0 = torch.distributions.Normal(actor(x), log_std.exp()).log_prob(raw).sum(-1)
            max_abs_log_ratio0 = float((lp0 - old_lp).abs().max())
        pg_losses, v_losses = [], []
        rows = x.shape[0]
        for _ in range(epochs):
            perm = torch.randperm(rows, device=device)
            for mb in perm.chunk(minibatches):
                dist = torch.distributions.Normal(actor(x[mb]), log_std.exp())
                ratio = torch.exp(dist.log_prob(raw[mb]).sum(-1) - old_lp[mb])
                pg = -torch.min(ratio * a[mb], ratio.clamp(1 - clip, 1 + clip) * a[mb]).mean()
                vl = 0.5 * (value(v_in[mb]) - r[mb]).pow(2).mean()
                opt.zero_grad(set_to_none=True)
                (pg + vl).backward()
                torch.nn.utils.clip_grad_norm_([*actor.parameters(), *critic.parameters(), log_std], 1.0)
                opt.step()
                pg_losses.append(float(pg.detach())); v_losses.append(float(vl.detach()))
        torch.cuda.synchronize(device)
        episodes = int(counters[:, _lib.CNT_EPISODES].sum())
        mean_return = float(ret_sums[:, 0].sum()) / episodes if episodes else float("nan")
        stats = dict(iter=it, episodes=episodes, mean_return=mean_return, pg_loss=pg_losses, v_loss=v_losses,
                     max_abs_log_ratio0=max_abs_log_ratio0, seconds=time.perf_counter() - t0)
        history.append(stats)
        if log:
            log(f"iter {it:3d}  episodes {episodes:8d}  mean return {mean_return:9.3f}  pg {pg_losses[-1]:+.4f}  "
                f"v {v_losses[-1]:.4f}  |log ratio0| {max_abs_log_ratio0:.1e}  {stats['seconds']:.2f} s")
    if save:
        torch.save({"actor": {k: v.cpu() for k, v in actor.state_dict().items()}, "log_std": log_std.detach().cpu()}, save)
    return history


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--steps", type=int, default=50, help="rollout steps per iteration")
    ap.add_argument("--sigma-obs", type=float, nargs="+", default=[0.0, 0.02, 0.05],
                    help="observation-noise std of each env group (env i is in group i %% len)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--save", metavar="PATH", help="write the trained actor and log_std here (torch.save)")
    args = ap.parse_args(argv)
    train(args.envs, args.iters, args.steps, tuple(args.sigma_obs), args.seed, save=args.save)


if __name__ == "__main__":
    main()
