"""Batched front-ends for the reference's evaluation drivers (SURVEY.md 8f rank 1).

They launch fused rollouts (policy generated in-kernel, episodes logged on the device) and re-emit
the reference's result-dict schemas, so ``EvaluationMetrics.compute_aggregate_metrics``,
``format_metrics_report``, ``SeedVarianceAnalyzer.compute_variance_statistics`` and the robustness
analysis run unchanged on the output:

  evaluate_heldout_set_batched  -> Evaluator.evaluate_heldout_set       (evaluation/evaluator.py:191-271)
  evaluate_with_noise_batched   -> RobustnessTester.evaluate_with_noise (evaluation/robustness_tests.py:240-328)
  run_robustness_sweep_batched  -> RobustnessTester.run_robustness_sweep (:330-407)
  evaluate_seeds_batched        -> SeedVarianceAnalyzer.evaluate_with_seeds (evaluation/seed_variance.py:44-78)

Wherever a policy name is taken, an ``MlpPolicy`` is accepted too: it acts inside the same one-episode fused launch
(``rollout(policy=mlp)``), reads the (possibly noisy) observation, and its episodes are replayed step by step through
``env.policy_actions``.  Each rank of a multi-GPU run passes its own ``MlpPolicy`` on its own device.

Reset draws follow the reference exactly (``rng="numpy"``: env (object o, episode e) is seeded with
``seed + e`` like evaluator.py:222, so all objects share the same initial joint / spawn draws); the
policy randomness is Philox, because the reference's policies draw from process-global NumPy state
that has no batched equivalent (SURVEY.md Appendix A-11).
"""
from typing import Tuple, Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .env import BatchedManipulationEnv
from .policy import MlpPolicy

FAILURE_TYPES = _lib.LABELS_METRICS


def count_rows(counts) -> List[List[float]]:
    """Count-encoded contact rows exactly as evaluation/evaluator.py:148-150 builds them."""
    return [[1.0 if i < int(c) else 0.0 for i in range(5)] for c in counts]


def aggregate_metrics(episodes: Sequence[Dict], max_steps: int = 200) -> Dict:
    """Same keys and values as EvaluationMetrics.compute_aggregate_metrics (evaluation/metrics.py:126-203);
    labels come from the device (``failure_type`` key) instead of being re-derived on the host."""
    if not episodes:
        return {}
    n = len(episodes)
    succ = [bool(e["success"]) for e in episodes]
    lens = [int(e["episode_steps"]) for e in episodes]
    contacts = [int(e["num_contacts"]) for e in episodes]
    labels = [e.get("failure_type") for e in episodes]
    freq = {name: {"count": labels.count(name), "frequency": float(labels.count(name) / n)} for name in FAILURE_TYPES}
    s_len = [l for l, s in zip(lens, succ) if s]
    f_len = [l for l, s in zip(lens, succ) if not s]
    s_con = [c for c, s in zip(contacts, succ) if s]
    f_con = [c for c, s in zip(contacts, succ) if not s]
    mean = lambda xs: float(np.mean(xs)) if xs else None
    return {
        "grasp_success_rate": float(np.mean(succ)),
        "mean_episode_length": float(np.mean(lens)),
        "std_episode_length": float(np.std(lens)),
        "failure_type_frequency": freq,
        "total_episodes": n,
        "successful_episodes": len(s_len),
        "failed_episodes": len(f_len),
        "mean_contacts": float(np.mean(contacts)),
        "mean_success_length": mean(s_len),
        "mean_success_contacts": mean(s_con),
        "mean_failure_length": mean(f_len),
        "mean_failure_contacts": mean(f_con),
    }


def _check_policy(policy, device):
    """Refuse, before anything is launched, an ``MlpPolicy`` on another device than ``device``."""
    if isinstance(policy, MlpPolicy):
        dev = torch.device(device)
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if policy.device != dev:
            raise ValueError(f"the policy lives on {policy.device}, the env on {dev}")


def _replay_policy(policy) -> Dict:
    """The policy entries of an episode's ``replay`` record: the name, or "mlp" and the network's hash."""
    if isinstance(policy, MlpPolicy):
        return {"policy": "mlp", "policy_sha256": policy.sha256()}
    return {"policy": policy}


def _label(code, table):
    return None if int(code) == _lib.LABEL_NONE else table[int(code)]


def _episode_dict(rec, counts, size, mass, friction, max_steps=200, success_threshold=3):
    la, lb = int(rec["label_metrics"]), int(rec["label_taxonomy"])
    if int(rec["var_tie"]) == 1 and counts is not None:
        # the device met an exact variance tie without the history at hand: decide it here with np.var's own arithmetic
        # (evaluation/metrics.py:77-80, evaluation/failure_taxonomy.py:189,219-230)
        la, lb = _lib.classify_counts(bool(rec["success"]), int(rec["steps"]), int(rec["final_contacts"]),
                                      int(rec["final_contacts"]), counts, max_steps=max_steps,
                                      success_threshold=success_threshold)
    d = {
        "episode_reward": float(rec["episode_reward"]),
        "episode_steps": int(rec["steps"]),
        "success": bool(rec["success"]),
        "num_contacts": int(rec["final_contacts"]),
        "final_contacts": int(rec["final_contacts"]),
        "contact_history": count_rows(counts) if counts is not None else [],
        "object_size": float(size),
        "object_mass": float(mass),
        "friction_coefficient": float(friction),
        "failure_type": _label(la, _lib.LABELS_METRICS),
        "failure_mode": _label(lb, _lib.LABELS_TAXONOMY),
    }
    return d


def _heldout_shard(heldout_set, policy, n_eps, seeds, reward_type, max_episode_steps, device, policy_seed,
                   contact_history, actions, lo, hi):
    """Envs [lo, hi) of the (object, episode) batch -> {global env index: (record, per-step counts)}.
    Reset seeds, groups and Philox keys depend on the GLOBAL env index only, so any partition of the batch
    (one shard per GPU) produces the records of the unpartitioned run."""
    objs = heldout_set.heldout_objects
    n_obj = len(objs)
    cfgs = [heldout_set.get_eval_config(k) for k in range(n_obj)]
    m = hi - lo
    pad = max(m, 2) - m
    group_of_env = np.concatenate([np.arange(lo, hi) // n_eps, np.zeros(pad, np.int64)])
    env = BatchedManipulationEnv(m + pad, device, max_episode_steps=max_episode_steps, reward_type=reward_type,
                                 track_episodes=True, rng="numpy", groups=cfgs, seed=policy_seed, env_gid0=lo,
                                 group_of_env=group_of_env)
    env_seeds = [seeds[i % n_eps] for i in range(lo, hi)] + [0] * pad
    env.reset(seed=env_seeds)
    kw = {}
    if policy == "external":
        a = torch.as_tensor(actions, dtype=torch.float32).reshape(max_episode_steps, -1, 15)[:, lo:hi]
        if pad:
            a = torch.cat([a, torch.zeros(max_episode_steps, pad, 15)], 1)
        kw["actions"] = a
    # exactly the caller loop bound: at most max_episode_steps steps per episode (evaluator.py:135)
    recs = _run_one_episode_each(env, max_episode_steps, policy, True, max_episode_steps, contact_history, kw)
    return {lo + i: (recs[i][0].copy(), None if recs[i][1] is None else recs[i][1].copy()) for i in range(m)}


def evaluate_heldout_set_batched(heldout_set, policy: str = "heuristic", num_episodes_per_object: int = 5,
                                 seed: Optional[int] = None, reward_type: str = "dense", max_episode_steps: int = 200,
                                 device="cuda", policy_seed: int = 0, contact_history: bool = True,
                                 actions=None, shard: Optional[Tuple[int, int]] = None) -> Dict:
    """All (object, episode) pairs of Evaluator.evaluate_heldout_set as ONE batch.

    ``policy``: "heuristic" | "random" (fused, Philox), an ``MlpPolicy`` on ``device`` (fused, the network acting on
    every env's observation, its exploration keyed by ``policy_seed``), or "external" with ``actions`` of shape
    [max_episode_steps, n_objects * n_episodes, 15] (env index = object * n_episodes + episode).  Every episode's
    ``replay`` entry holds what ``replay_episode`` needs; for an MLP it records ``"policy": "mlp"`` and the network's
    ``policy_sha256``.

    Multi-GPU: with ``torch.distributed`` initialised (or an explicit ``shard=(rank, world_size)``) every rank
    runs a contiguous slice of the batch on its own GPU and the per-episode records are all-gathered, so every
    rank returns the complete result -- identical to the single-GPU one.  Pass a ``seed`` in that case (an
    unseeded run draws different episode seeds on every rank)."""
    import torch.distributed as dist
    from .distributed import shard_range
    _check_policy(policy, device)
    objs = heldout_set.heldout_objects
    n_obj, n_eps = len(objs), int(num_episodes_per_object)
    n = n_obj * n_eps
    if seed is None:
        seeds = [int(s) for s in np.random.default_rng(None).integers(0, 2 ** 31, n_eps)]   # evaluator.py:222
    else:
        seeds = [int(seed) + e for e in range(n_eps)]
    distributed = shard is None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    rank, world = shard if shard is not None else ((dist.get_rank(), dist.get_world_size()) if distributed else (0, 1))
    lo, hi = shard_range(n, rank, world)
    recs = _heldout_shard(heldout_set, policy, n_eps, seeds, reward_type, max_episode_steps, device, policy_seed,
                          contact_history, actions, lo, hi)
    if distributed:
        parts = [None] * world
        dist.all_gather_object(parts, recs)
        recs = {k: v for part in parts for k, v in part.items()}
    elif shard is not None and world > 1:
        return {"shard_records": recs, "range": (lo, hi)}          # caller merges (tests, custom launchers)
    return _heldout_result(heldout_set, recs, n_eps, seeds, policy, policy_seed, reward_type, max_episode_steps)


def _heldout_result(heldout_set, recs, n_eps, seeds, policy, policy_seed, reward_type, max_episode_steps) -> Dict:
    """Result dictionary of Evaluator.evaluate_heldout_set (evaluation/evaluator.py:191-271) from episode records."""
    objs = heldout_set.heldout_objects
    n_obj = len(objs)
    env_seeds = [seeds[i % n_eps] for i in range(n_obj * n_eps)]
    replay_policy = _replay_policy(policy)
    size, mass, fric = ([o.size for o in objs], [o.mass for o in objs], [o.friction for o in objs])
    all_results, object_results = [], {}
    for o in range(n_obj):
        obj_results = []
        for e in range(n_eps):
            rec, counts = recs[o * n_eps + e]
            d = _episode_dict(rec, counts, size[o], mass[o], fric[o], max_episode_steps)
            d["object_idx"], d["episode"] = o, e
            # everything needed to re-run exactly this episode with full capture (replay_episode)
            d["replay"] = {"object_idx": o, "reset_seed": env_seeds[o * n_eps + e], "env_gid": int(rec["env_gid"]),
                           "philox_episode": int(rec["episode"]), **replay_policy, "policy_seed": int(policy_seed),
                           "reward_type": reward_type, "max_episode_steps": int(max_episode_steps)}
            obj_results.append(d)
            all_results.append(d)
        object_results[o] = {
            "object_properties": {"size": size[o], "mass": mass[o], "friction": fric[o]},
            "episodes": obj_results,
            "mean_reward": float(np.mean([r["episode_reward"] for r in obj_results])),
            "mean_steps": float(np.mean([r["episode_steps"] for r in obj_results])),
            "success_rate": float(np.mean([1.0 if r["success"] else 0.0 for r in obj_results])),
        }
    metrics = aggregate_metrics(all_results, max_episode_steps)
    per_object_metrics = {o: aggregate_metrics(v["episodes"], max_episode_steps) for o, v in object_results.items()}
    overall = {
        "num_objects": n_obj,
        "total_episodes": len(all_results),
        "overall_success_rate": metrics["grasp_success_rate"],
        "mean_reward": float(np.mean([r["episode_reward"] for r in all_results])),
        "std_reward": float(np.std([r["episode_reward"] for r in all_results])),
        "mean_steps": metrics["mean_episode_length"],
    }
    return {"overall_stats": overall, "per_object_results": object_results, "all_episodes": all_results,
            "metrics": metrics, "per_object_metrics": per_object_metrics}


def _run_one_episode_each(env, k_steps, policy, respawn, loop_max_steps, with_history, kw):
    """One fused launch in one-episode mode; {env index: (record, per-step contact counts)}."""
    n = env.num_envs
    env.enable_episode_log(capacity=n)
    if with_history:
        env.enable_history(k_steps)
    env._rollout_steps = 0
    env.rollout(k_steps, policy=policy, respawn=respawn, loop_max_steps=loop_max_steps, one_episode=True, **kw)
    log = env.read_episode_log()
    idx = log["env_gid"].astype(np.int64) - env.env_gid0
    hist = env._hist[:, :n].cpu().numpy() if with_history else None
    out = {}
    for r, i in zip(log, idx):
        counts = hist[:int(r["steps"]), i] if hist is not None else None
        out[int(i)] = (r, counts)
    if len(out) != n:
        raise RuntimeError(f"{n - len(out)} envs did not finish an episode within {k_steps} steps")
    return out


def evaluate_with_noise_batched(eval_config, policy: str = "heuristic", observation_noise_std: float = 0.0,
                                dynamics_noise_std: float = 0.0, num_episodes: int = 20, seed: Optional[int] = None,
                                reward_type: str = "dense", max_episode_steps: int = 200, device="cuda",
                                num_replicas: int = 1, policy_seed: int = 0,
                                shard: Optional[Tuple[int, int]] = None) -> Dict:
    """RobustnessTester.evaluate_with_noise: ONE env object reused for ``num_episodes`` episodes -- the
    object is respawned only for the first one and stays where the previous episode left it afterwards
    (evaluation/robustness_tests.py:260,282; envs/manipulation_env.py:156-161); every episode is one
    fused launch in one-episode mode followed by the reference's own reset(seed + episode).  ``num_replicas``
    independent copies of that experiment run side by side (replica r is seeded with seed + 1000 r).
    Dynamics noise is drawn in-kernel.  Observation noise reaches an ``MlpPolicy``, which acts on the noisy
    observation; the shipped in-kernel policies ("heuristic", "random") ignore observations (SURVEY.md 3.5), so
    for them it cannot change the trajectory and is only recorded in the output.
    With ``torch.distributed`` initialised (or ``shard=(rank, world_size)``) the replicas are spread over the ranks
    and the records all-gathered; every rank returns the complete, GPU-count-independent result."""
    import torch.distributed as dist
    from .distributed import shard_range
    _check_policy(policy, device)
    distributed = shard is None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    rank, world = shard if shard is not None else ((dist.get_rank(), dist.get_world_size()) if distributed else (0, 1))
    if world > 1 and seed is None:
        raise ValueError("pass a seed when the replicas are spread over several ranks")
    lo, hi = shard_range(int(num_replicas), rank, world)          # this rank's replicas; Philox keys use the global index
    m = hi - lo
    n = max(m, 2)
    base = int(np.random.default_rng(None).integers(0, 2 ** 31)) if seed is None else int(seed)
    env = BatchedManipulationEnv(n, device, max_episode_steps=max_episode_steps, reward_type=reward_type,
                                 track_episodes=True, rng="numpy", groups=[eval_config],
                                 group_sigma_obs=observation_noise_std, group_sigma_dyn=dynamics_noise_std,
                                 seed=policy_seed if seed is None else base, env_gid0=lo)
    local = {lo + r: [] for r in range(m)}
    for ep in range(int(num_episodes)):
        # robustness_tests.py:281-282: reset(seed = seed + episode) on the SAME env object -- the first
        # reset samples the spawn, later ones keep the position the previous episode ended at
        env.reset(seed=[base + 1000 * (lo + r) + ep for r in range(n)])
        env._episode.fill_(ep)                       # distinct Philox policy / noise streams per episode
        recs = _run_one_episode_each(env, max_episode_steps, policy, False, max_episode_steps, True, {})
        for r in range(m):
            rec, counts = recs[r]
            d = _episode_dict(rec, counts, eval_config.object_size, eval_config.object_mass, eval_config.friction_coefficient,
                                  max_episode_steps)
            local[lo + r].append({k: d[k] for k in ("success", "episode_steps", "num_contacts", "final_contacts",
                                                    "contact_history", "episode_reward", "failure_type", "failure_mode")})
    if distributed:
        parts = [None] * world
        dist.all_gather_object(parts, local)
        local = {k: v for part in parts for k, v in part.items()}
    elif shard is not None and world > 1:
        return {"shard_replicas": local, "range": (lo, hi)}          # caller merges (tests, custom launchers)
    replicas = [local[r] for r in range(int(num_replicas))]
    episodes = [e for eps in replicas for e in eps]
    return {"episodes": episodes, "metrics": aggregate_metrics(episodes, max_episode_steps),
            "noise_levels": {"observation_noise_std": observation_noise_std, "dynamics_noise_std": dynamics_noise_std},
            "replicas": replicas}


def run_robustness_sweep_batched(eval_config, observation_noise_levels, dynamics_noise_levels, policy="heuristic",
                                 num_episodes=20, seed=None, **kw) -> Dict:
    """Same cells and result layout as RobustnessTester.run_robustness_sweep (:330-407)."""
    run = lambda so, sd: evaluate_with_noise_batched(eval_config, policy, so, sd, num_episodes, seed, **kw)
    results = {"baseline": run(0.0, 0.0)}
    results["observation_noise"] = {so: run(so, 0.0) for so in observation_noise_levels if so > 0.0}
    results["dynamics_noise"] = {sd: run(0.0, sd) for sd in dynamics_noise_levels if sd > 0.0}
    combined = {}
    for so in list(observation_noise_levels)[:3]:
        for sd in list(dynamics_noise_levels)[:3]:
            if so > 0.0 or sd > 0.0:
                combined[f"obs_{so:.3f}_dyn_{sd:.3f}"] = run(so, sd)
    results["combined_noise"] = combined
    return results


def evaluate_seeds_batched(heldout_set, seeds: Sequence[int], policy="heuristic", num_episodes_per_object=5,
                           reward_type="dense", max_episode_steps=200, device="cuda") -> Dict[int, Dict]:
    """SeedVarianceAnalyzer.evaluate_with_seeds: {seed: evaluate_heldout_set result}; feed it to the
    reference's compute_variance_statistics unchanged (evaluation/seed_variance.py:80-196)."""
    return {int(s): evaluate_heldout_set_batched(heldout_set, policy, num_episodes_per_object, int(s), reward_type,
                                                 max_episode_steps, device, policy_seed=int(s))
            for s in seeds}


def replay_episode(eval_config, reset_seed: int, env_gid: int, philox_episode: int = 0, policy="heuristic",
                   policy_seed: int = 0, reward_type: str = "dense", max_episode_steps: int = 200, device="cuda",
                   dynamics_noise_std: float = 0.0) -> Dict:
    """Re-run ONE episode of a fused rollout step by step with full capture.  Trajectories are a pure
    function of (reset draws, Philox key, global env id, episode index), so any episode a rollout logged can
    be reproduced bit for bit later -- this is how failed episodes get the ``states`` / ``actions`` /
    ``contact_history`` that FailureLogger.log_episode stores (evaluation/failure_logger.py:48-119), without
    the rollout kernel having to write trajectories for a million envs.  ``policy``: "heuristic", "random" or the
    ``MlpPolicy`` that ran the episode; every action comes from ``env.policy_actions``.
    Returns {"states": [T+1 x obs[45]], "actions": [T x a[15]], "contacts": [T+1 count-encoded rows],
    "episode": per-episode dict} in the layout evaluation/evaluator.py:118-173 records."""
    _check_policy(policy, device)
    env = BatchedManipulationEnv(2, device, max_episode_steps=max_episode_steps, reward_type=reward_type, rng="numpy",
                                 groups=[eval_config], seed=policy_seed, env_gid0=int(env_gid),
                                 dynamics_noise_std=dynamics_noise_std, reward_components=False)
    obs, info = env.reset(seed=[int(reset_seed), int(reset_seed)])
    env._episode.fill_(int(philox_episode))
    states = [obs[0].cpu().numpy().copy()]
    n0 = int(info["num_contacts"][0])
    contacts = [[1.0 if i < n0 else 0.0 for i in range(5)]]
    actions, total, steps, success = [], 0.0, 0, False
    for _ in range(int(max_episode_steps)):
        a = env.policy_actions(policy)
        obs, rew, te, tr, info = env.step(a)
        actions.append(a[0].cpu().numpy().copy())
        states.append(obs[0].cpu().numpy().copy())
        nc = int(info["num_contacts"][0])
        contacts.append([1.0 if i < nc else 0.0 for i in range(5)])
        total += float(rew[0])
        steps += 1
        if bool(te[0]) or bool(tr[0]):
            success = bool(te[0])
            break
    episode = {"episode_reward": total, "episode_steps": steps, "success": success, "num_contacts": nc,
               "final_contacts": nc, "contact_history": contacts[1:], "object_size": float(eval_config.object_size),
               "object_mass": float(eval_config.object_mass), "friction_coefficient": float(eval_config.friction_coefficient)}
    return {"states": states, "actions": actions, "contacts": contacts, "episode": episode}


def log_failures_batched(result: Dict, heldout_set, failure_logger, device="cuda", policy=None) -> int:
    """Feed every failed episode of an ``evaluate_heldout_set_batched`` result to an (unchanged)
    FailureLogger, re-creating its full trajectory by deterministic replay; returns the number logged.
    Mirrors the logging branch of Evaluator.evaluate_episode (evaluation/evaluator.py:97-185).
    Episodes of an ``MlpPolicy`` are replayed with ``policy``, which must be that network: when the result holds failed
    such episodes and ``policy`` is missing or its ``sha256()`` differs from the recorded one, ValueError is raised before
    anything is launched."""
    mlp_hashes = {ep["replay"]["policy_sha256"] for ep in result["all_episodes"]
                  if not ep["success"] and "replay" in ep and ep["replay"]["policy"] == "mlp"}
    if mlp_hashes:
        if not isinstance(policy, MlpPolicy):
            raise ValueError("the result holds failed MlpPolicy episodes: pass the policy that ran them (policy=...)")
        _check_policy(policy, device)
        if mlp_hashes != {policy.sha256()}:
            raise ValueError("the policy given is not the network that ran the result's episodes (policy_sha256 differs)")
    logged = 0
    for ep in result["all_episodes"]:
        if ep["success"] or "replay" not in ep or ep["replay"]["policy"] not in ("random", "heuristic", "mlp"):
            continue
        rp = ep["replay"]
        cfg = heldout_set.get_eval_config(rp["object_idx"])
        tr = replay_episode(cfg, rp["reset_seed"], rp["env_gid"], rp["philox_episode"],
                            policy if rp["policy"] == "mlp" else rp["policy"], rp["policy_seed"],
                            rp["reward_type"], rp["max_episode_steps"], device)
        if tr["episode"]["episode_steps"] != ep["episode_steps"] or tr["episode"]["final_contacts"] != ep["final_contacts"]:
            raise RuntimeError("replay diverged from the logged episode")
        metadata = {"seed": rp["reset_seed"], "object_size": ep["object_size"], "object_mass": ep["object_mass"],
                    "friction_coefficient": ep["friction_coefficient"], "env_gid": rp["env_gid"],
                    "philox_seed": rp["policy_seed"], "eval_config": cfg.to_dict() if hasattr(cfg, "to_dict") else {}}
        data = {k: v for k, v in ep.items() if k != "replay"}
        failure_logger.log_episode(episode_data=data, states=tr["states"], actions=tr["actions"], contacts=tr["contacts"],
                                   metadata=metadata, max_steps=rp["max_episode_steps"])
        logged += 1
    return logged
