"""Generate the golden fixtures in tests/golden/ by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference or oracle/_ref):

    python tests/golden/make_golden.py

The reference is imported under oracle/gym_stub (gymnasium is not installed in the image);
numpy 2.3.5 / NEP 50 promotion is part of the pinned behaviour (SURVEY.md Appendix A-16).
Outputs (committed):
    traj.npz     per-step obs / reward / components / flags for 30 trajectories
    noise.npz    CombinedNoiseWrapper trajectories with the wrapper's normal draws recorded
    labels.npz   both failure classifiers on synthetic episodes (ties included)
    episodes.npz Evaluator.evaluate_episode / run_episode records with the policy's actions
    learner.npz  run_episode + SimpleLearner on a reused env, with the learner's normal draws recorded
    scheduler.npz CurriculumScheduler decisions on random success streams
    anchors.json scalar anchors quoted in SURVEY.md 8c and the reference tests' known answers
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from oracle import ref_harness  # noqa: E402

R = ref_harness.load()
CC = R.CurriculumConfig
T_STEPS = 210

VARIABLE = dict(object_size=0.05, object_size_range=(0.03, 0.07), object_mass=0.1,
                object_mass_range=(0.05, 0.15), friction_coefficient=0.5, friction_range=(0.3, 0.7),
                spawn_distance=0.15, spawn_distance_range=(0.10, 0.20), spawn_x_range=(-0.1, 0.1),
                spawn_y_range=(-0.1, 0.1), spawn_z_range=(0.05, 0.2))   # experiments/config_variable.json


def configs():
    return {"default": CC(), "easy": CC.easy(), "medium": CC.medium(), "hard": CC.hard(),
            "variable": CC(**VARIABLE)}


def action_for(style, rng):
    if style == 0:
        return rng.uniform(-1.2, 1.2, 15).astype(np.float32)           # exercises the clamp
    if style == 1:
        return (np.float32(-0.5) + rng.uniform(-0.1, 0.1, 15).astype(np.float32)).astype(np.float32)
    if style == 2:
        return np.full(15, -0.5, np.float32)
    return rng.normal(0, 0.6, 15).astype(np.float32)


def gen_traj():
    out = {k: [] for k in ("jp0", "size", "mass", "friction", "pos", "keep_pos", "chain", "dense", "max_steps",
                            "weights", "actions", "obs", "reward", "comps", "terminated", "truncated",
                            "num_contacts", "op_final")}
    names = []
    case = 0
    for cname, cfg in configs().items():
        for rtype in ("dense", "sparse"):
            for seed in range(3):
                style = case % 4
                max_steps = 50 if case % 5 == 0 else 200
                weights = (2.0, 0.25, 0.7, 0.1) if (case % 7 == 3 and rtype == "dense") else (1.0, 0.5, 0.3, 0.2)
                shaping = R.rewards.RewardShaping(*weights) if rtype == "dense" else None
                env = R.DexterousManipulationEnv(reward_type=rtype, curriculum_config=cfg,
                                                 max_episode_steps=max_steps, reward_shaping=shaping)
                rng = np.random.default_rng(7000 + case)
                n_eps = 2 if seed == 0 else 1        # 2nd episode: reused env keeps the object position
                for ep in range(n_eps):
                    obs0, _ = env.reset(seed=100 * case + seed + ep)
                    out["jp0"].append(env.joint_positions.copy())
                    out["size"].append(env.object_size); out["mass"].append(env.object_mass)
                    out["friction"].append(env.friction_coefficient)
                    out["pos"].append(env.object_position.astype(np.float32).copy())
                    out["keep_pos"].append(ep > 0); out["chain"].append(len(names) - 1 if ep > 0 else -1)
                    out["dense"].append(rtype == "dense"); out["max_steps"].append(max_steps)
                    out["weights"].append(weights)
                    acts, obs, rew, comps, te, tr, nc = [], [obs0], [], [], [], [], []
                    for _ in range(T_STEPS):
                        a = action_for(style, rng)
                        o, r, term, trunc, info = env.step(a)
                        acts.append(a); obs.append(o); rew.append(r)
                        rc = info["reward_components"]
                        comps.append([rc["distance"], rc["contact"], rc["closure"], rc["stability"]])
                        te.append(term); tr.append(trunc); nc.append(info["num_contacts"])
                    out["actions"].append(acts); out["obs"].append(obs); out["reward"].append(rew)
                    out["comps"].append(comps); out["terminated"].append(te); out["truncated"].append(tr)
                    out["num_contacts"].append(nc); out["op_final"].append(np.asarray(env.object_position, np.float64))
                    names.append(f"{cname}/{rtype}/seed{seed}/ep{ep}/style{style}")
                case += 1
    arr = dict(
        jp0=np.asarray(out["jp0"], np.float32), size=np.asarray(out["size"], np.float64),
        mass=np.asarray(out["mass"], np.float64), friction=np.asarray(out["friction"], np.float64),
        pos=np.asarray(out["pos"], np.float32), keep_pos=np.asarray(out["keep_pos"], bool),
        chain=np.asarray(out["chain"], np.int32), dense=np.asarray(out["dense"], bool),
        max_steps=np.asarray(out["max_steps"], np.int32), weights=np.asarray(out["weights"], np.float64),
        actions=np.asarray(out["actions"], np.float32), obs=np.asarray(out["obs"], np.float32),
        reward=np.asarray(out["reward"], np.float64), comps=np.asarray(out["comps"], np.float64),
        terminated=np.asarray(out["terminated"], bool), truncated=np.asarray(out["truncated"], bool),
        num_contacts=np.asarray(out["num_contacts"], np.uint8), op_final=np.asarray(out["op_final"], np.float64),
        names=np.asarray(names))
    # The seed-2 trajectories are left out to keep the file under 1 MB.  The other 30 still cover every configuration,
    # both reward types, all four action styles, both episode limits and every reused-env (chained) episode.
    keep = np.array([i for i, name in enumerate(names) if "/seed2/" not in name])
    remap = {int(old): new for new, old in enumerate(keep)}
    arr = {k: v[keep] for k, v in arr.items()}
    arr["chain"] = np.asarray([remap[int(c)] if c >= 0 else -1 for c in arr["chain"]], np.int32)
    np.savez_compressed(os.path.join(HERE, "traj.npz"), **arr)
    print("traj.npz:", len(keep), "trajectories x", T_STEPS, "steps;",
          "terminated steps:", int(arr["terminated"].sum()), "truncated steps:", int(arr["truncated"].sum()))


def gen_noise():
    """evaluation/robustness_tests.py:140-211.  The wrapper owns default_rng(seed); its draws are
    reset -> 45 obs normals, each step -> 15 action normals then 45 obs normals (only for sigma > 0).
    A twin generator with the same seed replays them so they can be stored as pre-drawn tensors."""
    T = 80
    recs = {k: [] for k in ("jp0", "size", "mass", "friction", "pos", "sigma_obs", "sigma_dyn", "actions",
                            "dyn_noise", "obs_noise", "obs", "reward", "terminated", "truncated", "num_contacts")}
    cells = [(0.05, 0.0), (0.0, 0.05), (0.01, 0.1), (0.1, 0.01), (0.2, 0.2), (0.0, 0.0)]
    for k, (so, sd) in enumerate(cells):
        cfg = [CC.hard(), CC.medium(), CC(**VARIABLE)][k % 3]
        base = R.DexterousManipulationEnv(curriculum_config=cfg, reward_type="dense", max_episode_steps=60)
        env = R.robustness_tests.CombinedNoiseWrapper(base, observation_noise_std=so, dynamics_noise_std=sd, seed=50 + k)
        twin = np.random.default_rng(50 + k)
        prng = np.random.default_rng(900 + k)
        obs0, _ = env.reset(seed=11 + k)
        on = [twin.normal(0, so, 45).astype(np.float32) if so > 0 else np.zeros(45, np.float32)]
        recs["jp0"].append(base.joint_positions.copy()); recs["size"].append(base.object_size)
        recs["mass"].append(base.object_mass); recs["friction"].append(base.friction_coefficient)
        recs["pos"].append(base.object_position.astype(np.float32).copy())
        recs["sigma_obs"].append(so); recs["sigma_dyn"].append(sd)
        acts, dn, obs, rew, te, tr, nc = [], [], [obs0], [], [], [], []
        for _ in range(T):
            a = (np.float32(-0.5) + prng.uniform(-0.6, 0.6, 15).astype(np.float32)).astype(np.float32)
            dn.append(twin.normal(0, sd, 15).astype(np.float32) if sd > 0 else np.zeros(15, np.float32))
            o, r, term, trunc, info = env.step(a)
            on.append(twin.normal(0, so, 45).astype(np.float32) if so > 0 else np.zeros(45, np.float32))
            acts.append(a); obs.append(o); rew.append(r); te.append(term); tr.append(trunc); nc.append(info["num_contacts"])
        recs["actions"].append(acts); recs["dyn_noise"].append(dn); recs["obs_noise"].append(on)
        recs["obs"].append(obs); recs["reward"].append(rew); recs["terminated"].append(te)
        recs["truncated"].append(tr); recs["num_contacts"].append(nc)
    np.savez_compressed(
        os.path.join(HERE, "noise.npz"),
        jp0=np.asarray(recs["jp0"], np.float32), size=np.asarray(recs["size"]), mass=np.asarray(recs["mass"]),
        friction=np.asarray(recs["friction"]), pos=np.asarray(recs["pos"], np.float32),
        sigma_obs=np.asarray(recs["sigma_obs"]), sigma_dyn=np.asarray(recs["sigma_dyn"]),
        actions=np.asarray(recs["actions"], np.float32), dyn_noise=np.asarray(recs["dyn_noise"], np.float32),
        obs_noise=np.asarray(recs["obs_noise"], np.float32), obs=np.asarray(recs["obs"], np.float32),
        reward=np.asarray(recs["reward"], np.float64), terminated=np.asarray(recs["terminated"], bool),
        truncated=np.asarray(recs["truncated"], bool), num_contacts=np.asarray(recs["num_contacts"], np.uint8),
        max_steps=np.int32(60))
    print("noise.npz:", len(cells), "cells x", T, "steps")


def count_rows(counts):
    return [[1.0 if i < c else 0.0 for i in range(5)] for c in counts]   # evaluator.py:148-150


def gen_labels():
    M = R.metrics.EvaluationMetrics(3)
    Tx = R.failure_taxonomy.FailureClassifier(3)
    ma = {ft.value: i for i, ft in enumerate(R.metrics.FailureType)}
    mb = {fm.value: i for i, fm in enumerate(R.failure_taxonomy.FailureMode)}
    rng = np.random.default_rng(2024)
    N, LMAX = 4000, 210
    counts = np.zeros((N, LMAX), np.uint8); length = np.zeros(N, np.int32)
    steps = np.zeros(N, np.int32); num = np.zeros(N, np.int32); final = np.zeros(N, np.int32)
    succ = np.zeros(N, bool); la = np.zeros(N, np.int8); lb = np.zeros(N, np.int8); conf = np.zeros(N)
    var = np.full(N, np.nan)
    lens = [0, 1, 2, 4, 5, 6, 7, 8, 9, 10, 11, 12, 15, 16, 17, 31, 64, 100, 127, 128, 129, 136, 150, 199, 200, 201, 210]
    for i in range(N):
        L = int(rng.choice(lens))
        mode = i % 6
        if mode == 0: c = rng.integers(0, 6, L)
        elif mode == 1: c = rng.integers(0, 3, L)
        elif mode == 2: c = np.sort(rng.integers(0, 6, L))[::-1]
        elif mode == 3: c = rng.choice([0, 4], L)
        elif mode == 4: c = rng.choice([0, 2], L)
        else: c = np.concatenate([rng.integers(2, 5, L // 2), rng.integers(0, 2, L - L // 2)])
        c = np.asarray(c, np.int64)
        counts[i, :L] = c; length[i] = L
        steps[i] = int(rng.choice([L, L, L, 200, 50]))
        final[i] = int(c[-1]) if (L and i % 3) else int(rng.integers(0, 4))
        num[i] = final[i] if i % 2 else int(rng.integers(0, 4))
        succ[i] = (i % 13 == 0)
        ep = {"success": bool(succ[i]), "episode_steps": int(steps[i]), "num_contacts": int(num[i]),
              "final_contacts": int(final[i]), "contact_history": count_rows(c)}
        ra = M.classify_failure(ep, 200)
        rb, cf = Tx.classify(ep, 200)
        la[i] = -1 if ra is None else ma[ra.value]
        lb[i] = -1 if rb is None else mb[rb.value]
        conf[i] = list(cf.values())[0] if cf else 0.0
        if L > 1:
            var[i] = float(np.var([int(x) for x in c]))
    np.savez_compressed(os.path.join(HERE, "labels.npz"), counts=counts, length=length, steps=steps, num=num,
                        final=final, success=succ, label_metrics=la, label_taxonomy=lb, confidence=conf, var=var,
                        max_steps=np.int32(200))
    print("labels.npz:", N, "episodes; label histogram (metrics):", np.bincount(la + 1, minlength=7).tolist(),
          "(taxonomy):", np.bincount(lb + 1, minlength=7).tolist())


class RecordingPolicy:
    def __init__(self, inner):
        self.inner = inner
        self.actions = []

    def select_action(self, obs):
        a = self.inner.select_action(obs)
        self.actions.append(np.asarray(a, np.float32).copy())
        return a

    def reset(self):
        self.inner.reset()


def gen_episodes():
    """Whole-episode records through the reference's own callers: Evaluator.evaluate_episode
    (evaluation/evaluator.py:71-189, fresh env per episode, success = terminated) and run_episode
    (training/episode_utils.py:13-55, reused env, success always False)."""
    M = R.metrics.EvaluationMetrics(3)
    Tx = R.failure_taxonomy.FailureClassifier(3)
    ma = {ft.value: i for i, ft in enumerate(R.metrics.FailureType)}
    mb = {fm.value: i for i, fm in enumerate(R.failure_taxonomy.FailureMode)}
    TMAX = 200
    recs = {k: [] for k in ("kind", "jp0", "size", "mass", "friction", "pos", "keep_pos", "actions", "n_steps",
                            "success", "episode_reward", "final_contacts", "label_metrics", "label_taxonomy",
                            "max_steps", "loop_max_steps", "dense")}

    def pad(acts):
        a = np.zeros((TMAX, 15), np.float32)
        a[:len(acts)] = np.asarray(acts, np.float32)
        return a

    # Evaluator flow
    np.random.seed(0)
    train = CC(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))
    held_big = R.heldout_objects.HeldOutObjectSet(train_config=train, num_heldout_objects=6, seed=123)
    held_small = R.heldout_objects.HeldOutObjectSet(train_config=train, eval_size_range=(0.02, 0.035),
                                                    num_heldout_objects=6, seed=7)   # mostly TIMEOUT failures
    for obj_idx in range(6):
        held = held_big if obj_idx < 3 else held_small
        for ep_i in range(3):
            for (max_steps, rtype) in ((200, "dense"), (40, "sparse")):
                env_probe = R.DexterousManipulationEnv(curriculum_config=held.get_eval_config(obj_idx))
                pol = RecordingPolicy(R.policies.HeuristicPolicy(env_probe.action_space))
                ev = R.evaluator.Evaluator(pol, held, reward_type=rtype, max_episode_steps=max_steps)
                cfg = held.get_eval_config(obj_idx)
                seed = 42 + ep_i
                res = ev.evaluate_episode(cfg, seed=seed)
                probe = R.DexterousManipulationEnv(curriculum_config=cfg); probe.reset(seed=seed)
                recs["kind"].append(0); recs["jp0"].append(probe.joint_positions.copy())
                recs["size"].append(probe.object_size); recs["mass"].append(probe.object_mass)
                recs["friction"].append(probe.friction_coefficient)
                recs["pos"].append(probe.object_position.astype(np.float32).copy()); recs["keep_pos"].append(False)
                recs["actions"].append(pad(pol.actions)); recs["n_steps"].append(res["episode_steps"])
                recs["success"].append(res["success"]); recs["episode_reward"].append(res["episode_reward"])
                recs["final_contacts"].append(res["final_contacts"])
                ra = M.classify_failure(res, max_steps); rb, _ = Tx.classify(res, max_steps)
                recs["label_metrics"].append(-1 if ra is None else ma[ra.value])
                recs["label_taxonomy"].append(-1 if rb is None else mb[rb.value])
                recs["max_steps"].append(max_steps); recs["loop_max_steps"].append(max_steps)
                recs["dense"].append(rtype == "dense")
    # run_episode flow on a reused env (2nd+ episodes keep the object position), shorter loop bound
    np.random.seed(1)
    for cname, cfg in (("easy", CC.easy()), ("hard", CC.hard()), ("variable", CC(**VARIABLE))):
        env = R.DexterousManipulationEnv(curriculum_config=cfg, reward_type="dense", max_episode_steps=200)
        pol = RecordingPolicy(R.policies.HeuristicPolicy(env.action_space))
        for ep_i in range(3):
            pol.actions = []
            # run_episode calls env.reset() without a seed: seed the env's generator explicitly first
            env._np_random = np.random.Generator(np.random.PCG64(np.random.SeedSequence(500 + ep_i)))
            prev_pos = None if env.object_position is None else np.asarray(env.object_position, np.float64).copy()
            success, steps, total = R.episode_utils.run_episode(env, pol, max_steps=120)
            # recover the reset draws with a twin env driven by the same generator state
            twin = R.DexterousManipulationEnv(curriculum_config=cfg, reward_type="dense", max_episode_steps=200)
            twin._np_random = np.random.Generator(np.random.PCG64(np.random.SeedSequence(500 + ep_i)))
            if prev_pos is not None:
                twin.object_position = prev_pos
            twin.reset()
            recs["kind"].append(1); recs["jp0"].append(twin.joint_positions.copy())
            recs["size"].append(twin.object_size); recs["mass"].append(twin.object_mass)
            recs["friction"].append(twin.friction_coefficient)
            recs["pos"].append(twin.object_position.astype(np.float32).copy()); recs["keep_pos"].append(ep_i > 0)
            recs["actions"].append(pad(pol.actions)); recs["n_steps"].append(steps)
            recs["success"].append(success); recs["episode_reward"].append(total)
            recs["final_contacts"].append(int(np.sum(env.contacts > 0.5)))
            recs["label_metrics"].append(-2); recs["label_taxonomy"].append(-2)   # not produced by this caller
            recs["max_steps"].append(200); recs["loop_max_steps"].append(120); recs["dense"].append(True)
    np.savez_compressed(
        os.path.join(HERE, "episodes.npz"),
        kind=np.asarray(recs["kind"], np.int32), jp0=np.asarray(recs["jp0"], np.float32),
        size=np.asarray(recs["size"]), mass=np.asarray(recs["mass"]), friction=np.asarray(recs["friction"]),
        pos=np.asarray(recs["pos"], np.float32), keep_pos=np.asarray(recs["keep_pos"], bool),
        actions=np.asarray(recs["actions"], np.float32), n_steps=np.asarray(recs["n_steps"], np.int32),
        success=np.asarray(recs["success"], bool), episode_reward=np.asarray(recs["episode_reward"], np.float64),
        final_contacts=np.asarray(recs["final_contacts"], np.int32),
        label_metrics=np.asarray(recs["label_metrics"], np.int32), label_taxonomy=np.asarray(recs["label_taxonomy"], np.int32),
        max_steps=np.asarray(recs["max_steps"], np.int32), loop_max_steps=np.asarray(recs["loop_max_steps"], np.int32),
        dense=np.asarray(recs["dense"], bool))
    print("episodes.npz:", len(recs["kind"]), "episodes; successes:", int(np.sum(recs["success"])),
          "lengths:", sorted(set(recs["n_steps"]))[:12])


def gen_anchors():
    a = -0.5 * np.ones(15, np.float32)
    anchors = {"numpy": np.__version__, "reference_form": ref_harness.kind()}
    env = R.DexterousManipulationEnv()
    obs, info = env.reset(seed=0)
    anchors["reset_seed0_obs0_3"] = [float(x) for x in obs[:3]]
    anchors["reset_seed0_object_position"] = [float(x) for x in info["object_position"]]
    env = R.DexterousManipulationEnv(reward_type="dense"); env.reset(seed=0)
    ret = 0.0; rs = []
    for t in range(200):
        obs, r, te, tr, info = env.step(a); ret += r; rs.append(r)
        if t == 0:
            anchors["default_dense_z1"] = float(info["object_position"][2])
    anchors["default_dense_r1"] = rs[0]; anchors["default_dense_r2"] = rs[1]
    anchors["default_dense_return200"] = ret; anchors["default_dense_jp0_after200"] = float(obs[0])
    env = R.DexterousManipulationEnv(reward_type="dense", curriculum_config=CC.easy()); env.reset(seed=0)
    ret = 0.0
    for t in range(200):
        obs, r, te, tr, info = env.step(a); ret += r
        if te:
            anchors["easy_dense_term_step"] = t + 1; anchors["easy_dense_term_nc"] = info["num_contacts"]
            anchors["easy_dense_r_term"] = r; anchors["easy_dense_return"] = ret
            break
    env = R.DexterousManipulationEnv(reward_type="sparse", curriculum_config=CC.hard()); env.reset(seed=0)
    ret = 0.0
    for t in range(200):
        obs, r, te, tr, info = env.step(a); ret += r
    anchors["hard_sparse_return200"] = ret
    env = R.DexterousManipulationEnv(max_episode_steps=5); env.reset(seed=0)
    anchors["truncated_flags_max5"] = [bool(env.step(a)[3]) for _ in range(8)]
    # asserted known answers of the reference's own tests
    # (episode dicts restated as data: per-step contact counts + the label the test asserts)
    anchors["known_answers"] = [
        {"src": "tests/test_failure_taxonomy.py:60-73", "episode_steps": 200, "num_contacts": 2, "final_contacts": 2,
         "counts": [], "taxonomy": ["timeout"]},
        {"src": "tests/test_failure_taxonomy.py:87-106", "episode_steps": 50, "num_contacts": 1, "final_contacts": 1,
         "counts": [max(0, 4 - i // 5) for i in range(20)], "taxonomy": ["slippage"]},
        {"src": "tests/test_failure_taxonomy.py:153-176", "episode_steps": 50, "num_contacts": 2, "final_contacts": 2,
         "counts": [2] * 20, "taxonomy": ["misalignment"]},
        {"src": "tests/test_failure_taxonomy.py:189-212", "episode_steps": 50, "num_contacts": 0, "final_contacts": 0,
         "counts": [3] * 5 + [0] * 5, "taxonomy": ["object_dropped"]},
        {"src": "tests/test_evaluation_metrics.py:68-78", "episode_steps": 200, "num_contacts": 2, "final_contacts": 2,
         "counts": [], "metrics": ["timeout"]},
        {"src": "tests/test_evaluation_metrics.py:80-90", "episode_steps": 100, "num_contacts": 1, "final_contacts": 1,
         "counts": [], "metrics": ["insufficient_contacts", "misaligned_grasp"]},
        {"src": "tests/test_evaluation_metrics.py:93-103", "episode_steps": 50, "num_contacts": 2, "final_contacts": 0,
         "counts": [], "metrics": ["object_dropped"]},
    ]
    with open(os.path.join(HERE, "anchors.json"), "w") as fh:
        json.dump(anchors, fh, indent=1)
    print("anchors.json written")


def gen_scheduler():
    """experiments/curriculum_scheduler.py:141-222,77-139: progression decisions and interpolated
    configs for random success streams (the batched driver must reproduce them)."""
    rng = np.random.default_rng(99)
    recs = {k: [] for k in ("kw", "success", "steps", "progressed", "level", "size", "mass", "friction")}
    for trial in range(12):
        kw = [float(rng.choice([0.3, 0.5, 0.7])), int(rng.choice([5, 20, 50])), int(rng.choice([5, 15, 20])),
              int(rng.choice([3, 5, 7]))]
        sch = R.CurriculumScheduler(CC.easy(), CC.hard(), success_rate_threshold=kw[0],
                                    min_episodes_before_progression=kw[1], window_size=kw[2], progression_steps=kw[3])
        p = rng.uniform(0.2, 0.9)
        succ = rng.random(300) < p
        steps = rng.integers(1, 200, 300)
        prog, lvl, sz, ms, fr = [], [], [], [], []
        for a, b in zip(succ, steps):
            prog.append(sch.update(bool(a), int(b)))
            c = sch.get_current_config()
            lvl.append(sch.current_difficulty_level); sz.append(c.object_size); ms.append(c.object_mass)
            fr.append(c.friction_coefficient)
        recs["kw"].append(kw); recs["success"].append(succ); recs["steps"].append(steps); recs["progressed"].append(prog)
        recs["level"].append(lvl); recs["size"].append(sz); recs["mass"].append(ms); recs["friction"].append(fr)
    np.savez_compressed(os.path.join(HERE, "scheduler.npz"), **{k: np.asarray(v) for k, v in recs.items()})
    print("scheduler.npz: 12 streams x 300 episodes; progressions:", int(np.sum(recs["progressed"])))


def gen_learner():
    """run_episode (training/episode_utils.py:13-55) with SimpleLearner (policies/simple_learner.py) on ONE reused
    env object, 4 consecutive episodes per case; the learner's np.random.normal draws are recorded so that they
    can be replayed as pre-drawn tensors (select_action: sigma 0.3 -> float32; update: sigma lr, float64)."""
    K, EPS = 60, 4
    rec = {k: [] for k in ("dense", "jp0", "size", "mass", "friction", "pos", "act_noise", "upd_noise", "steps",
                           "reward", "final_mean", "final_contacts")}
    orig = np.random.normal
    for cname in ("easy", "medium", "hard"):
        cfg = getattr(CC, cname)()
        for rtype in ("dense", "sparse"):
            env = R.DexterousManipulationEnv(curriculum_config=cfg, reward_type=rtype, max_episode_steps=200)
            pol = R.policies.SimpleLearner(env.action_space, learning_rate=0.01)
            draws = []

            def recorder(loc, scale, size=None):
                x = orig(loc, scale, size=size)
                draws.append((scale, np.array(x)))
                return x

            np.random.normal = recorder
            np.random.seed(5)
            jp0, pos, act, upd, steps, rew, fc = [], [], [], [], [], [], []
            try:
                for ep in range(EPS):
                    env._np_random = np.random.Generator(np.random.PCG64(np.random.SeedSequence(11 + ep)))
                    twin = R.DexterousManipulationEnv(curriculum_config=cfg)
                    twin._np_random = np.random.Generator(np.random.PCG64(np.random.SeedSequence(11 + ep)))
                    twin.reset()
                    jp0.append(twin.joint_positions.copy()); pos.append(twin.object_position.astype(np.float32))
                    before = len(draws)
                    _, n_steps, total = R.episode_utils.run_episode(env, pol, max_steps=K)
                    a = np.zeros((K, 15), np.float32); u = np.zeros((K, 15), np.float64); t = -1
                    for scale, x in draws[before:]:
                        if scale == 0.3:
                            t += 1; a[t] = x.astype(np.float32)
                        else:
                            u[t] = x
                    act.append(a); upd.append(u); steps.append(n_steps); rew.append(total)
                    fc.append(int(np.sum(env.contacts > 0.5)))
            finally:
                np.random.normal = orig
            rec["dense"].append(rtype == "dense"); rec["jp0"].append(jp0); rec["pos"].append(pos)
            rec["size"].append(cfg.object_size); rec["mass"].append(cfg.object_mass); rec["friction"].append(cfg.friction_coefficient)
            rec["act_noise"].append(act); rec["upd_noise"].append(upd); rec["steps"].append(steps); rec["reward"].append(rew)
            rec["final_mean"].append(pol.mean_action.copy()); rec["final_contacts"].append(fc)
    np.savez_compressed(os.path.join(HERE, "learner.npz"), loop_max_steps=np.int32(K),
                        **{k: np.asarray(v) for k, v in rec.items()})
    print("learner.npz:", len(rec["dense"]), "cases x", EPS, "episodes; steps:", rec["steps"])


if __name__ == "__main__":
    gen_learner()
    gen_scheduler()
    gen_traj()
    gen_noise()
    gen_labels()
    gen_episodes()
    gen_anchors()
