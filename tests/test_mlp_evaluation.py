"""Evaluating and replaying MLP policies: ``dexsim_fill_mlp_actions``, ``env.policy_actions`` and the evaluation
front-ends with an ``MlpPolicy``.

The action fill is checked against the fused rollout: an env stepped with ``step(policy_actions(mlp))`` must reproduce
a recorded ``rollout(policy=mlp)`` of the same batch bit for bit, every step, and equal the three-launch composition
clip(mlp.mean(observation) + std * fill_normal(stream 4)).  The front-ends are checked against a one-episode recorded
rollout of the same batch (an independent path to the states and actions a replay rebuilds), against their own shards,
and, where the reference is present, against the unmodified ``Evaluator``."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib
from dexterous_rl_manipulation_b200 import evaluation as ev

STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
         "_ep_return", "_ep_stats")
T = 15                               # episode length of the action-fill comparisons
K = 40                               # steps per comparison: two full episodes and part of a third
STD = tuple(0.05 + 0.02 * j for j in range(15))
G = 3


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


def _net(hidden, act, seed, closing=False):
    """A random nn.Sequential; ``closing``: the output layer's bias at -0.5 and its weights scaled down, so that the
    policy grasps about as the heuristic does (episodes both succeed and fail) while still reading the observation."""
    torch.manual_seed(seed)
    A = torch.nn.ReLU if act == "relu" else torch.nn.Tanh
    sizes = (45,) + tuple(hidden)
    layers = []
    for i, o in zip(sizes[:-1], sizes[1:]):
        layers += [torch.nn.Linear(i, o), A()]
    net = torch.nn.Sequential(*layers, torch.nn.Linear(sizes[-1], 15))
    if closing:
        with torch.no_grad():
            net[-1].bias.fill_(-0.5)
            net[-1].weight.mul_(0.1)
    return net


def _groups():
    CC = dx.CurriculumConfig
    return [CC(object_size=s, object_size_range=(0.7 * s, 1.3 * s), object_mass=m, object_mass_range=(0.5 * m, 1.5 * m),
               friction_coefficient=f, friction_range=(0.6 * f, min(1.0, 1.4 * f)))
            for s, m, f in ((0.08, 0.05, 0.8), (0.05, 0.1, 0.5), (0.03, 0.2, 0.3))]


def _map(kind, n, seed):
    """(group_of_env or None, env_gid0): an explicit random map, or the default map across the 2^32 wrap."""
    if kind == "random":
        return np.random.default_rng(seed).integers(0, G, n), 0
    return None, 2 ** 32 - n // 2


def _group_of_env(env, goe):
    if goe is not None:
        return torch.as_tensor(goe, dtype=torch.int64, device=env.device)
    gid = torch.arange(env.num_envs, dtype=torch.int64, device=env.device) + env.env_gid0
    return (gid & 0xFFFFFFFF) % G


def _sigma_of_env(env, goe, so):
    s = torch.tensor(np.broadcast_to(np.asarray(so, np.float32), (G,)).copy(), device=env.device)
    return s[_group_of_env(env, goe)]


def _fill_normal(env, stream, rows):
    out = torch.zeros(rows, env.ld, dtype=torch.float32, device=env.device)
    _lib.check(env._lib.dexsim_fill_normal(C.byref(env._state), C.byref(env._params), stream, rows, C.c_float(1.0),
                                           out.data_ptr(), env._stream()), "dexsim_fill_normal")
    return out[:, :env.num_envs].t()


def _policy_input(env, sigma_env):
    """The observation step() returns for the env's current state: obs + sigma * z (stream 3) where sigma > 0."""
    obs = env._obs[:, :env.num_envs].t()
    if not bool((sigma_env > 0).any()):
        return obs
    z = _fill_normal(env, _lib.RNG_STREAM_OBS, 45)
    return torch.where(sigma_env[:, None] > 0, obs + sigma_env[:, None] * z, obs)


def _composition(env, pol, x):
    """The three-launch action: clip(mlp.mean(x) + std * fill_normal(stream 4, 15 rows), -1, 1)."""
    mean = pol.mean(x)
    if pol.action_std is not None:
        mean = mean + pol.action_std[:15] * _fill_normal(env, 4, 15)
    return mean.clamp(-1.0, 1.0)


def _pair(n, reward, so, sd, kind, seed):
    goe, gid0 = _map(kind, n, seed)
    common = dict(max_episode_steps=T, reward_type=reward, track_episodes=True, seed=seed, respawn=True,
                  groups=_groups(), group_sigma_obs=so, group_sigma_dyn=sd, env_gid0=gid0, group_of_env=goe)
    rec = dx.BatchedManipulationEnv(n, "cuda", **common)
    stepped = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, loop_max_steps=T, **common)
    rec.reset(seed=seed)
    stepped.reset(seed=seed)
    return rec, stepped, goe


# (n, reward, policy: (activation, hidden) or a name, action_std, per-group sigma_obs, per-group sigma_dyn, group map)
FILL_CASES = [
    (100, "dense", ("relu", (64, 64)), STD, (0.0, 0.05, 0.0), (0.0, 0.0, 0.1), "random"),
    (4173, "sparse", ("tanh", (45,)), None, (0.02, 0.0, 0.0), (0.0, 0.1, 0.0), "wrap"),
    (4173, "dense", ("tanh", (7, 64)), 0.1, 0.0, 0.0, "random"),
    (70_001, "dense", ("relu", (32,)), STD, (0.05, 0.05, 0.05), (0.05, 0.0, 0.0), "wrap"),
    (70_001, "sparse", ("relu", (64, 7)), None, (0.0, 0.03, 0.0), 0.0, "random"),
    (4173, "dense", "heuristic", None, (0.0, 0.05, 0.0), (0.0, 0.0, 0.1), "wrap"),
    (100, "sparse", "random", None, 0.0, (0.05, 0.0, 0.0), "random"),
]


# ---- GPU: the action fill against the fused rollout ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,reward,spec,std,so,sd,kind", FILL_CASES)
def test_step_with_policy_actions_equals_rollout(gpu, n, reward, spec, std, so, sd, kind):
    seed = n % 97 + 3
    rec, stepped, goe = _pair(n, reward, so, sd, kind, seed)
    mlp = isinstance(spec, tuple)
    pol = dx.MlpPolicy.from_torch(_net(spec[1], spec[0], seed), action_std=std) if mlp else spec
    sigma_env = _sigma_of_env(stepped, goe, so)
    noisy = sigma_env > 0
    rec.enable_trajectory(K, final_observation=True)
    rec.enable_episode_log(4 * n)
    rec.rollout(K, policy=pol)
    tr = rec.trajectory
    ends, ret = [], torch.zeros(n, dtype=torch.float64, device="cuda")
    gid = (torch.arange(n, dtype=torch.int64, device="cuda") + stepped.env_gid0) & 0xFFFFFFFF
    for t in range(K):
        a = stepped.policy_actions(pol)
        assert a.shape == (n, 15) and a.dtype == torch.float32 and a.is_contiguous()
        assert torch.equal(a, tr["action"][t]), (t, "action vs rollout")
        if mlp:
            assert torch.equal(a, _composition(stepped, pol, _policy_input(stepped, sigma_env))), (t, "composition")
        episode, sc = stepped._episode[:n].clone(), stepped._step_count[:n].clone()
        obs, rew, term, trunc, info = stepped.step(a)
        assert torch.equal(obs[noisy], _policy_input(stepped, sigma_env)[noisy]), (t, "noisy observation")
        assert torch.equal(tr["obs"][t], stepped._obs[:, :n].t()), (t, "obs")
        fin = info["finished"]
        for name, want in (("reward", rew), ("terminated", term), ("truncated", trunc), ("finished", fin)):
            assert torch.equal(tr[name][t], want), (t, name)
        sel = fin & ~noisy                   # step_final returns the NOISY terminal observation where noise is on
        assert torch.equal(tr["final_observation"][t][sel], info["final_observation"][sel]), (t, "final")
        ret += rew.to(torch.float64)
        for i in torch.nonzero(fin).flatten().tolist():
            ends.append((int(gid[i]), int(episode[i]), int(sc[i]) + 1, bool(term[i]), t, float(ret[i])))
        ret[fin] = 0.0
    for k in STATE:
        assert torch.equal(getattr(rec, k)[..., :n], getattr(stepped, k)[..., :n]), k
    assert torch.equal(rec.counters, stepped.counters)
    torch.testing.assert_close(rec.ret_sums, stepped.ret_sums, rtol=1e-9, atol=0.0)
    # the rollout's episode log against the episodes step() ended (its reward: the float32 step rewards summed)
    log = np.sort(rec.read_episode_log(), order=["env_gid", "episode"])
    ends.sort()
    assert len(log) == len(ends) > 0
    got = [(int(r["env_gid"]), int(r["episode"]), int(r["steps"]), bool(r["success"]), int(r["t_end"])) for r in log]
    assert got == [e[:5] for e in ends]
    np.testing.assert_allclose(log["episode_reward"], [e[5] for e in ends], rtol=1e-5, atol=1e-6)
    if mlp:
        assert 0.05 < float((tr["action"].abs() < 1).float().mean())       # not saturated everywhere


@pytest.mark.gpu
def test_next_step_mode_policy_actions_equal_composition(gpu):
    n = 4173
    goe, _ = _map("random", n, 5)
    so = (0.0, 0.04, 0.02)
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=T, reward_type="dense", track_episodes=True, seed=5,
                                    groups=_groups(), group_sigma_obs=so, group_sigma_dyn=(0.05, 0.0, 0.0),
                                    group_of_env=goe, auto_reset=True, loop_max_steps=T, autoreset_mode="next_step")
    env.reset(seed=5)
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 6), action_std=STD)
    sigma_env = _sigma_of_env(env, goe, so)
    pending = 0
    for t in range(K):
        a = env.policy_actions(pol)
        assert torch.equal(a, _composition(env, pol, _policy_input(env, sigma_env))), t
        _, _, _, _, info = env.step(a)
        pending += int(info["finished"].sum())
    assert pending > 0


@pytest.mark.gpu
@pytest.mark.parametrize("n", [33, 4173])
def test_fill_reads_only_the_state_and_writes_only_its_columns(gpu, n):
    """At the C ABI, with ld > n: the action buffer between guard bands; the guards, columns n .. ld-1, every state
    array, the counters and the return sums are left as they were."""
    goe, _ = _map("random", n, 7)
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=T, reward_type="dense", track_episodes=True, seed=7,
                                    groups=_groups(), group_sigma_obs=(0.05, 0.0, 0.02), group_of_env=goe)
    env.reset(seed=7)
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "tanh", 8), action_std=STD)
    for _ in range(3):
        env.step(env.policy_actions(pol))
    ld, guard = env.ld, 4096
    assert ld > n
    nbytes = 15 * ld * 4
    big = torch.full((nbytes + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
    inner = big[guard:guard + nbytes].view(torch.float32).view(15, ld)
    pattern = inner.clone()
    before = {k: getattr(env, k).clone() for k in STATE}
    counters, ret_sums = env.counters.clone(), env.ret_sums.clone()
    env._sync_groups()
    rc = env._lib.dexsim_fill_mlp_actions(C.byref(env._state), C.byref(env._params), env._ptr(env._groups_dev),
                                          env._ptr(env._goe), C.byref(pol._struct), inner.data_ptr(), env._stream())
    torch.cuda.synchronize()
    assert rc == 0
    assert bool((big[:guard] == 0xA5).all()) and bool((big[-guard:] == 0xA5).all())
    assert torch.equal(inner[:, n:], pattern[:, n:])
    for k in STATE:
        assert torch.equal(getattr(env, k), before[k]), k
    assert torch.equal(env.counters, counters) and torch.equal(env.ret_sums, ret_sums)
    assert torch.equal(inner[:, :n].t(), env.policy_actions(pol))


# ---- GPU: the evaluation front-ends ------------------------------------------------------------------------------------
class _Obj:
    def __init__(self, s, m, f):
        self.size, self.mass, self.friction = s, m, f


class _Held:                                   # duck type of evaluation/heldout_objects.py:39-143
    heldout_objects = [_Obj(0.03, 0.2, 0.1), _Obj(0.05, 0.2, 0.2), _Obj(0.09, 0.2, 0.25)]

    def get_eval_config(self, k):
        o = self.heldout_objects[k]
        return dx.CurriculumConfig(object_size=o.size, object_mass=o.mass, friction_coefficient=o.friction)


class _RecordingLogger:
    """Duck type of evaluation/failure_logger.py::FailureLogger: records every log_episode call."""

    def __init__(self):
        self.calls = []

    def log_episode(self, **kw):
        self.calls.append(kw)


HELD_T, HELD_EPS, HELD_SEED, POLICY_SEED = 60, 4, 42, 9


def _recorded_batch(held, pol, n_eps, seed, T_, policy_seed):
    """The held-out batch as evaluate_heldout_set_batched builds it, run as one recorded one-episode rollout:
    (observation after reset [n, 45], trajectory)."""
    n_obj = len(held.heldout_objects)
    n = n_obj * n_eps
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=T_, reward_type="dense", track_episodes=True,
                                    rng="numpy", groups=[held.get_eval_config(k) for k in range(n_obj)],
                                    seed=policy_seed, group_of_env=np.arange(n) // n_eps)
    obs0, _ = env.reset(seed=[seed + i % n_eps for i in range(n)])
    obs0 = obs0.clone()
    env.enable_trajectory(T_)
    env.rollout(T_, policy=pol, respawn=True, loop_max_steps=T_, one_episode=True)
    return obs0, {k: v.clone() for k, v in env.trajectory.items()}


def _assert_replay_equals_rows(tr, obs0, rows, i, steps):
    assert len(tr["states"]) == steps + 1 and len(tr["actions"]) == steps
    assert np.array_equal(tr["states"][0], obs0[i].cpu().numpy())
    for t in range(steps):
        assert np.array_equal(tr["states"][t + 1], rows["obs"][t][i].cpu().numpy()), (i, t, "state")
        assert np.array_equal(tr["actions"][t], rows["action"][t][i].cpu().numpy()), (i, t, "action")


@pytest.mark.gpu
@pytest.mark.parametrize("std", [0.3, None], ids=["stochastic", "deterministic"])
def test_heldout_evaluation_replays_and_shards(gpu, std):
    held = _Held()
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 12, closing=True), action_std=std)
    res = ev.evaluate_heldout_set_batched(held, policy=pol, num_episodes_per_object=HELD_EPS, seed=HELD_SEED,
                                          reward_type="dense", max_episode_steps=HELD_T, policy_seed=POLICY_SEED)
    eps = res["all_episodes"]
    assert len(eps) == 3 * HELD_EPS
    assert any(not e["success"] for e in eps)
    obs0, rows = _recorded_batch(held, pol, HELD_EPS, HELD_SEED, HELD_T, POLICY_SEED)
    for i, ep in enumerate(eps):
        rp = ep["replay"]
        assert rp["policy"] == "mlp" and rp["policy_sha256"] == pol.sha256() and rp["policy_seed"] == POLICY_SEED
        tr = ev.replay_episode(held.get_eval_config(rp["object_idx"]), rp["reset_seed"], rp["env_gid"],
                               rp["philox_episode"], pol, rp["policy_seed"], rp["reward_type"], rp["max_episode_steps"])
        assert tr["episode"]["episode_steps"] == ep["episode_steps"] and tr["episode"]["success"] == ep["success"]
        assert tr["episode"]["final_contacts"] == ep["final_contacts"]
        assert tr["episode"]["contact_history"] == ep["contact_history"]
        assert tr["episode"]["episode_reward"] == pytest.approx(ep["episode_reward"], rel=1e-5)
        _assert_replay_equals_rows(tr, obs0, rows, i, ep["episode_steps"])
    merged = {}
    for r in range(3):
        part = ev.evaluate_heldout_set_batched(held, policy=pol, num_episodes_per_object=HELD_EPS, seed=HELD_SEED,
                                               reward_type="dense", max_episode_steps=HELD_T, policy_seed=POLICY_SEED,
                                               shard=(r, 3))
        merged.update(part["shard_records"])
    again = ev._heldout_result(held, merged, HELD_EPS, [HELD_SEED + e for e in range(HELD_EPS)], pol, POLICY_SEED,
                               "dense", HELD_T)
    assert again["all_episodes"] == eps and again["metrics"] == res["metrics"]


@pytest.mark.gpu
def test_robustness_observation_noise_reaches_the_mlp(gpu):
    cfg = _Held().get_eval_config(1)
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 13, closing=True))      # deterministic: only the input differs
    kw = dict(num_episodes=3, seed=7, max_episode_steps=50, num_replicas=48)
    for policy, differs in ((pol, True), ("heuristic", False)):
        clean = ev.evaluate_with_noise_batched(cfg, policy, 0.0, 0.0, **kw)
        noisy = ev.evaluate_with_noise_batched(cfg, policy, 0.05, 0.0, **kw)
        assert len(clean["episodes"]) == len(noisy["episodes"]) == 3 * 48
        assert (clean["episodes"] != noisy["episodes"]) == differs, policy
    whole = ev.evaluate_with_noise_batched(cfg, pol, 0.05, 0.05, **kw)
    merged = {}
    for r in range(3):
        merged.update(ev.evaluate_with_noise_batched(cfg, pol, 0.05, 0.05, shard=(r, 3), **kw)["shard_replicas"])
    assert [merged[r] for r in range(48)] == whole["replicas"]
    sweep = ev.run_robustness_sweep_batched(cfg, [0.0, 0.05], [0.0, 0.05], policy=pol, num_episodes=2, seed=7,
                                            max_episode_steps=40, num_replicas=8)
    assert set(sweep) == {"baseline", "observation_noise", "dynamics_noise", "combined_noise"}
    assert list(sweep["observation_noise"]) == [0.05] and list(sweep["dynamics_noise"]) == [0.05]
    assert set(sweep["combined_noise"]) == {"obs_0.000_dyn_0.050", "obs_0.050_dyn_0.000", "obs_0.050_dyn_0.050"}
    cells = [sweep["baseline"], *sweep["observation_noise"].values(), *sweep["dynamics_noise"].values(),
             *sweep["combined_noise"].values()]
    for cell in cells:
        assert set(cell) == {"episodes", "metrics", "noise_levels", "replicas"} and len(cell["episodes"]) == 16
        assert set(cell["metrics"]["failure_type_frequency"]) == set(ev.FAILURE_TYPES)


@pytest.mark.gpu
def test_seed_variance_returns_one_result_per_seed(gpu):
    held = _Held()
    pol = dx.MlpPolicy.from_torch(_net((32,), "tanh", 14, closing=True), action_std=0.2)
    res = ev.evaluate_seeds_batched(held, [1, 2, 3], policy=pol, num_episodes_per_object=2, max_episode_steps=40)
    assert sorted(res) == [1, 2, 3]
    for s, r in res.items():
        assert r["overall_stats"]["total_episodes"] == 6 and len(r["all_episodes"]) == 6
        assert set(r["metrics"]) >= {"grasp_success_rate", "failure_type_frequency"}
        assert all(e["replay"]["policy_seed"] == s and e["replay"]["policy"] == "mlp" for e in r["all_episodes"])
    assert res[1]["all_episodes"] != res[2]["all_episodes"]       # the seed reaches the reset draws and the policy


@pytest.mark.gpu
def test_failure_logging_replays_the_mlp(gpu, monkeypatch):
    held = _Held()
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 15, closing=True), action_std=0.3)
    res = ev.evaluate_heldout_set_batched(held, policy=pol, num_episodes_per_object=HELD_EPS, seed=HELD_SEED,
                                          max_episode_steps=HELD_T, policy_seed=POLICY_SEED)
    failed = [(i, e) for i, e in enumerate(res["all_episodes"]) if not e["success"]]
    assert failed
    obs0, rows = _recorded_batch(held, pol, HELD_EPS, HELD_SEED, HELD_T, POLICY_SEED)
    log = _RecordingLogger()
    assert ev.log_failures_batched(res, held, log, policy=pol) == len(failed) == len(log.calls)
    for call, (i, ep) in zip(log.calls, failed):
        assert call["episode_data"]["episode_steps"] == ep["episode_steps"] and "replay" not in call["episode_data"]
        assert call["metadata"]["seed"] == ep["replay"]["reset_seed"]
        assert call["metadata"]["philox_seed"] == POLICY_SEED
        _assert_replay_equals_rows({"states": call["states"], "actions": call["actions"]}, obs0, rows, i,
                                   ep["episode_steps"])
    # a missing policy or another network of the same architecture is refused before anything is replayed
    other = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 16, closing=True), action_std=0.3)

    def no_replay(*a, **k):
        raise AssertionError("replayed before the policy was checked")

    monkeypatch.setattr(ev, "replay_episode", no_replay)
    for bad in (None, other, "heuristic"):
        log = _RecordingLogger()
        with pytest.raises(ValueError):
            ev.log_failures_batched(res, held, log, policy=bad)
        assert log.calls == []


# ---- reference parity (where the reference is present) ------------------------------------------------------------------
REF_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mlp_reference.c")
REF_CFLAGS = ["-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fexcess-precision=standard", "-msse2",
              "-mfpmath=sse"]


class _ReferenceMlpPolicy:
    """A deterministic ReLU MLP for the reference's Evaluator: select_action = clip(mlp_reference_mean(obs), -1, 1) with
    tests/mlp_reference.c, the C restatement of the kernel's arithmetic."""

    def __init__(self, params, hidden):
        cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
        if cc is None:
            pytest.skip("needs a C compiler for the reference")
        so = os.path.join(tempfile.mkdtemp(prefix="mlp_reference_"), "mlp_reference.so")
        subprocess.run([cc] + REF_CFLAGS + ["-shared", "-o", so, REF_SRC, "-lm"], check=True)
        self.lib = C.CDLL(so)
        self.lib.mlp_reference_mean.restype = None
        self.params = np.ascontiguousarray(params, dtype=np.float32)
        self.hidden = (C.c_int32 * 2)(*[int(h) for h in (list(hidden) + [0])[:2]])
        self.nh = len(hidden)

    def reset(self):
        pass

    def select_action(self, obs):
        x = np.ascontiguousarray(np.asarray(obs, dtype=np.float32).reshape(1, 45))
        out = np.empty((1, 15), np.float32)
        self.lib.mlp_reference_mean(self.params.ctypes.data_as(C.c_void_p), C.c_int32(self.nh), self.hidden,
                                    C.c_int32(0), x.ctypes.data_as(C.c_void_p), C.c_int64(1),
                                    out.ctypes.data_as(C.c_void_p))
        return np.clip(out[0], -1.0, 1.0).astype(np.float32)


@pytest.mark.gpu
def test_heldout_front_end_matches_reference_evaluator(gpu, tmp_path):
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("reference (source or byte-compiled) not present")
    import importlib
    R = ref_harness.load()
    T_, n_eps = 60, 3
    train = R.CurriculumConfig(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))
    held = R.heldout_objects.HeldOutObjectSet(train_config=train, eval_size_range=(0.025, 0.09), num_heldout_objects=6,
                                              seed=5)
    net = _net((64, 64), "relu", 17, closing=True)
    pol = dx.MlpPolicy.from_torch(net)
    ref_pol = _ReferenceMlpPolicy(pol.params.cpu().numpy(), pol.hidden)
    ref = R.evaluator.Evaluator(ref_pol, held, reward_type="dense", max_episode_steps=T_).evaluate_heldout_set(n_eps, seed=42)
    got = ev.evaluate_heldout_set_batched(held, policy=pol, num_episodes_per_object=n_eps, seed=42, reward_type="dense",
                                          max_episode_steps=T_)
    assert len(ref["all_episodes"]) == len(got["all_episodes"]) == 6 * n_eps
    for e0, e1 in zip(ref["all_episodes"], got["all_episodes"]):
        for k in ("episode_steps", "success", "num_contacts", "final_contacts", "contact_history", "object_size",
                  "object_mass", "friction_coefficient", "object_idx", "episode"):
            assert e0[k] == e1[k], k
        assert e1["episode_reward"] == pytest.approx(e0["episode_reward"], rel=1e-12, abs=1e-12)
    for k, v in ref["metrics"].items():
        assert got["metrics"][k] == (pytest.approx(v) if isinstance(v, float) else v), k
    flog = importlib.import_module("evaluation.failure_logger").FailureLogger(log_dir=str(tmp_path),
                                                                              save_full_trajectories=True)
    failed = [e for e in got["all_episodes"] if not e["success"]]
    assert ev.log_failures_batched(got, held, flog, policy=pol) == len(failed) == len(flog.logged_episodes)
    for entry, ep in zip(flog.logged_episodes, failed):
        assert entry["failure_mode"] == ep["failure_mode"] and entry["episode_steps"] == ep["episode_steps"]
    assert os.path.exists(flog.save())


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_fill_mlp_actions_errors_before_any_device_call():
    L = _lib.lib()
    buf = (C.c_char * 512)()
    ptr = (C.addressof(buf) + 15) & ~15                     # non-NULL, 16-byte aligned, never dereferenced
    st = _lib.DexsimState()
    st.n, st.ld = 0, 32                                     # n == 0: a valid call returns before touching the device
    for name, _ in _lib.DexsimState._fields_[2:12]:
        setattr(st, name, ptr)
    p = _lib.DexsimParams()
    p.reward_type, p.success_threshold, p.num_groups, p.max_episode_steps = 1, 3, 1, 200
    pol = _lib.DexsimMlpPolicy(ptr, 2, (C.c_int32 * 2)(64, 64), _lib.ACT_RELU, ptr)

    def call(st_=st, p_=p, groups=ptr, goe=None, policy=pol, actions=ptr):
        return L.dexsim_fill_mlp_actions(None if st_ is None else C.byref(st_), None if p_ is None else C.byref(p_),
                                         groups, goe, None if policy is None else C.byref(policy), actions, None)

    assert call() == 0 and call(goe=ptr) == 0
    assert call(st_=None) == -1001 and call(p_=None) == -1001 and call(policy=None) == -1001
    assert call(actions=None) == -1001 and call(groups=None) == -1001
    pol.params = None
    assert call() == -1001
    pol.params = ptr + 4
    assert call() == -1003                                  # DEXSIM_E_ALIGN
    pol.params = ptr
    pol.action_std = ptr + 8
    assert call() == -1003
    pol.action_std = None
    assert call() == 0                                      # a deterministic policy
    pol.action_std = ptr
    for nh, hid, act in ((0, (8, 8), 0), (3, (8, 8), 0), (1, (0, 8), 0), (1, (65, 8), 0), (2, (8, 0), 0),
                         (2, (8, 65), 0), (1, (8, 8), 2), (1, (8, 8), -1)):
        pol.num_hidden, pol.hidden[0], pol.hidden[1], pol.activation = nh, hid[0], hid[1], act
        assert call() == -1004, (nh, hid, act)             # DEXSIM_E_PARAM
    pol.num_hidden, pol.hidden[0], pol.hidden[1], pol.activation = 2, 64, 64, _lib.ACT_RELU
    for g in (0, 257):
        p.num_groups = g
        assert call() == -1005                              # DEXSIM_E_GROUPS
    p.num_groups = 1
    st.n = -1
    assert call() == -1002
    st.n, st.ld = 33, 32
    assert call() == -1002                                  # ld < n
    st.n, st.ld = 0, 48
    assert call() == -1002                                  # ld % 32
    st.ld = 32
    st.obs = ptr + 4
    assert call() == -1003
    st.obs = ptr
    assert call() == 0


def _fake_policy(device="cuda:1", seed=0, std=0.1, hidden=(8,), act="relu"):
    """An MlpPolicy object built on the host (no device copy): enough for the checks that run before any launch."""
    pol = dx.MlpPolicy.__new__(dx.MlpPolicy)
    params, hid, a = dx.MlpPolicy.pack(_net(hidden, act, seed))
    pol.device, pol.hidden, pol.activation, pol.params = torch.device(device), tuple(hid), a, params
    pol.action_std = None if std is None else torch.cat([torch.full((15,), float(std)), torch.zeros(1)])
    return pol


class _EnvStub:
    device = torch.device("cuda", 0)
    _did_reset = True


def test_policy_actions_host_errors():
    f = dx.BatchedManipulationEnv.policy_actions
    for bad in ("external", "learner", "mlp", 3, None):
        with pytest.raises(ValueError):
            f(_EnvStub(), bad)
    with pytest.raises(ValueError, match="lives on cuda:1"):
        f(_EnvStub(), _fake_policy("cuda:1"))


def test_front_ends_refuse_a_policy_on_another_device():
    pol = _fake_policy("cuda:1")
    cfg = _Held().get_eval_config(0)
    calls = [
        lambda: ev.evaluate_heldout_set_batched(_Held(), policy=pol, seed=1, device="cuda:0"),
        lambda: ev.evaluate_heldout_set_batched(_Held(), policy=pol, seed=1, device="cuda:0", shard=(0, 2)),
        lambda: ev.evaluate_with_noise_batched(cfg, pol, 0.05, 0.0, seed=1, device="cuda:0"),
        lambda: ev.run_robustness_sweep_batched(cfg, [0.0, 0.05], [0.0], policy=pol, seed=1, device="cuda:0"),
        lambda: ev.evaluate_seeds_batched(_Held(), [1, 2], policy=pol, device="cuda:0"),
        lambda: ev.replay_episode(cfg, 1, 0, 0, pol, device="cuda:0"),
    ]
    for c in calls:
        with pytest.raises(ValueError, match="lives on cuda:1"):
            c()


def test_policy_hash_identifies_the_network():
    base = _fake_policy("cuda:0")
    h = base.sha256()
    assert h == _fake_policy("cuda:0").sha256() and len(h) == 64
    for other in (_fake_policy("cuda:0", seed=1), _fake_policy("cuda:0", std=0.2), _fake_policy("cuda:0", std=None),
                  _fake_policy("cuda:0", act="tanh"), _fake_policy("cuda:0", hidden=(8, 8))):
        assert other.sha256() != h


def test_log_failures_refuses_a_missing_or_different_policy():
    pol = _fake_policy("cuda:0")
    ep = {"success": False, "episode_steps": 3, "final_contacts": 0,
          "replay": {"policy": "mlp", "policy_sha256": pol.sha256(), "object_idx": 0}}
    result = {"all_episodes": [ep]}
    for bad in (None, "heuristic", _fake_policy("cuda:0", seed=1), _fake_policy("cuda:0", std=0.2)):
        log = _RecordingLogger()
        with pytest.raises(ValueError):
            ev.log_failures_batched(result, _Held(), log, device="cuda:0", policy=bad)
        assert log.calls == []
    with pytest.raises(ValueError, match="lives on cuda:0"):                 # the right network on the wrong device
        ev.log_failures_batched(result, _Held(), _RecordingLogger(), device="cuda:1", policy=pol)
    # a result without MLP episodes needs no policy
    assert ev.log_failures_batched({"all_episodes": [dict(ep, success=True)]}, _Held(), _RecordingLogger(),
                                   device="cuda:0") == 0
