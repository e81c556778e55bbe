"""Behaviour-policy record of the MLP rollout (``dexsim_rollout_mlp_record``, ``enable_trajectory(policy_record=True)``).

The record is checked against a same-step auto-reset twin stepped with ``step()`` (the approach of
tests/test_rollout_mlp.py): at every step the twin's policy input x is what ``step()`` returned (noisy where the group's
sigma_obs > 0), z = ``fill_normal(4)``, raw = mean(x) + std * z, and

- ``policy_obs`` row t equals x bit for bit; where sigma_obs = 0 it also equals ``obs`` row t-1;
- ``raw_action`` equals raw bit for bit and ``action`` equals clip(raw);
- ``log_prob`` equals the C reference ``log_prob_reference`` (tests/log_prob_reference.c) on those z bit for bit, and
  torch's ``Normal(actor(policy_obs), std).log_prob(raw_action).sum(-1)`` lies within ``_lp_bound`` of it."""
import ctypes as C
import math
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

import test_rollout_mlp as M

U = 2.0 ** -24
POLICY_KEYS = ("policy_obs", "raw_action", "log_prob")


LP_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "log_prob_reference.c")
_lp_lib = None


def _reference_log_prob(std, z):
    """log_prob_reference of tests/log_prob_reference.c, compiled once per session into a temporary directory with the
    flags of the MLP reference: std [15], z [n, 15] -> [n] float32."""
    global _lp_lib
    if _lp_lib is None:
        cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
        if cc is None:
            pytest.skip("needs a C compiler for the reference")
        so = os.path.join(tempfile.mkdtemp(prefix="log_prob_reference_"), "log_prob_reference.so")
        subprocess.run([cc] + M.REF_CFLAGS + ["-shared", "-o", so, LP_SRC, "-lm"], check=True)
        _lp_lib = C.CDLL(so)
        _lp_lib.log_prob_reference.restype = None
    std = np.ascontiguousarray(std, np.float32)
    z = np.ascontiguousarray(z, np.float32).reshape(-1, 15)
    out = np.empty(z.shape[0], np.float32)
    _lp_lib.log_prob_reference(std.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p), C.c_int64(z.shape[0]),
                               out.ctypes.data_as(C.c_void_p))
    return out


def _lp_bound(z, std, mean_err, raw):
    """|torch log_prob - record| per row.  torch recomputes z' = (raw - mu') / std from its own mean mu', which differs
    from the kernel's by at most 2 * mean_err (both within mean_err of the float64 mean); raw itself carries one rounding
    of the product and one of the sum, so z' - z <= E_j = (2 mean_err_j + 2U (|raw_j| + std_j |z_j|)) / std_j (plus the
    division's rounding); -0.5 z^2 then moves by at most (|z_j| + E_j) E_j.  Both sides sum 15 terms and a constant in
    float32: at most 32 U of the sum of their magnitudes."""
    z, std, mean_err, raw = (np.asarray(a, np.float64) for a in (z, std, mean_err, raw))
    E = (2 * mean_err + 2 * U * (np.abs(raw) + std * np.abs(z))) / std + 4 * U * np.abs(z)
    mags = 0.5 * z * z + np.abs(np.log(std)) + 0.5 * math.log(2 * math.pi)
    return ((np.abs(z) + E) * E).sum(-1) + 32 * U * mags.sum(-1) + 1e-6


def _assert_record_equals_twin(twin, tr, pol, sigma_env, where, upto=None):
    """Step the twin through the recorded rows and compare the policy record (and the action) row by row."""
    n = twin.num_envs
    std = None if pol.action_std is None else pol.action_std[:15]
    clean = sigma_env == 0
    for t in range(tr["obs"].shape[0]):
        x = M._policy_input(twin, sigma_env)
        live = torch.ones(n, dtype=torch.bool, device="cuda") if upto is None else t <= upto
        prev = twin._obs[:, :n].t()
        assert torch.equal(tr["policy_obs"][t][live], x[live]), (where, t, "policy_obs")
        if t > 0:
            assert torch.equal(tr["policy_obs"][t][live & clean], tr["obs"][t - 1][live & clean]), (where, t, "obs t-1")
        else:
            assert torch.equal(tr["policy_obs"][0][clean], prev[clean]), (where, "start observation")
        raw = pol.mean(x)
        if std is not None:
            z = M._fill_normal(twin, 4, 15)
            raw = raw + std * z
            lp = _reference_log_prob(std.cpu().numpy(), z.cpu().numpy())
            got = tr["log_prob"][t].cpu().numpy()
            keep = live.cpu().numpy()
            assert M._same_bits(got[keep], lp[keep]), (where, t, "log_prob")
        else:
            assert "log_prob" not in tr
        assert torch.equal(tr["raw_action"][t][live], raw[live]), (where, t, "raw_action")
        act = raw.clamp(-1.0, 1.0)
        assert torch.equal(tr["action"][t][live], act[live]), (where, t, "action = clip(raw_action)")
        twin.step(act.contiguous())


STD = M.STD
# (n, reward, respawn, loop bound, activation, hidden, action_std, per-group sigma_obs, per-group sigma_dyn)
CASES = [
    (100, "dense", True, None, "relu", (64, 64), STD, (0.0, 0.05, 0.0), (0.0, 0.0, 0.1)),
    (4096 + 77, "sparse", False, 6, "tanh", (45,), None, (0.02, 0.0, 0.0), (0.0, 0.1, 0.0)),
    (20_000, "dense", True, 6, "tanh", (64, 64), STD, (0.03, 0.0, 0.01), (0.0, 0.05, 0.05)),
    (70_001, "dense", False, None, "relu", (7,), 0.3, (0.05, 0.05, 0.0), (0.05, 0.0, 0.0)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,reward,respawn,loop,act,hidden,std,so,sd", CASES)
def test_record_equals_step_twin(n, reward, respawn, loop, act, hidden, std, so, sd):
    K = 12
    rec, twin = M._pair(n, reward, respawn, loop, so, sd)
    pol = dx.MlpPolicy.from_torch(M._net(hidden, act, n + 1), action_std=std)
    sigma_env = M._sigma_of_env(rec, so)
    rec.enable_trajectory(K, final_observation=True, policy_record=True)
    for call in range(2):
        rec.rollout(K, policy=pol, respawn=respawn, loop_max_steps=loop)
        tr = rec.trajectory
        assert tr["policy_obs"].shape == (K, n, 45) and tr["raw_action"].shape == (K, n, 15)
        _assert_record_equals_twin(twin, tr, pol, sigma_env, call)
    M._assert_same_end(rec, twin)
    assert int(tr["finished"].sum()) > 0
    if std is not None:                             # the clip is active: raw_action differs from action somewhere
        assert bool((tr["raw_action"].abs() > 1).any())


@pytest.mark.gpu
def test_torch_log_prob_within_bound():
    """What a PPO learner computes from the record in torch agrees with the kernel's log_prob."""
    n, K = 20_000, 10
    rec, twin = M._pair(n, "dense", True, None, (0.0, 0.05, 0.02), 0.0)
    net = M._net((64, 64), "relu", 5)
    pol = dx.MlpPolicy.from_torch(net, action_std=STD)
    rec.enable_trajectory(K, policy_record=True)
    rec.rollout(K, policy=pol)
    tr = rec.trajectory
    x = tr["policy_obs"].reshape(-1, 45)
    std = pol.action_std[:15].cpu()
    with torch.no_grad():
        mu = net.cuda()(x)
        lp = torch.distributions.Normal(mu, pol.action_std[:15]).log_prob(tr["raw_action"].reshape(-1, 15)).sum(-1)
    kmean = pol.mean(x)
    z = ((tr["raw_action"].reshape(-1, 15) - kmean) / pol.action_std[:15]).cpu().numpy()
    _, mean_err = M._bound(pol.params.cpu().numpy(), (64, 64), "relu", x.cpu().numpy())
    bound = _lp_bound(z, std.numpy(), mean_err, tr["raw_action"].reshape(-1, 15).cpu().numpy())
    diff = np.abs(lp.cpu().numpy().astype(np.float64) - tr["log_prob"].reshape(-1).cpu().numpy())
    assert np.all(diff <= bound), float((diff - bound).max())
    assert float(np.median(bound)) < 1e-2          # tight enough to catch a wrong constant or a misplaced std


@pytest.mark.gpu
@pytest.mark.parametrize("final", [False, True])
def test_record_changes_nothing_else(final):
    """The policy record leaves every other output as a plain MLP recording leaves it."""
    n = 5000
    kw = dict(max_episode_steps=M.MAX_STEPS, reward_type="dense", track_episodes=True, seed=9, groups=M._ranged_groups(),
              group_sigma_obs=(0.0, 0.05, 0.0), group_sigma_dyn=(0.0, 0.0, 0.05))
    pol = dx.MlpPolicy.from_torch(M._net((64, 64), "relu", 71), action_std=STD)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    for e in (a, b):
        e.reset(seed=9)
        e.enable_episode_log(60 * n)
        e.enable_history(60)
    a.enable_trajectory(25, final_observation=final, policy_record=True)
    b.enable_trajectory(25, final_observation=final)
    for k in (25, 20, 15):
        a.rollout(k, policy=pol, respawn=False)
        b.rollout(k, policy=pol, respawn=False)
        ta, tb = a.trajectory, b.trajectory
        assert set(ta) == set(tb) | set(POLICY_KEYS)
        for name, v in tb.items():
            if name == "final_observation":
                v, w = v[tb["finished"]], ta[name][tb["finished"]]
            else:
                w = ta[name]
            assert torch.equal(v, w), name
    M._assert_same_end(a, b)
    assert np.array_equal(a.read_episode_log(), b.read_episode_log())
    assert torch.equal(a._hist, b._hist)


@pytest.mark.gpu
def test_one_episode_rows_after_stop_untouched():
    n, K = 4096 + 77, M.MAX_STEPS + 6
    rec, twin = M._pair(n, "dense", False, None, (0.0, 0.04, 0.0))
    pol = dx.MlpPolicy.from_torch(M._net((64, 64), "relu", 41), action_std=0.1)
    rec.enable_trajectory(K, final_observation=True, policy_record=True)
    for name in POLICY_KEYS:
        rec._traj[name].fill_(float("nan"))
    rec.rollout(K, policy=pol, one_episode=True, respawn=False)
    tr = rec.trajectory
    fin = tr["finished"].to(torch.uint8)
    assert bool((fin.sum(0) == 1).all())
    end = fin.argmax(0)
    _assert_record_equals_twin(twin, tr, pol, M._sigma_of_env(rec, (0.0, 0.04, 0.0)), "one_episode", upto=end)
    rows = torch.arange(K, device="cuda")[:, None]
    after = rows > end[None, :]
    assert bool(after.any())
    for name in POLICY_KEYS:
        v = tr[name]
        nan = torch.isnan(v) if v.dim() == 2 else torch.isnan(v).all(-1)
        written = ~torch.isnan(v) if v.dim() == 2 else ~torch.isnan(v).any(-1)
        assert bool(nan[after].all()) and bool(written[~after].all()), name


@pytest.mark.gpu
@pytest.mark.parametrize("n", [130, 70_001])
def test_no_writes_outside_record(n):
    cap, k, guard = 16, 10, 4096
    rec, _ = M._pair(n, "dense", True, None, (0.0, 0.05, 0.0), (0.0, 0.0, 0.05))
    pol = dx.MlpPolicy.from_torch(M._net((64, 64), "tanh", 91), action_std=STD)
    rec.enable_trajectory(cap, final_observation=True, policy_record=True)
    bands = {}
    for name in POLICY_KEYS:
        t = rec._traj[name]
        nbytes = t.numel() * t.element_size()
        big = torch.full((nbytes + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
        rec._traj[name] = big[guard:guard + nbytes].view(t.dtype).view(t.shape)
        bands[name] = (big, rec._traj[name], rec._traj[name].clone())
    rec.rollout(k, policy=pol, loop_max_steps=4)
    torch.cuda.synchronize()
    for name, (big, inner, pattern) in bands.items():
        assert bool((big[:guard] == 0xA5).all()) and bool((big[-guard:] == 0xA5).all()), name
        assert torch.equal(inner[k:], pattern[k:]), (name, "rows past k")
        assert torch.equal(inner[..., n:], pattern[..., n:]), (name, "columns past n")
        assert not torch.equal(inner[:k, ..., :n], pattern[:k, ..., :n]), (name, "written")
    assert int(rec.trajectory["finished"].sum()) > 0


@pytest.mark.gpu
def test_truncation_wave_at_full_size():
    """1,048,576 envs whose episodes all end at the bound on the same step, twice in an 8-step recorded rollout."""
    n, K, T = 1 << 20, 8, 3
    kw = dict(max_episode_steps=T, reward_type="dense", track_episodes=True, seed=21,
              curriculum_config=dx.CurriculumConfig.hard())
    rec = dx.BatchedManipulationEnv(n, "cuda", **kw)
    twin = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, respawn=True,
                                     loop_max_steps=T, **kw)
    for e in (rec, twin):
        e._params.success_threshold = 6
        e.reset(seed=21)
    pol = dx.MlpPolicy.from_torch(M._net((64, 64), "relu", 51), action_std=STD)
    rec.enable_trajectory(K, final_observation=True, policy_record=True)
    rec.rollout(K, policy=pol)
    tr = rec.trajectory
    assert [t for t in range(K) if bool(tr["finished"][t].all())] == [T - 1, 2 * T - 1]
    _assert_record_equals_twin(twin, tr, pol, torch.zeros(n, device="cuda"), "wave")
    M._assert_same_end(rec, twin)


@pytest.mark.gpu
def test_python_guards():
    env = dx.BatchedManipulationEnv(256, "cuda", max_episode_steps=10, reward_type="dense", track_episodes=True, seed=1)
    env.reset(seed=1)
    env.enable_trajectory(5, policy_record=True)
    with pytest.raises(ValueError):
        env.rollout(5, policy="random")             # only an MlpPolicy fills the record
    net = M._net((8,), "relu", 2)
    for bad in (0.0, -0.1, float("nan"), float("inf"), [0.1] * 14 + [0.0]):
        with pytest.raises(ValueError):
            env.rollout(5, policy=dx.MlpPolicy.from_torch(net, action_std=bad))
    env.rollout(5, policy=dx.MlpPolicy.from_torch(net))          # deterministic: no density, no log_prob
    tr = env.trajectory
    assert "log_prob" not in tr and torch.equal(tr["raw_action"].clamp(-1, 1), tr["action"])
    env.rollout(5, policy=dx.MlpPolicy.from_torch(net, action_std=0.2))
    assert env.trajectory["log_prob"].shape == (5, 256)


# ---- the PPO example -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ppo_example_two_iterations():
    """Two iterations at 4,096 envs with observation noise: before the first update the torch actor reproduces the
    recorded log-probabilities (|log ratio| below 1e-3: _lp_bound with the example's std >= e^-1.1 and mean errors
    of order 1e-6), and every loss is finite."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    try:
        import ppo_mlp
    finally:
        sys.path.pop(0)
    hist = ppo_mlp.train(envs=4096, iters=2, steps=16, sigma_obs=(0.0, 0.05), seed=3, log=None)
    assert len(hist) == 2
    assert hist[0]["max_abs_log_ratio0"] < 1e-3
    for h in hist:
        assert all(math.isfinite(v) for v in h["pg_loss"] + h["v_loss"])
        assert math.isfinite(h["max_abs_log_ratio0"])


# ---- CPU -------------------------------------------------------------------------------------------------------------
def test_reference_log_prob_within_float32_bound_of_float64():
    rng = np.random.default_rng(3)
    for std in (np.full(15, 0.1), np.asarray(STD), rng.uniform(1e-3, 5.0, 15)):
        std = std.astype(np.float32)
        z = rng.normal(0, 1, (4000, 15)).astype(np.float32)
        z[:10] *= 8                                 # tails
        got = _reference_log_prob(std, z).astype(np.float64)
        z64 = z.astype(np.float64)
        want = -0.5 * (z64 * z64).sum(-1) - np.log(std.astype(np.float64)).sum() - 7.5 * math.log(2 * math.pi)
        mags = 0.5 * (z64 * z64).sum(-1) + np.abs(np.log(std.astype(np.float64))).sum() + 7.5 * math.log(2 * math.pi)
        assert np.all(np.abs(got - want) <= 18 * U * mags)


def test_errors_before_any_device_call():
    L = _lib.lib()
    assert L.dexsim_sizeof_policy_record() == C.sizeof(_lib.DexsimPolicyRecord) == 24
    buf = (C.c_char * 512)()
    ptr = (C.addressof(buf) + 15) & ~15
    st = _lib.DexsimState()
    st.n, st.ld = 0, 32
    for name, _ in _lib.DexsimState._fields_[2:]:
        setattr(st, name, ptr)
    p = _lib.DexsimParams()
    p.reward_type, p.success_threshold, p.num_groups, p.max_episode_steps = 1, 3, 1, 200
    rio = _lib.DexsimRolloutIO()
    pol = _lib.DexsimMlpPolicy(ptr, 2, (C.c_int32 * 2)(64, 64), _lib.ACT_RELU, ptr)
    tr = _lib.DexsimTrajectory(ptr, ptr, ptr, ptr, ptr, ptr, 5)
    prec = _lib.DexsimPolicyRecord(ptr, ptr, ptr)

    def call(k=5, policy=pol, traj=tr, fo=ptr, rec=prec):
        return L.dexsim_rollout_mlp_record(C.byref(st), C.byref(p), ptr, None, k, C.byref(rio),
                                           None if policy is None else C.byref(policy),
                                           None if traj is None else C.byref(traj), fo,
                                           None if rec is None else C.byref(rec), None)

    assert call() == 0 and call(fo=None) == 0
    assert call(rec=None) == -1001 and call(traj=None, fo=None) == -1001 and call(policy=None) == -1001
    for name in ("obs", "raw_action", "log_prob"):
        setattr(prec, name, ptr + 4)
        assert call() == -1003, name
        setattr(prec, name, None)
        assert call() == 0, name                    # every array is optional
        setattr(prec, name, ptr)
    pol.action_std = None
    assert call() == -1004                          # log_prob of a deterministic policy
    prec.log_prob = None
    assert call() == 0
    prec.log_prob, pol.action_std = ptr, ptr
    # the errors of dexsim_rollout_mlp
    assert call(k=0) == -1002 and call(k=6) == -1002 and call(fo=ptr + 4) == -1003
    pol.num_hidden = 3
    assert call() == -1004
    pol.num_hidden = 2
    rio.actions = ptr
    assert call() == -1004
    rio.actions = None
    tr.obs = None
    assert call() == -1001
    tr.obs = ptr
    p.num_groups = 0
    assert call() == -1005
    p.num_groups = 1
    assert call() == 0
