"""MLP policy inside the fused rollout (``MlpPolicy``, ``dexsim_rollout_mlp``, ``dexsim_mlp_policy_mean``).

The arithmetic contract (include/dexsim.h): every neuron is an ascending fmaf chain from 0 and one float32 bias
addition; ReLU is exact, tanh is the device tanhf.  A C restatement (``tests/mlp_reference.c``, built here with the
oracle's flags) is the reference: with ReLU the mean kernel must equal it bit for bit, with tanh both must lie within the
error bound ``_bound`` of a float64 forward pass.

The fusion is checked against a same-step auto-reset twin stepped with ``step()``: at every step the twin's action is
clip(mean(observation) + std * fill_normal(stream 4)), the mean computed by ``dexsim_mlp_policy_mean`` on the
observation ``step()`` returned (noisy where the group's sigma_obs > 0), and every recorded row, the final state, the
counters and the return sums must equal the twin's bit for bit."""
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

STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
         "_ep_return", "_ep_stats")
MAX_STEPS = 20
U = 2.0 ** -24                   # unit roundoff of float32
TINY = 2.0 ** -149               # smallest subnormal: the absolute error of one rounding in the subnormal range
TANHF_ULP = 2                    # CUDA Programming Guide, Mathematical Functions: tanhf, maximum 2 ulp (glibc: 2 ulp too)


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


REF_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mlp_reference.c")
# the flags of oracle/Makefile: no contraction, no fast math, SSE2 float arithmetic
REF_CFLAGS = ["-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fexcess-precision=standard", "-msse2",
              "-mfpmath=sse"]
_ref_lib = None


def _reference_mean(params, hidden, act, obs):
    """mlp_reference_mean of tests/mlp_reference.c, compiled once per session into a temporary directory:
    obs [n, 45] -> [n, 15] float32."""
    global _ref_lib
    if _ref_lib is None:
        cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
        if cc is None:
            pytest.skip("needs a C compiler for the reference")
        so = os.path.join(tempfile.mkdtemp(prefix="mlp_reference_"), "mlp_reference.so")
        subprocess.run([cc] + REF_CFLAGS + ["-shared", "-o", so, REF_SRC, "-lm"], check=True)
        _ref_lib = C.CDLL(so)
        _ref_lib.mlp_reference_mean.restype = None
    params = np.ascontiguousarray(params, dtype=np.float32)
    obs = np.ascontiguousarray(obs, dtype=np.float32).reshape(-1, 45)
    hid = (C.c_int32 * 2)(*[int(h) for h in (list(hidden) + [0])[:2]])
    out = np.empty((obs.shape[0], 15), np.float32)
    _ref_lib.mlp_reference_mean(params.ctypes.data_as(C.c_void_p), C.c_int32(len(hidden)), hid,
                                C.c_int32(0 if act == "relu" else 1), obs.ctypes.data_as(C.c_void_p),
                                C.c_int64(obs.shape[0]), out.ctypes.data_as(C.c_void_p))
    return out


def _net(hidden, act, seed):
    torch.manual_seed(seed)
    A = torch.nn.ReLU if act == "relu" else torch.nn.Tanh
    sizes = (45,) + tuple(hidden)
    layers = []
    for i, o in zip(sizes[:-1], sizes[1:]):
        layers += [torch.nn.Linear(i, o), A()]
    return torch.nn.Sequential(*layers, torch.nn.Linear(sizes[-1], 15))


def _layers(params, hidden):
    """Packed params -> [(W [out, in], b [out])] as float64 arrays."""
    p = np.asarray(params, np.float32).astype(np.float64)
    sizes, out, at = (45,) + tuple(hidden) + (15,), [], 0
    for i, o in zip(sizes[:-1], sizes[1:]):
        out.append((p[at:at + o * i].reshape(o, i), p[at + o * i:at + o * i + o]))
        at += o * i + o
    return out


def _bound(params, hidden, act, obs):
    """float64 forward pass and a rigorous bound on |float32 result - it| per output, [n, 15] each.

    One layer with exact inputs x, computed inputs x^ = x + e (|e| <= E) and n inputs: the fmaf chain plus the bias
    addition is n + 1 roundings of partial sums bounded by sum |W||x^| + |b|, so (Higham, Accuracy and Stability,
    eq. 3.5) |y^ - (W x^ + b)| <= g(n + 1) (|W| (|x| + E) + |b|) + (n + 1) TINY, g(k) = k u / (1 - k u); and
    |W x^ - W x| <= |W| E.  ReLU is 1-Lipschitz and exact.  tanh is 1-Lipschitz and tanhf adds at most TANHF_ULP ulp
    of its result, an ulp of t being at most 2u |t| (+ TINY below the normal range)."""
    g = lambda k: k * U / (1 - k * U)
    x = np.asarray(obs, np.float32).astype(np.float64)
    err = np.zeros_like(x)
    layers = _layers(params, hidden)
    for li, (W, b) in enumerate(layers):
        n_in = W.shape[1]
        y = x @ W.T + b
        mag = (np.abs(x) + err) @ np.abs(W).T + np.abs(b)
        e = err @ np.abs(W).T + g(n_in + 1) * mag + (n_in + 1) * TINY
        if li < len(layers) - 1:
            if act == "relu":
                y = np.maximum(y, 0.0)
            else:
                y = np.tanh(y)
                e = e + TANHF_ULP * 2 * U * (np.abs(y) + e) + TANHF_ULP * TINY
        x, err = y, e
    return x, err


def _same_bits(a, b):
    """Bit-equal float32 arrays, any NaN matching any NaN (the payload of a NaN the arithmetic creates is the
    platform's)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


def _obs_batch(n, seed):
    """Observations of the kind stepping produces: joints in [-1, 1], small velocities, object pose, 0/1 contacts."""
    r = np.random.default_rng(seed)
    o = np.empty((n, 45), np.float32)
    o[:, :15] = r.uniform(-1, 1, (n, 15))
    o[:, 15:30] = r.normal(0, 0.05, (n, 15))
    o[:, 30:33] = r.uniform(-0.2, 0.3, (n, 3))
    o[:, 33:37] = (1, 0, 0, 0)
    o[:, 37:40] = r.normal(0, 0.1, (n, 3))
    o[:, 40:45] = r.integers(0, 2, (n, 5))
    return o


def _hostile(n, seed):
    """NaN, +-inf, 1e30, subnormals and signed zeros scattered over ordinary observations."""
    o = _obs_batch(n, seed)
    r = np.random.default_rng(seed + 1)
    special = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30, 1e-40, -1e-40, 1e-45, 0.0, -0.0], np.float32)
    mask = r.random(o.shape) < 0.05
    o[mask] = r.choice(special, int(mask.sum()))
    return o


SHAPES = [(1,), (7,), (45,), (64,), (1, 64), (7, 45), (64, 7), (64, 64)]


# ---- CPU -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hidden", SHAPES)
@pytest.mark.parametrize("act", ["relu", "tanh"])
def test_reference_mean_within_float32_bound_of_float64(hidden, act):
    params, _, _ = dx.MlpPolicy.pack(_net(hidden, act, 3))
    obs = _obs_batch(2000, 4)
    got = _reference_mean(params.numpy(), hidden, act, obs).astype(np.float64)
    ref, bound = _bound(params.numpy(), hidden, act, obs)
    assert np.all(np.abs(got - ref) <= bound)
    assert np.all(bound < 1e-4)                  # the bound is tight enough to catch a misplaced term


@pytest.mark.parametrize("hidden", SHAPES)
@pytest.mark.parametrize("act", ["relu", "tanh"])
def test_packing_plus_reference_equals_torch_forward(hidden, act):
    """A transposed or misordered layer would not come within a float32 summation-order tolerance of torch."""
    net = _net(hidden, act, 11)
    params, hid, a = dx.MlpPolicy.pack(net)
    assert list(hid) == list(hidden) and a == act
    obs = _obs_batch(500, 12)
    got = _reference_mean(params.numpy(), hid, a, obs)
    with torch.no_grad():
        want = net(torch.from_numpy(obs)).numpy()
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5)


def test_from_torch_rejects_unsupported_modules():
    nn = torch.nn
    bad = [
        nn.Linear(45, 15),
        nn.Sequential(nn.Linear(45, 15)),
        nn.Sequential(nn.Linear(45, 8), nn.Sigmoid(), nn.Linear(8, 15)),
        nn.Sequential(nn.Linear(45, 8), nn.ReLU(), nn.Linear(8, 8), nn.Tanh(), nn.Linear(8, 15)),
        nn.Sequential(nn.Linear(44, 8), nn.ReLU(), nn.Linear(8, 15)),
        nn.Sequential(nn.Linear(45, 8), nn.ReLU(), nn.Linear(8, 14)),
        nn.Sequential(nn.Linear(45, 8), nn.ReLU(), nn.Linear(9, 15)),
        nn.Sequential(nn.Linear(45, 65), nn.ReLU(), nn.Linear(65, 15)),
        nn.Sequential(nn.Linear(45, 8, bias=False), nn.ReLU(), nn.Linear(8, 15)),
        nn.Sequential(nn.Linear(45, 8), nn.ReLU(), nn.Linear(8, 8), nn.ReLU(), nn.Linear(8, 8), nn.ReLU(),
                      nn.Linear(8, 15)),
        nn.Sequential(nn.Linear(45, 8), nn.ReLU(), nn.Dropout(), nn.Linear(8, 15)),
    ]
    for m in bad:
        with pytest.raises(ValueError):
            dx.MlpPolicy.pack(m)


def test_errors_before_any_device_call():
    """Each argument error of dexsim_rollout_mlp and dexsim_mlp_policy_mean comes back before the device is touched."""
    L = _lib.lib()
    assert L.dexsim_sizeof_mlp_policy() == C.sizeof(_lib.DexsimMlpPolicy) == 32
    buf = (C.c_char * 512)()
    ptr = (C.addressof(buf) + 15) & ~15                     # any non-NULL, 16-byte aligned address: never dereferenced
    st = _lib.DexsimState()
    st.n, st.ld = 0, 32                                     # n == 0: a valid call returns before touching the device
    for name, _ in _lib.DexsimState._fields_[2:]:
        setattr(st, name, ptr)
    p = _lib.DexsimParams()
    p.reward_type, p.success_threshold, p.num_groups, p.max_episode_steps = 1, 3, 1, 200
    rio = _lib.DexsimRolloutIO()
    pol = _lib.DexsimMlpPolicy(ptr, 2, (C.c_int32 * 2)(64, 64), _lib.ACT_RELU, ptr)
    tr = _lib.DexsimTrajectory(ptr, ptr, ptr, ptr, ptr, ptr, 5)

    def call(k=5, policy=pol, traj=tr, fo=ptr):
        return L.dexsim_rollout_mlp(C.byref(st), C.byref(p), ptr, None, k, C.byref(rio),
                                    None if policy is None else C.byref(policy), None if traj is None else C.byref(traj),
                                    fo, None)

    def mean(policy=pol, obs=ptr, n=0, ld=32, out=ptr):
        return L.dexsim_mlp_policy_mean(None if policy is None else C.byref(policy), obs, n, ld, out, None)

    assert call() == 0 and call(traj=None, fo=None) == 0 and call(fo=None) == 0 and mean() == 0
    for f in (call, mean):
        assert f(policy=None) == -1001                      # DEXSIM_E_NULL
        pol.params = None
        assert f() == -1001
        pol.params = ptr + 4
        assert f() == -1003                                 # DEXSIM_E_ALIGN
        pol.params = ptr
        pol.action_std = ptr + 8
        assert f() == -1003
        pol.action_std = None
        assert f() == 0                                     # a deterministic policy
        pol.action_std = ptr
        for nh, hid, act in ((0, (8, 8), 0), (3, (8, 8), 0), (1, (0, 8), 0), (1, (65, 8), 0), (2, (8, 0), 0),
                             (2, (8, 65), 0), (1, (8, 8), 2), (1, (8, 8), -1)):
            pol.num_hidden, pol.hidden[0], pol.hidden[1], pol.activation = nh, hid[0], hid[1], act
            assert f() == -1004, (nh, hid, act)             # DEXSIM_E_PARAM
        pol.num_hidden, pol.hidden[0], pol.hidden[1], pol.activation = 1, 64, 0, _lib.ACT_TANH   # hidden[1] ignored
        assert f() == 0
        pol.num_hidden, pol.hidden[0], pol.hidden[1], pol.activation = 2, 64, 64, _lib.ACT_RELU
    # the rollout's own arguments
    assert call(traj=None) == -1001                         # final_obs without a trajectory
    assert call(fo=ptr + 4) == -1003
    assert call(k=0) == -1002 and call(k=6) == -1002        # k_steps < 1, k_steps > capacity
    for name in ("actions", "learner_mean", "learner_best", "learner_act_noise", "learner_upd_noise"):
        setattr(rio, name, ptr)
        assert call() == -1004, name                        # an MLP launch takes no actions and no learner
        setattr(rio, name, None)
    for name in ("obs", "action", "reward", "terminated", "truncated", "finished"):
        setattr(tr, name, None)
        assert call() == -1001, name
        setattr(tr, name, ptr + 4)
        assert call() == -1003, name
        setattr(tr, name, ptr)
    p.num_groups = 0
    assert call() == -1005                                  # rollout_launch's checks apply
    p.num_groups = 1
    try:
        _lib.set_rollout_impl("split")                      # never the 5-lanes-per-env kernel
        assert call() == 0 and call(traj=None, fo=None) == 0
    finally:
        _lib.set_rollout_impl("auto")
    # the mean's sizes
    assert mean(n=-1) == -1002 and mean(n=33, ld=32) == -1002 and mean(n=5, ld=40) == -1002
    assert mean(n=5, obs=None) == -1001 and mean(n=5, out=None) == -1001
    # dexsim_rollout's accepted policy kinds are unchanged: the MLP's internal kind is refused there
    assert L.dexsim_rollout(C.byref(st), C.byref(p), ptr, None, 5, 4, C.byref(rio), None) == -1004


# ---- GPU: the mean kernel -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("hidden", SHAPES)
def test_mean_kernel_relu_bit_exact_vs_reference(gpu, hidden):
    pol = dx.MlpPolicy.from_torch(_net(hidden, "relu", 21))
    for obs in (_obs_batch(3001, 22), _hostile(3001, 23)):
        got = pol.mean(torch.from_numpy(obs)).cpu().numpy()
        want = _reference_mean(pol.params.cpu().numpy(), hidden, "relu", obs)
        assert _same_bits(got, want)
    assert np.isnan(want).any() and not np.isnan(want).all()


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", SHAPES)
def test_mean_kernel_tanh_within_bound(gpu, hidden):
    pol = dx.MlpPolicy.from_torch(_net(hidden, "tanh", 31))
    obs = _obs_batch(3001, 32)
    got = pol.mean(torch.from_numpy(obs)).cpu().numpy().astype(np.float64)
    ref, bound = _bound(pol.params.cpu().numpy(), hidden, "tanh", obs)
    assert np.all(np.abs(got - ref) <= bound)


# ---- GPU: the fused rollout against a step() twin -------------------------------------------------------------------
def _ranged_groups():
    CC = dx.CurriculumConfig
    return [CC(object_size=s, object_size_range=(0.7 * s, 1.3 * s), object_mass=m, object_mass_range=(0.5 * m, 1.5 * m),
               friction_coefficient=f, friction_range=(0.6 * f, min(1.0, 1.4 * f)))
            for s, m, f in ((0.08, 0.05, 0.8), (0.05, 0.1, 0.5), (0.03, 0.2, 0.3))]


def _pair(n, reward="dense", respawn=True, loop=None, sigma_obs=0.0, sigma_dyn=0.0, seed=5, **kw):
    common = dict(max_episode_steps=MAX_STEPS, reward_type=reward, track_episodes=True, seed=seed, respawn=respawn,
                  groups=_ranged_groups(), group_sigma_obs=sigma_obs, group_sigma_dyn=sigma_dyn, **kw)
    rec = dx.BatchedManipulationEnv(n, "cuda", **common)
    twin = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True,
                                     loop_max_steps=MAX_STEPS if loop is None else loop, **common)
    rec.reset(seed=seed); twin.reset(seed=seed)
    return rec, twin


def _fill_normal(env, stream, rows):
    out = torch.zeros(rows, env.ld, dtype=torch.float32, device=env.device)
    _lib.check(env._lib.dexsim_fill_normal(C.byref(env._state), C.byref(env._params), stream, rows, C.c_float(1.0),
                                           out.data_ptr(), env._stream()), "dexsim_fill_normal")
    return out[:, :env.num_envs].t()


def _sigma_of_env(env, sigma_obs):
    G = env.num_groups
    s = torch.tensor(np.broadcast_to(np.asarray(sigma_obs, np.float32), (G,)).copy(), device=env.device)
    gid = torch.arange(env.num_envs, device=env.device, dtype=torch.int64) + env.env_gid0
    return s[gid % G]


def _policy_input(env, sigma_env):
    """What step() returns for the env's current state: obs + sigma * z (stream 3) where sigma > 0."""
    obs = env._obs[:, :env.num_envs].t()
    if not bool((sigma_env > 0).any()):
        return obs
    z = _fill_normal(env, _lib.RNG_STREAM_OBS, 45)
    return torch.where(sigma_env[:, None] > 0, obs + sigma_env[:, None] * z, obs)


def _twin_action(twin, pol, x):
    mean = pol.mean(x)
    if pol.action_std is not None:
        mean = mean + pol.action_std[:15] * _fill_normal(twin, 4, 15)
    return mean.clamp(-1.0, 1.0)


def _assert_rows_equal_twin(twin, tr, pol, sigma_env, where, upto=None):
    """Step the twin through the recorded rows.  `upto` [n]: compare env i only on rows t <= upto[i] (one_episode)."""
    n = twin.num_envs
    for t in range(tr["obs"].shape[0]):
        x = _policy_input(twin, sigma_env)
        act = _twin_action(twin, pol, x)
        live = torch.ones(n, dtype=torch.bool, device="cuda") if upto is None else t <= upto
        assert torch.equal(tr["action"][t][live], act[live]), (where, t, "action")
        obs, rew, term, trunc, info = twin.step(act.contiguous())
        noisy = sigma_env > 0
        assert torch.equal(obs[noisy], _policy_input(twin, sigma_env)[noisy]), (where, t, "noisy observation")
        fin = info["finished"]
        # one_episode: the ending row holds the terminal observation (the env is not reset), the twin's final one
        before = live if upto is None else t < upto
        assert torch.equal(tr["obs"][t][before], twin._obs[:, :n].t()[before]), (where, t, "obs")
        if upto is not None:
            ending = t == upto
            assert torch.equal(tr["obs"][t][ending], info["final_observation"][ending]), (where, t, "terminal obs")
        for name, want in (("reward", rew), ("terminated", term), ("truncated", trunc), ("finished", fin)):
            assert torch.equal(tr[name][t][live], want[live]), (where, t, name)
        # step_final returns the NOISY terminal observation where noise is on; the recording holds the env's own
        sel = fin & live & ~noisy
        assert torch.equal(tr["final_observation"][t][sel], info["final_observation"][sel]), (where, t, "final")


def _assert_same_end(a, b):
    n = a.num_envs
    for k in STATE:
        assert torch.equal(getattr(a, k)[..., :n], getattr(b, k)[..., :n]), k
    assert torch.equal(a.counters, b.counters)
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0.0)


STD = tuple(0.05 + 0.02 * j for j in range(15))
# (n, reward, respawn, loop bound, activation, hidden, action_std, per-group sigma_obs, per-group sigma_dyn)
TWIN_CASES = [
    (100, "dense", True, None, "relu", (64, 64), STD, (0.0, 0.05, 0.0), (0.0, 0.0, 0.1)),
    (4096 + 77, "sparse", False, 6, "tanh", (45,), None, (0.02, 0.0, 0.0), (0.0, 0.1, 0.0)),
    (4096 + 77, "dense", True, 6, "tanh", (7, 64), STD, 0.0, 0.0),
    (70_001, "dense", False, None, "relu", (1,), STD, (0.05, 0.05, 0.05), (0.05, 0.0, 0.0)),
    (70_001, "sparse", True, 6, "relu", (64, 7), None, (0.0, 0.03, 0.0), 0.0),
    (20_000, "dense", True, None, "tanh", (64, 64), STD, (0.03, 0.0, 0.01), (0.0, 0.05, 0.05)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,reward,respawn,loop,act,hidden,std,so,sd", TWIN_CASES)
def test_rollout_rows_equal_step_twin(gpu, n, reward, respawn, loop, act, hidden, std, so, sd):
    K = 12
    rec, twin = _pair(n, reward, respawn, loop, so, sd)
    pol = dx.MlpPolicy.from_torch(_net(hidden, act, n), action_std=std)
    sigma_env = _sigma_of_env(rec, so)
    rec.enable_trajectory(K, final_observation=True)
    finished = 0
    for call in range(2):                      # two consecutive calls: the second starts where the first left off
        rec.rollout(K, policy=pol, respawn=respawn, loop_max_steps=loop)
        tr = rec.trajectory
        assert tr["action"].shape == (K, n, 15) and float(tr["action"].abs().max()) <= 1.0
        _assert_rows_equal_twin(twin, tr, pol, sigma_env, call)
        finished += int(tr["finished"].sum())
    _assert_same_end(rec, twin)
    assert finished > 0
    a = tr["action"]
    assert 0.05 < float((a.abs() < 1).float().mean())           # the policy is not saturated everywhere


@pytest.mark.gpu
def test_one_episode_rows_equal_step_twin(gpu):
    n, K = 4096 + 77, MAX_STEPS + 6
    rec, twin = _pair(n, "dense", False, None)
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 41), action_std=0.1)
    rec.enable_trajectory(K, final_observation=True)
    rec.rollout(K, policy=pol, one_episode=True, respawn=False)
    tr = rec.trajectory
    fin = tr["finished"].to(torch.uint8)
    assert bool((fin.sum(0) == 1).all())
    end = fin.argmax(0)
    _assert_rows_equal_twin(twin, tr, pol, torch.zeros(n, device="cuda"), "one_episode", upto=end)
    cols = torch.arange(n, device="cuda")
    assert torch.equal(tr["final_observation"][end, cols], rec._obs[:, :n].t())
    assert int(rec.counters[:, _lib.CNT_EPISODES].sum()) == n


@pytest.mark.gpu
def test_truncation_wave_at_full_size(gpu):
    """1,048,576 envs whose episodes all end at the bound on the same step, twice in an 8-step recorded rollout."""
    n, K, T = 1 << 20, 8, 3
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=T, reward_type="dense", track_episodes=True, seed=21, curriculum_config=CC.hard())
    rec = dx.BatchedManipulationEnv(n, "cuda", **kw)
    twin = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, respawn=True,
                                     loop_max_steps=T, **kw)
    for e in (rec, twin):
        e._params.success_threshold = 6          # five fingers: no episode terminates, every one ends at the bound
        e.reset(seed=21)
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 51), action_std=STD)
    rec.enable_trajectory(K, final_observation=True)
    rec.rollout(K, policy=pol)
    tr = rec.trajectory
    waves = [t for t in range(K) if bool(tr["finished"][t].all())]
    assert waves == [T - 1, 2 * T - 1] and int(tr["finished"].sum()) == 2 * n
    _assert_rows_equal_twin(twin, tr, pol, torch.zeros(n, device="cuda"), "wave")
    _assert_same_end(rec, twin)


@pytest.mark.gpu
def test_three_shards_equal_one(gpu):
    """Shards with env_gid0 offsets produce, concatenated, what one env of all their envs produces."""
    n, K, parts = 3 * 4099, 12, 3
    kw = dict(max_episode_steps=MAX_STEPS, reward_type="dense", track_episodes=True, seed=61, groups=_ranged_groups(),
              group_sigma_obs=(0.0, 0.04, 0.02), group_sigma_dyn=(0.05, 0.0, 0.0))
    pol = dx.MlpPolicy.from_torch(_net((32, 16), "tanh", 62), action_std=STD)
    whole = dx.BatchedManipulationEnv(n, "cuda", **kw)
    shards = [dx.BatchedManipulationEnv(n // parts, "cuda", env_gid0=s * (n // parts), **kw) for s in range(parts)]
    for e in [whole] + shards:
        e.reset(seed=61)
        e.enable_trajectory(K, final_observation=True)
        e.enable_episode_log(4 * n)
        for _ in range(2):
            e.rollout(K, policy=pol)
    for name, v in whole.trajectory.items():
        cat = torch.cat([s.trajectory[name] for s in shards], dim=1)
        fin = whole.trajectory["finished"]
        if name == "final_observation":
            v, cat = v[fin], cat[fin]
        assert torch.equal(v, cat), name
    for k in STATE:
        assert torch.equal(getattr(whole, k)[..., :n], torch.cat([getattr(s, k)[..., :n // parts] for s in shards], -1)), k
    assert torch.equal(whole.counters, sum(s.counters for s in shards))
    la = whole.read_episode_log()
    lb = np.sort(np.concatenate([s.read_episode_log() for s in shards]), order=["t_end", "env_gid"])
    assert len(la) > 0 and np.array_equal(la, lb)


@pytest.mark.gpu
@pytest.mark.parametrize("final", [False, True])
def test_recording_changes_nothing_else(gpu, final):
    """A recording MLP rollout and a plain one leave identical state, counters, return sums, episode log and history."""
    n = 5000
    kw = dict(max_episode_steps=MAX_STEPS, reward_type="dense", track_episodes=True, seed=9, groups=_ranged_groups(),
              group_sigma_obs=(0.0, 0.05, 0.0), group_sigma_dyn=(0.0, 0.0, 0.05))
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 71), action_std=STD)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    for e in (a, b):
        e.reset(seed=9)
        e.enable_episode_log(60 * n)
        e.enable_history(60)
    a.enable_trajectory(25, final_observation=final)
    for k in (25, 20, 15):
        a.rollout(k, policy=pol, respawn=False)
        b.rollout(k, policy=pol, respawn=False)
    _assert_same_end(a, b)
    la, lb = a.read_episode_log(), b.read_episode_log()
    assert a.episode_log_overflow == 0 and len(la) > n and np.array_equal(la, lb)
    assert torch.equal(a._hist, b._hist)


@pytest.mark.gpu
def test_observation_noise_changes_the_trajectory(gpu):
    """With a policy that reads the observation, sigma_obs > 0 changes the actions and the states reached; the
    heuristic policy, which ignores the observation, reaches the same state with and without the noise."""
    n, K = 4096, 10
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "relu", 81))         # deterministic: only the input can differ
    runs = []
    for so in (0.0, 0.05):
        e = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=MAX_STEPS, reward_type="dense", track_episodes=True,
                                      seed=3, observation_noise_std=so)
        e.reset(seed=3)
        e.enable_trajectory(K)
        e.rollout(K, policy=pol)
        runs.append({k: v.clone() for k, v in e.trajectory.items()})
    clean, noisy = runs
    assert not torch.equal(clean["action"][0], noisy["action"][0])
    assert not torch.equal(clean["obs"][-1], noisy["obs"][-1])
    # the random and heuristic policies ignore the observation: the same noise changes nothing for them
    outs = []
    for so in (0.0, 0.05):
        e = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=MAX_STEPS, reward_type="dense", track_episodes=True,
                                      seed=3, observation_noise_std=so)
        e.reset(seed=3)
        e.rollout(K, policy="heuristic")
        outs.append(e._obs[:, :n].clone())
    assert torch.equal(outs[0], outs[1])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [130, 70_001])
def test_no_writes_outside_buffers(gpu, n):
    """The params, the trajectory buffers and the state arrays sit between guard bands filled with a byte pattern:
    nothing outside them is written, the params not at all, and nothing past column n or row k."""
    cap, k, guard = 16, 10, 4096
    rec, _ = _pair(n, "dense", True, None, (0.0, 0.05, 0.0), (0.0, 0.0, 0.05))
    pol = dx.MlpPolicy.from_torch(_net((64, 64), "tanh", 91), action_std=STD)
    bands = {}

    def banded(t):
        nbytes = t.numel() * t.element_size()
        big = torch.full((nbytes + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
        inner = big[guard:guard + nbytes].view(t.dtype).view(t.shape)
        inner.copy_(t)
        return big, inner

    big, pol.params = banded(pol.params)
    pol._struct.params = pol.params.data_ptr()
    bands["params"] = (big, pol.params, pol.params.clone())
    rec.enable_trajectory(cap, final_observation=True)
    for name, t in list(rec._traj.items()):
        big, rec._traj[name] = banded(t)
        bands["traj_" + name] = (big, rec._traj[name], None)
    for name in ("_obs", "_op64", "_step_count", "_episode", "_ep_return", "_ep_stats"):
        big, inner = banded(getattr(rec, name))
        setattr(rec, name, inner)
        bands[name] = (big, inner, None)
    rec._refresh_structs()
    pattern = {name: inner.clone() for name, (_, inner, _) in bands.items()}
    rec.rollout(k, policy=pol, loop_max_steps=4)
    torch.cuda.synchronize()
    for name, (big, inner, same) in bands.items():
        assert bool((big[:guard] == 0xA5).all()) and bool((big[-guard:] == 0xA5).all()), name
        if same is not None:
            assert torch.equal(inner, same), name
        if name.startswith("traj_"):
            assert torch.equal(inner[k:], pattern[name][k:]), (name, "rows past k")
            assert torch.equal(inner[..., n:], pattern[name][..., n:]), (name, "columns past n")
        elif name != "params":
            assert torch.equal(inner[..., n:], pattern[name][..., n:]), (name, "columns past n")
    assert int(rec.trajectory["finished"].sum()) > 0
