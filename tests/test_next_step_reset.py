"""Next-step auto-reset (``autoreset_mode="next_step"``, ``dexsim_step_next_reset``).

The step that ends an episode returns its terminal observation and flags ``finished``; the env's next step ignores its
action and resets it, returning the first observation of the new episode, reward 0 and both flags False.  These tests
hold the mode to three yardsticks: a twin env without auto-reset that is reset by hand where the next-step env has a
pending reset (every output and state array, every step), the same-step auto-reset (counters, return sums, states) and
``final_observation=True`` (terminal and first observations)."""
import ctypes as C

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
         "_ep_return", "_ep_stats")
NEXT = dict(auto_reset=True, autoreset_mode="next_step")


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


@pytest.fixture
def step_kernel():
    """Pin the step to the register-resident kernel, the pipeline's narrow tile or its wide tile; restored afterwards."""
    def choose(impl):
        _lib.set_step_impl("tma" if impl == "tma_wide" else impl)
        _lib.set_step_tile("wide" if impl == "tma_wide" else "narrow" if impl == "tma" else "auto")
    yield choose
    _lib.set_step_impl("auto")
    _lib.set_step_tile("auto")


# (n, full tracking, respawn, loop_max_steps, noise): ragged sizes; counts-only and full tracking; both respawn modes;
# an episode bound below max_episode_steps; per-group and env-level in-kernel noise, pre-drawn noise and none
CASES = [
    (1000, False, True, 0, "group"),
    (4096 + 77, True, False, 3, "predrawn"),
    (224 * 19 + 3, False, False, 3, "none"),
    (4096 + 77, True, True, 0, "env"),
]
KERNELS = ["register", "tma", "tma_wide"]
MAX_STEPS = 20
GROUP_SIGMA_OBS = [0.02, 0.0, 0.05]
ENV_SIGMA_OBS = 0.03


def _kwargs(n, track, respawn, loop, noise, seed=11):
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=MAX_STEPS, reward_type="dense", respawn=respawn, loop_max_steps=loop, track_episodes=track,
              seed=seed, groups=[CC.easy(), CC.medium(), CC.hard()], reward_components=(n % 2 == 1))
    if noise == "group":
        kw.update(group_sigma_obs=GROUP_SIGMA_OBS, group_sigma_dyn=[0.0, 0.1, 0.05])
    elif noise == "env":
        kw.update(observation_noise_std=ENV_SIGMA_OBS, dynamics_noise_std=0.05)
    return kw


def _inputs(gen, n, noise):
    act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
    if noise != "predrawn":
        return act, {}
    return act, dict(obs_noise=torch.randn(n, 45, device="cuda", generator=gen) * 0.03,
                     dyn_noise=torch.randn(n, 15, device="cuda", generator=gen) * 0.05)


def _no_success_when_bounded(loop, *envs):
    """With a loop bound, no episode can succeed (five fingers, threshold six): the bound, not an early success, ends them."""
    if loop:
        for e in envs:
            e._params.success_threshold = 6


def _done(env):
    n = env.num_envs
    d = env._terminated[:n].bool() | env._truncated[:n].bool()
    if env.loop_max_steps > 0:
        d |= env._step_count[:n] >= env.loop_max_steps
    return d


def _contacts(env):
    n = env.num_envs
    return sum(((env._cmask[:n] >> f) & 1) for f in range(5)).to(torch.uint8)


def _reset_obs(env, noise, extra):
    """Batch-first observation of `env`'s current state with the observation noise a next-step reset draws for it: the
    pre-drawn tensor, or Philox normals keyed by the state's (episode, step count) -- dexsim_fill_normal's numbers."""
    n, ld = env.num_envs, env.ld
    obs = env._obs[:, :n]
    if noise == "none":
        return obs.t().clone()
    if noise == "predrawn":
        return (obs.t() + extra["obs_noise"]).contiguous()
    sigmas = [ENV_SIGMA_OBS] if noise == "env" else GROUP_SIGMA_OBS
    group = torch.arange(n, device="cuda") % len(sigmas)
    z = torch.zeros(45, n, device="cuda")
    buf = torch.zeros(45, ld, device="cuda")
    for g, s in enumerate(sigmas):
        _lib.check(env._lib.dexsim_fill_normal(env._state_ref, env._params_ref, _lib.RNG_STREAM_OBS, 45, C.c_float(s),
                                               buf.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   "dexsim_fill_normal")
        z[:, group == g] = buf[:, :n][:, group == g]
    return (obs + z).t().contiguous()


def _assert_states_equal(a, b, where):
    n = a.num_envs
    for k in STATE:
        x, y = getattr(a, k), getattr(b, k)
        assert (x is None and y is None) or torch.equal(x[..., :n], y[..., :n]), (where, k)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("n,track,respawn,loop,noise", CASES)
def test_next_step_equals_a_twin_without_auto_reset(gpu, step_kernel, kernel, n, track, respawn, loop, noise):
    """A resets on the step after an episode ends; B is the same env without auto-reset, reset by hand before the step
    where A has a pending reset, its pending columns restored after the step (A did not step them)."""
    step_kernel(kernel)
    kw = _kwargs(n, track, respawn, loop, noise)
    a = dx.BatchedManipulationEnv(n, "cuda", **NEXT, **kw)
    b = dx.BatchedManipulationEnv(n, "cuda", auto_reset=False, **kw)
    _no_success_when_bounded(loop, a, b)
    a.reset(seed=11); b.reset(seed=11)
    gen = torch.Generator(device="cuda").manual_seed(3)
    group = torch.arange(n, device="cuda") % 3
    eps, succ, steps = (torch.zeros(3, dtype=torch.float64, device="cuda") for _ in range(3))
    pending = torch.zeros(n, dtype=torch.bool, device="cuda")
    resets = loop_ended = 0
    for t in range(3 * MAX_STEPS):
        act, extra = _inputs(gen, n, noise)
        if bool(pending.any()):
            b.reset(options={"mask": pending})
        snap = {k: getattr(b, k).clone() for k in STATE if getattr(b, k) is not None}
        want_reset_obs, want_nc = _reset_obs(b, noise, extra), _contacts(b)
        oa, ra, ta, ua, ia = a.step(act, **extra)
        ob, rb, tb, ub, ib = b.step(act, **extra)
        keep = ~pending
        # envs A stepped: B's step outputs, bit for bit (the noisy observation when noise is on)
        assert torch.equal(oa[keep], ob[keep]), t
        assert torch.equal(ra[keep], rb[keep]) and torch.equal(ta[keep], tb[keep]) and torch.equal(ua[keep], ub[keep]), t
        assert torch.equal(ia["num_contacts"][keep], ib["num_contacts"][keep]), t
        # envs A reset: B's reset outputs
        assert torch.equal(oa[pending], want_reset_obs[pending]), t
        assert not bool(ra[pending].any()) and not bool(ta[pending].any()) and not bool(ua[pending].any()), t
        assert torch.equal(ia["num_contacts"][pending], want_nc[pending]), t
        if "reward_components" in ia:
            for k, v in ia["reward_components"].items():
                assert torch.equal(v[keep], ib["reward_components"][k][keep]) and not bool(v[pending].any()), (t, k)
        done = _done(b) & keep
        assert torch.equal(ia["finished"], done), t
        eps += torch.bincount(group[done], minlength=3)
        succ += torch.bincount(group[done & tb], minlength=3)
        steps += torch.bincount(group[done], weights=b._step_count[:n][done].double(), minlength=3)
        loop_ended += int((done & ~tb & ~ub).sum())
        resets += int(pending.sum())
        for k, v in snap.items():
            getattr(b, k)[..., :n][..., pending] = v[..., :n][..., pending]
        _assert_states_equal(a, b, t)
        pending = done
    assert resets > n                                             # several reset waves went through
    assert (loop_ended > 0) == (loop > 0)                         # the loop bound did end episodes
    assert torch.equal(a.counters[:, _lib.CNT_EPISODES].double(), eps)
    assert torch.equal(a.counters[:, _lib.CNT_SUCCESSES].double(), succ)
    assert torch.equal(a.counters[:, _lib.CNT_SUM_STEPS].double(), steps)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("track", [False, True])
def test_truncation_waves_match_same_step_and_final_observation(gpu, step_kernel, kernel, track):
    """Every episode ends at the loop bound.  A (next step) against C (same-step auto-reset) and F (final_observation),
    which do not step while A runs its reset step: counters, return sums and states equal C's; A's observation at the
    end of an episode is F's final observation, and at the reset step what F and C returned when they reset."""
    step_kernel(kernel)
    n, loop = 4096 + 77, 5
    kw = _kwargs(n, track, True, loop, "none")
    a = dx.BatchedManipulationEnv(n, "cuda", **NEXT, **kw)
    c = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, **kw)
    f = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, **kw)
    _no_success_when_bounded(loop, a, c, f)
    for e in (a, c, f):
        e.reset(seed=11)
    gen = torch.Generator(device="cuda").manual_seed(5)
    waves, reset_obs = 0, None
    for t in range(4 * (loop + 1) + 2):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
        oa, ra, ta, ua, ia = a.step(act)
        fin = ia["finished"]
        if reset_obs is not None:                                 # A's reset step: C and F skip this action
            assert torch.equal(oa, reset_obs), t
            assert not bool(ra.any()) and not bool(ta.any()) and not bool(ua.any()) and not bool(fin.any()), t
            reset_obs = None
            _assert_states_equal(a, c, t)
            continue
        oc, rc, tc, uc, ic = c.step(act)
        of, _, _, _, i_f = f.step(act)
        assert torch.equal(ra, rc) and torch.equal(ta, tc) and torch.equal(ua, uc), t
        assert torch.equal(fin, ic["finished"]) and torch.equal(fin, i_f["finished"]), t
        if bool(fin.any()):
            assert bool(fin.all()), t
            waves += 1
            assert torch.equal(oa, i_f["final_observation"]), t
            assert torch.equal(of, oc), t
            reset_obs = of.clone()
        else:
            assert torch.equal(oa, oc), t
            _assert_states_equal(a, c, t)
        assert torch.equal(a.counters, c.counters), t
    assert waves >= 3
    torch.testing.assert_close(a.ret_sums, c.ret_sums, rtol=1e-9, atol=0.0)
    assert int(a.counters[:, _lib.CNT_EPISODES].sum()) == waves * n
    if track:
        assert float(a.ret_sums.abs().sum()) > 0.0


@pytest.mark.gpu
def test_reset_wave_at_full_size(gpu):
    """1,048,576 envs whose episodes all truncate on the same step: every env flags finished together, and every env
    resets on the step after, returning the twin's reset observation."""
    n, T = 1 << 20, 6
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=T, reward_type="dense", respawn=True, track_episodes=False, seed=21, curriculum_config=CC.hard())
    a = dx.BatchedManipulationEnv(n, "cuda", **NEXT, **kw)
    b = dx.BatchedManipulationEnv(n, "cuda", auto_reset=False, **kw)
    for e in (a, b):
        e._params.success_threshold = 6          # five fingers: no episode can terminate, every one truncates at once
        e.reset(seed=21)
    gen = torch.Generator(device="cuda").manual_seed(1)
    all_envs = torch.ones(n, dtype=torch.bool, device="cuda")
    waves, pending = 0, False
    for t in range(2 * (T + 2)):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
        if pending:
            b.reset(options={"mask": all_envs})
            oa, ra, ta, ua, ia = a.step(act)
            assert torch.equal(oa, b._obs[:, :n].t()), t
            assert not bool(ra.any() | ta.any() | ua.any() | ia["finished"].any()), t
            pending = False
        else:
            oa, ra, ta, ua, ia = a.step(act)
            ob, rb, tb, ub, _ = b.step(act)
            done = _done(b)
            fin = ia["finished"]
            assert torch.equal(fin, done), t
            assert int(fin.sum()) in (0, n), t                              # all at once or none
            assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(ta, tb) and torch.equal(ua, ub), t
            if bool(fin[0]):
                waves += 1
                pending = True
        _assert_states_equal(a, b, t)
    assert waves == 2
    assert int(a.counters[:, _lib.CNT_EPISODES].sum()) == 2 * n


@pytest.mark.gpu
def test_capture_step_replays_next_step_resets(gpu):
    n, steps = 16384, 8
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=15, reward_type="dense", curriculum_config=CC.easy(), respawn=True, loop_max_steps=15,
              track_episodes=True, seed=7, **NEXT)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    a.reset(seed=7); b.reset(seed=7)
    buf = torch.rand(steps, n, 15, device="cuda") * 2 - 1
    replay = b.capture_step(buf, steps=steps)
    finished = 0
    for it in range(6):
        buf.copy_(torch.rand(steps, n, 15, device="cuda") * 2 - 1)
        for k in range(steps):
            oa = a.step(buf[k])
            finished += int(oa[4]["finished"].sum())
        ob = replay()
        for x, y in zip(oa[:4], ob[:4]):
            assert torch.equal(x, y), it
        assert torch.equal(oa[4]["finished"], ob[4]["finished"]), it
        _assert_states_equal(a, b, it)
    assert torch.equal(a.counters, b.counters)
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0.0)
    assert finished > n


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["register", "tma"])
def test_resume_with_pending_resets(gpu, step_kernel, kernel):
    """state_dict() taken right after a step that ended episodes (their resets pending), loaded into a fresh env:
    both continue bit for bit."""
    step_kernel(kernel)
    n = 4096 + 77
    kw = dict(_kwargs(n, True, False, 0, "env"), **NEXT)
    a = dx.BatchedManipulationEnv(n, "cuda", **kw)
    a.reset(seed=11)
    gen = torch.Generator(device="cuda").manual_seed(8)
    for t in range(3 * MAX_STEPS):
        _, _, _, _, ia = a.step(torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1)
        if bool(ia["finished"].any()):
            break
    assert bool(ia["finished"].any())
    b = dx.BatchedManipulationEnv(n, "cuda", **kw)
    b.load_state_dict(a.state_dict())
    for t in range(2 * MAX_STEPS):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
        oa, ob = a.step(act), b.step(act)
        for x, y in zip(oa[:4], ob[:4]):
            assert torch.equal(x, y), t
        assert torch.equal(oa[4]["finished"], ob[4]["finished"]), t
        _assert_states_equal(a, b, t)
        assert torch.equal(a.counters, b.counters), t
    assert int(a.counters[:, _lib.CNT_EPISODES].sum()) > n


def test_argument_errors_before_any_device_call():
    """Each documented error of dexsim_step_next_reset comes back before the device is touched (no GPU needed), and the
    Python face rejects the combinations it does not support."""
    L = _lib.lib()
    buf = (C.c_char * 256)()
    ptr = (C.addressof(buf) + 15) & ~15                     # any non-NULL, 16-byte aligned address: never dereferenced
    st = _lib.DexsimState()
    st.n, st.ld = 0, 32                                     # n == 0: a valid call returns before touching the device
    for name, _ in _lib.DexsimState._fields_[2:12]:
        setattr(st, name, ptr)
    p = _lib.DexsimParams()
    p.reward_type, p.success_threshold, p.num_groups, p.max_episode_steps, p.auto_reset = 1, 3, 1, 200, 1
    io = _lib.DexsimStepIO()
    io.action = io.reward = io.terminated = io.truncated = io.num_contacts = io.finished = ptr
    call = lambda: L.dexsim_step_next_reset(C.byref(st), C.byref(p), ptr, None, C.byref(io), None)
    assert call() == 0
    p.auto_reset = 0
    assert call() == -1004                                  # DEXSIM_E_PARAM: no auto-reset
    p.auto_reset = 1
    io.host_static_rows = ptr
    assert call() == -1004                                  # DEXSIM_E_PARAM: host mirror of the observation
    io.host_static_rows = None
    io.flags = _lib.STEP_HOST_ALL_ROWS
    assert call() == -1004                                  # DEXSIM_E_PARAM: zero-copy host step
    io.flags = 0
    io.finished = None
    assert call() == -1001                                  # DEXSIM_E_NULL: no finished flags
    io.finished = ptr
    assert call() == 0
    BME = dx.BatchedManipulationEnv
    with pytest.raises(ValueError):
        BME(4, autoreset_mode="next_step")                                             # needs auto_reset=True
    with pytest.raises(ValueError):
        BME(4, auto_reset=True, final_observation=True, autoreset_mode="next_step")    # returns terminal obs itself
    with pytest.raises(ValueError):
        BME(4, auto_reset=True, autoreset_mode="next")                                 # unknown mode
    with pytest.raises(NotImplementedError):
        BME(1, auto_reset=True, autoreset_mode="next_step")                            # the drop-in single-env path
    env = BME.__new__(BME)                                  # the method checks come first: no device state needed
    env._next_step = True
    with pytest.raises(NotImplementedError):
        env.step_host(np.zeros((4, 15), np.float32))
    with pytest.raises(NotImplementedError):
        env.rollout(1)
