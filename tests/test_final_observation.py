"""Terminal observations of auto-reset stepping (``final_observation=True``, ``dexsim_step_final``).

An auto-reset env resets a finished episode in the same step, so the observation that ended the episode is gone by the
time step() returns.  With ``final_observation=True`` the step runs without the reset and a second pass resets the
finished envs after copying that observation into ``info["final_observation"]``.  These tests hold the two-pass step to
two yardsticks: a twin env without auto-reset that is reset by hand after every step (the final observation is what
that twin returns), and the default in-kernel auto-reset (everything else is what it produces)."""
import ctypes as C

import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
         "_ep_return", "_ep_stats")


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
# an episode bound below max_episode_steps; per-group and env-level in-kernel noise, and pre-drawn noise
CASES = [
    (1000, False, True, 0, "group"),
    (4096 + 77, True, False, 3, "predrawn"),
    (224 * 19 + 3, False, False, 3, "none"),
    (4096 + 77, True, True, 0, "env"),
]
KERNELS = ["register", "tma", "tma_wide"]
MAX_STEPS = 20


def _kwargs(n, track, respawn, loop, noise, seed=11):
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=MAX_STEPS, reward_type="dense", respawn=respawn, loop_max_steps=loop, track_episodes=track,
              seed=seed, groups=[CC.easy(), CC.medium(), CC.hard()], reward_components=(n % 2 == 1))
    if noise == "group":
        kw.update(group_sigma_obs=[0.02, 0.0, 0.05], group_sigma_dyn=[0.0, 0.1, 0.05])
    elif noise == "env":
        kw.update(observation_noise_std=0.03, dynamics_noise_std=0.05)
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


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("n,track,respawn,loop,noise", CASES)
def test_final_observation_equals_a_twin_without_auto_reset(gpu, step_kernel, kernel, n, track, respawn, loop, noise):
    """A steps with final observations; B is the same env without auto-reset, reset by hand where A finished."""
    step_kernel(kernel)
    kw = _kwargs(n, track, respawn, loop, noise)
    a = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, **kw)
    b = dx.BatchedManipulationEnv(n, "cuda", auto_reset=False, **kw)
    _no_success_when_bounded(loop, a, b)
    a.reset(seed=11); b.reset(seed=11)
    gen = torch.Generator(device="cuda").manual_seed(3)
    finished_total = loop_ended = 0
    for t in range(3 * MAX_STEPS):
        act, extra = _inputs(gen, n, noise)
        oa, ra, ta, ua, ia = a.step(act, **extra)
        ob, rb, tb, ub, _ = b.step(act, **extra)
        assert torch.equal(ra, rb) and torch.equal(ta, tb) and torch.equal(ua, ub), t
        done = _done(b)
        assert torch.equal(ia["finished"], done), t
        fo = ia["final_observation"]
        assert torch.equal(fo[done], ob[done]), t                 # bit for bit, B's noisy observation when noise is on
        finished_total += int(done.sum())
        loop_ended += int((done & ~tb & ~ub).sum())
        b.reset(options={"mask": done})
        for k in ("_obs", "_op64", "_step_count", "_episode"):
            assert torch.equal(getattr(a, k)[..., :n], getattr(b, k)[..., :n]), (t, k)
    assert finished_total > n                                     # several reset waves went through
    assert (loop_ended > 0) == (loop > 0)                         # the loop bound did end episodes
    assert int(a.counters[:, _lib.CNT_EPISODES].sum()) == finished_total


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("n,track,respawn,loop,noise", CASES)
def test_final_observation_leaves_auto_reset_results_unchanged(gpu, step_kernel, kernel, n, track, respawn, loop, noise):
    """A (two passes) against C (the in-kernel auto-reset): every state array, output, noisy observation and counter."""
    step_kernel(kernel)
    kw = _kwargs(n, track, respawn, loop, noise)
    a = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, **kw)
    c = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, **kw)
    _no_success_when_bounded(loop, a, c)
    a.reset(seed=11); c.reset(seed=11)
    gen = torch.Generator(device="cuda").manual_seed(5)
    for t in range(3 * MAX_STEPS):
        act, extra = _inputs(gen, n, noise)
        out_a, out_c = a.step(act, **extra), c.step(act, **extra)
        for x, y in zip(out_a[:4], out_c[:4]):
            assert torch.equal(x, y), t
        ia, ic = out_a[4], out_c[4]
        assert torch.equal(ia["finished"], ic["finished"]) and torch.equal(ia["num_contacts"], ic["num_contacts"]), t
        if "reward_components" in ic:
            for k in ic["reward_components"]:
                assert torch.equal(ia["reward_components"][k], ic["reward_components"][k]), (t, k)
        for k in STATE:
            x, y = getattr(a, k), getattr(c, k)
            assert (x is None and y is None) or torch.equal(x[..., :n], y[..., :n]), (t, k)
        if noise != "none":
            assert torch.equal(a._noisy_obs[:, :n], c._noisy_obs[:, :n]), t
        assert torch.equal(a.counters, c.counters), t
    torch.testing.assert_close(a.ret_sums, c.ret_sums, rtol=1e-9, atol=0.0)
    assert int(c.counters[:, _lib.CNT_EPISODES].sum()) > n
    if track:
        assert float(c.ret_sums.abs().sum()) > 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["register", "tma"])
def test_final_obs_written_only_for_finished_envs(gpu, step_kernel, kernel):
    """dexsim_step_final through ctypes, final_obs between NaN guard bands and pre-filled with NaN: only the columns of
    envs that finished are ever written."""
    step_kernel(kernel)
    n, guard = 4096 + 77, 8192
    env = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, **_kwargs(n, True, True, 0, "none"))
    env.reset(seed=2)
    ld = env.ld
    big = torch.full((45 * ld + 2 * guard,), float("nan"), device="cuda")
    fo = big[guard:guard + 45 * ld].view(45, ld)
    L = _lib.lib()
    gen = torch.Generator(device="cuda").manual_seed(9)
    ever = torch.zeros(n, dtype=torch.bool, device="cuda")
    for t in range(MAX_STEPS // 2):                                   # some envs finish, not all
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
        env._io.action, env._io.action_layout = act.data_ptr(), 1
        rc = L.dexsim_step_final(env._state_ref, env._params_ref, env._groups_ptr, env._goe_ptr, env._io_ref, fo.data_ptr(),
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        ever |= env._finished[:n].bool()
        torch.cuda.synchronize()
        assert bool(torch.isnan(big[:guard]).all()) and bool(torch.isnan(big[guard + 45 * ld:]).all()), t
        assert bool(torch.isnan(fo[:, :n][:, ~ever]).all()), t
        assert not bool(torch.isnan(fo[:, :n][:, ever]).any()), t
        assert bool(torch.isnan(fo[:, n:]).all()), t                  # padding columns
    assert 0 < int(ever.sum()) < n


@pytest.mark.gpu
def test_reset_wave_at_full_size(gpu):
    """1,048,576 envs whose episodes all truncate on the same step: every column of final_observation is written and
    equals the twin without auto-reset."""
    n, T = 1 << 20, 6
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=T, reward_type="dense", respawn=True, track_episodes=False, seed=21, curriculum_config=CC.hard())
    a = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, **kw)
    b = dx.BatchedManipulationEnv(n, "cuda", auto_reset=False, **kw)
    for e in (a, b):
        e._params.success_threshold = 6          # five fingers: no episode can terminate, every one truncates at once
        e.reset(seed=21)
    gen = torch.Generator(device="cuda").manual_seed(1)
    a._final_obs.fill_(float("nan"))
    waves = 0
    for t in range(2 * T + 3):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
        _, _, _, _, ia = a.step(act)
        ob, _, _, _, _ = b.step(act)
        done = _done(b)
        fin = ia["finished"]
        assert torch.equal(fin, done), t
        assert int(fin.sum()) in (0, n), t                              # all at once or none
        if bool(fin[0]):
            waves += 1
            assert not bool(torch.isnan(ia["final_observation"]).any()), t
            assert torch.equal(ia["final_observation"], ob), t
            a._final_obs.fill_(float("nan"))
            b.reset(options={"mask": done})
        assert torch.equal(a._obs[:, :n], b._obs[:, :n]) and torch.equal(a._episode[:n], b._episode[:n]), t
    assert waves == 2


@pytest.mark.gpu
def test_capture_step_replays_final_observations(gpu):
    n, steps = 16384, 8
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=15, reward_type="dense", curriculum_config=CC.easy(), auto_reset=True, respawn=True,
              loop_max_steps=15, track_episodes=True, seed=7, final_observation=True)
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
        assert torch.equal(a._final_obs, b._final_obs), it
        assert torch.equal(oa[4]["final_observation"], ob[4]["final_observation"]), it
    assert torch.equal(a._obs, b._obs) and torch.equal(a.counters, b.counters)
    assert finished > n


def test_argument_errors_before_any_device_call():
    """Each documented error of dexsim_step_final comes back before the device is touched (no GPU needed), and the
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
    call = lambda fo=ptr, pp=p, ii=io: L.dexsim_step_final(C.byref(st), C.byref(pp), ptr, None, C.byref(ii), fo, None)
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
    assert call(fo=None) == -1001                           # DEXSIM_E_NULL: no final_obs
    io.finished = None
    assert call() == -1001                                  # DEXSIM_E_NULL: no finished flags
    io.finished = ptr
    assert call() == 0
    with pytest.raises(ValueError):
        dx.BatchedManipulationEnv(4, final_observation=True)                       # needs auto_reset=True
    with pytest.raises(NotImplementedError):
        dx.BatchedManipulationEnv(1, auto_reset=True, final_observation=True)      # the drop-in single-env path
