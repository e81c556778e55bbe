"""Per-step trajectories recorded by the fused rollout (``enable_trajectory``, ``dexsim_rollout_record``).

Row t of a recorded call holds what the (t+1)-th step of the call would return from ``step()`` on a same-step auto-reset
env.  The yardstick is such a twin env, stepped with the same actions and noise: every recorded row must equal what the
twin's ``step()`` returned, bit for bit, and the two must end in the same state.  With an in-kernel policy the twin is fed
the recorded actions, so the recorded action is held to being exactly what ``step()`` needs."""
import ctypes as C

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
         "_ep_return", "_ep_stats")
MAX_STEPS = 20


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


def _ranged_groups():
    CC = dx.CurriculumConfig
    return [CC(object_size=s, object_size_range=(0.7 * s, 1.3 * s), object_mass=m, object_mass_range=(0.5 * m, 1.5 * m),
               friction_coefficient=f, friction_range=(0.6 * f, min(1.0, 1.4 * f)))
            for s, m, f in ((0.08, 0.05, 0.8), (0.05, 0.1, 0.5), (0.03, 0.2, 0.3))]


def _pair(n, reward="dense", respawn=True, loop=None, groups=None, seed=5, **kw):
    """The recording env and its step() twin: same-step auto-reset with the rollout's episode bound (rollout() defaults
    loop_max_steps to max_episode_steps, step() does not)."""
    common = dict(max_episode_steps=MAX_STEPS, reward_type=reward, track_episodes=True, seed=seed, respawn=respawn,
                  groups=groups if groups is not None else _ranged_groups(), **kw)
    rec = dx.BatchedManipulationEnv(n, "cuda", **common)
    twin = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, loop_max_steps=MAX_STEPS if loop is None else loop,
                                     **common)
    rec.reset(seed=seed); twin.reset(seed=seed)
    return rec, twin


def _assert_rows_equal_twin(twin, tr, actions, dyn_noise, where):
    """Step the twin through the recorded rows: every row must be what its step() returns."""
    for t in range(tr["obs"].shape[0]):
        extra = {} if dyn_noise is None else {"dyn_noise": dyn_noise[t]}
        obs, rew, term, trunc, info = twin.step(actions[t].contiguous(), **extra)
        assert torch.equal(tr["obs"][t], obs), (where, t, "obs")
        assert torch.equal(tr["reward"][t], rew), (where, t, "reward")
        assert torch.equal(tr["terminated"][t], term), (where, t, "terminated")
        assert torch.equal(tr["truncated"][t], trunc), (where, t, "truncated")
        assert torch.equal(tr["finished"][t], info["finished"]), (where, t, "finished")


def _assert_same_end(a, b):
    n = a.num_envs
    for k in STATE:
        assert torch.equal(getattr(a, k)[..., :n], getattr(b, k)[..., :n]), k
    assert torch.equal(a.counters, b.counters)
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0.0)


# (n, reward, respawn, loop bound, pre-drawn dynamics noise): ragged sizes, both rewards, both respawn modes, a loop bound
# below the episode limit, with and without noise; three groups with ranged size, mass and friction throughout
EXTERNAL_CASES = [
    (100, "dense", True, None, False),
    (4096 + 77, "sparse", False, 6, True),
    (4096 + 77, "dense", True, 6, False),
    (70_001, "dense", False, None, True),
    (70_001, "sparse", True, 6, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,reward,respawn,loop,noise", EXTERNAL_CASES)
def test_external_actions_rows_equal_step_twin(gpu, n, reward, respawn, loop, noise):
    K = 12
    rec, twin = _pair(n, reward, respawn, loop)
    rec.enable_trajectory(2 * K)
    gen = torch.Generator(device="cuda").manual_seed(n)
    finished = loop_ended = 0
    for call in range(2):                      # the second call starts at step_base K and still writes rows 0 .. K-1
        act = torch.rand(K, n, 15, device="cuda", generator=gen) * 2 - 1
        nz = torch.randn(K, n, 15, device="cuda", generator=gen) * 0.1 if noise else None
        rec.rollout(K, policy="external", actions=act, dyn_noise=nz, respawn=respawn, loop_max_steps=loop)
        tr = rec.trajectory
        assert "action" not in tr and tr["obs"].shape == (K, n, 45)
        _assert_rows_equal_twin(twin, tr, act, nz, call)
        finished += int(tr["finished"].sum())
        loop_ended += int((tr["finished"] & ~tr["terminated"] & ~tr["truncated"]).sum())
    _assert_same_end(rec, twin)
    assert finished > 0
    # the loop bound ends episodes -- max_episode_steps by default, one step before the truncation flag would -- and shows
    # only in `finished`.  Without respawn the object stays where a success left it and the next episodes terminate at
    # once, before any bound.
    assert loop_ended > 0 or not respawn


# in-kernel policies; sizes up to 8,192 envs take the 5-lanes-per-env kernel when not recording
POLICY_CASES = [
    ("random", 1000, False),
    ("heuristic", 8192, False),
    ("random", 4096 + 77, True),
    ("learner", 3000, True),
    ("heuristic", 70_001, True),
    ("learner", 70_001, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("policy,n,noise", POLICY_CASES)
def test_in_kernel_policy_rows_replay_on_step_twin(gpu, policy, n, noise):
    """The recorded actions (before dynamics noise), plus the same noise, reproduce every row and the final state."""
    K = 15
    rec, twin = _pair(n, "dense", True, None)
    rec.enable_trajectory(K)
    gen = torch.Generator(device="cuda").manual_seed(7)
    for call in range(2):
        nz = torch.randn(K, n, 15, device="cuda", generator=gen) * 0.1 if noise else None
        rec.rollout(K, policy=policy, dyn_noise=nz)
        tr = rec.trajectory
        assert tr["action"].shape == (K, n, 15) and float(tr["action"].abs().max()) <= 1.0
        _assert_rows_equal_twin(twin, tr, tr["action"], nz, call)
    _assert_same_end(rec, twin)
    assert int(rec.counters[:, _lib.CNT_EPISODES].sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("policy,n", [("random", 4096 + 77), ("heuristic", 70_001), ("learner", 5000)])
def test_recording_changes_nothing_else(gpu, policy, n):
    """Two envs run the same rollouts, one recording: state, counters, return sums, episode log, history and learner
    arrays come out identical."""
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=MAX_STEPS, reward_type="dense", track_episodes=True, seed=9,
              groups=[CC.easy(), CC.medium(), CC.hard()])
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    for e in (a, b):
        e.reset(seed=9)
        e.enable_episode_log(60 * n)            # room for an episode per env-step: an overflow drops records in atomic order
        e.enable_history(60)
    a.enable_trajectory(25)
    for k in (25, 20, 15):
        a.rollout(k, policy=policy, respawn=False)
        b.rollout(k, policy=policy, respawn=False)
    _assert_same_end(a, b)
    la, lb = a.read_episode_log(), b.read_episode_log()
    assert a.episode_log_overflow == 0 and len(la) > n and np.array_equal(la, lb)
    assert torch.equal(a._hist, b._hist)
    if policy == "learner":
        assert torch.equal(a._learner_mean, b._learner_mean) and torch.equal(a._learner_best, b._learner_best)


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["heuristic", "external"])
def test_one_episode_rows_stop_at_the_terminal_step(gpu, policy):
    """one_episode=True: the ending step's row holds the terminal observation and `finished`; later rows stay as the
    buffer was (NaN here)."""
    n, K = 4096 + 77, MAX_STEPS + 6
    rec, _ = _pair(n, "dense", False, None)
    rec.enable_trajectory(K)
    for name, buf in rec._traj.items():
        buf.fill_(float("nan") if buf.is_floating_point() else 7)
    act = torch.rand(K, n, 15, device="cuda") * 2 - 1
    rec.rollout(K, policy=policy, actions=act if policy == "external" else None, one_episode=True, respawn=False)
    tr, cols = rec.trajectory, torch.arange(n, device="cuda")
    fin = (rec._traj["finished"][:K, :n] == 1).to(torch.uint8)
    assert bool((fin.sum(0) == 1).all())                                    # every env ended exactly once
    end = fin.argmax(0)
    later = torch.arange(K, device="cuda")[:, None] > end[None, :]
    upto = ~later
    assert torch.equal(tr["obs"][end, cols], rec._obs[:, :n].t())        # the terminal observation: the env was not reset
    assert bool(tr["obs"][later].isnan().all()) and not bool(tr["obs"][upto].isnan().any())
    assert bool(tr["reward"][later].isnan().all()) and not bool(tr["reward"][upto].isnan().any())
    for name in ("terminated", "truncated", "finished"):
        raw = rec._traj[name][:K, :n]
        assert bool((raw[later] == 7).all()) and bool((raw[upto] <= 1).all()), name
    if policy != "external":
        assert bool(tr["action"][later].isnan().all()) and not bool(tr["action"][upto].isnan().any())
    assert int(rec.counters[:, _lib.CNT_EPISODES].sum()) == n


@pytest.mark.gpu
def test_truncation_wave_at_full_size(gpu):
    """1,048,576 envs whose episodes all truncate on the same step inside a recorded 8-step rollout: every row equals the
    twin's."""
    n, K, T = 1 << 20, 8, 3
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=T, reward_type="dense", track_episodes=True, seed=21, curriculum_config=CC.hard())
    rec = dx.BatchedManipulationEnv(n, "cuda", **kw)
    twin = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, respawn=True, loop_max_steps=T, **kw)
    for e in (rec, twin):
        e._params.success_threshold = 6          # five fingers: no episode terminates, every one ends at the bound
        e.reset(seed=21)
    rec.enable_trajectory(K)
    rec.rollout(K, policy="random")
    tr = rec.trajectory
    waves = [t for t in range(K) if bool(tr["finished"][t].all())]
    assert waves == [T - 1, 2 * T - 1] and int(tr["finished"].sum()) == 2 * n
    _assert_rows_equal_twin(twin, tr, tr["action"], None, "wave")
    _assert_same_end(rec, twin)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [130, 70_001])
def test_no_writes_outside_n_columns_and_k_rows(gpu, n):
    """The trajectory buffers sit between guard bands, filled with a byte pattern: nothing is written outside them, past
    column n or past row k, and the action buffer not at all when the caller holds the actions."""
    cap, k, guard = 16, 10, 4096
    rec, _ = _pair(n, "dense", True, None)
    rec.enable_trajectory(cap)
    bands = {}
    for name, t in rec._traj.items():
        nbytes = t.numel() * t.element_size()
        big = torch.full((nbytes + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
        rec._traj[name] = big[guard:guard + nbytes].view(t.dtype).view(t.shape)
        bands[name] = big
    pattern = {name: v.clone() for name, v in rec._traj.items()}

    def check(action_written):
        torch.cuda.synchronize()
        for name, big in bands.items():
            assert bool((big[:guard] == 0xA5).all()) and bool((big[-guard:] == 0xA5).all()), name
            now, was = rec._traj[name], pattern[name]
            assert torch.equal(now[k:], was[k:]), (name, "rows past k")
            assert torch.equal(now[..., n:], was[..., n:]), (name, "columns past n")
            if name != "action" or action_written:
                assert not torch.equal(now[:k, ..., :n], was[:k, ..., :n]), (name, "rows not written")
            else:
                assert torch.equal(now, was), name

    rec.rollout(k, policy="heuristic")
    check(True)
    for name, t in rec._traj.items():                  # back to the pattern, then a call with the caller's actions
        t.copy_(pattern[name])
    rec.rollout(k, policy="external", actions=torch.rand(k, n, 15, device="cuda") * 2 - 1)
    check(False)
    with pytest.raises(_lib.DexsimError) as err:       # k beyond the capacity: refused before anything runs
        rec.rollout(cap + 1, policy="heuristic")
    assert err.value.code == -1002
    check(False)


def test_record_errors_before_any_device_call():
    """Each documented error of dexsim_rollout_record comes back before the device is touched (no GPU needed), and
    dexsim_sizeof_trajectory matches the ctypes struct."""
    L = _lib.lib()
    assert L.dexsim_sizeof_trajectory() == C.sizeof(_lib.DexsimTrajectory) == 56
    buf = (C.c_char * 512)()
    ptr = (C.addressof(buf) + 15) & ~15                     # any non-NULL, 16-byte aligned address: never dereferenced
    st = _lib.DexsimState()
    st.n, st.ld = 0, 32                                     # n == 0: a valid call returns before touching the device
    for name, _ in _lib.DexsimState._fields_[2:]:
        setattr(st, name, ptr)
    p = _lib.DexsimParams()
    p.reward_type, p.success_threshold, p.num_groups, p.max_episode_steps = 1, 3, 1, 200
    rio = _lib.DexsimRolloutIO()
    rio.flags = _lib.ROLLOUT_NO_DYN_NOISE                   # eligible for the 5-lanes-per-env kernel with an in-kernel policy
    tr = _lib.DexsimTrajectory(ptr, ptr, ptr, ptr, ptr, ptr, 5)
    call = lambda k=5, kind=_lib.POLICY_RANDOM, traj=tr: L.dexsim_rollout_record(
        C.byref(st), C.byref(p), ptr, None, k, kind, C.byref(rio), None if traj is None else C.byref(traj), None)
    assert call() == 0
    assert call(traj=None) == -1001                         # DEXSIM_E_NULL: no trajectory
    assert call(k=6) == -1002                               # DEXSIM_E_SIZE: more steps than rows
    for name in ("obs", "action", "reward", "terminated", "truncated", "finished"):
        setattr(tr, name, None)
        assert call() == -1001, name                        # DEXSIM_E_NULL: a missing array
        setattr(tr, name, ptr + 4)
        assert call() == -1003, name                        # DEXSIM_E_ALIGN: a misaligned array
        setattr(tr, name, ptr)
    rio.actions = ptr
    tr.action = None
    assert call(kind=_lib.POLICY_EXTERNAL) == 0             # the caller's actions need not be recorded
    assert call() == -1001
    tr.action = ptr
    try:
        _lib.set_rollout_impl("split")
        assert call() == -1004                              # DEXSIM_E_PARAM: the 5-lanes-per-env kernel forced
        assert call(kind=_lib.POLICY_EXTERNAL) == 0         # not eligible for it: recorded by one thread per env
    finally:
        _lib.set_rollout_impl("auto")
    assert call() == 0
    env = dx.BatchedManipulationEnv.__new__(dx.BatchedManipulationEnv)
    env._traj = None
    with pytest.raises(RuntimeError):
        env.trajectory
