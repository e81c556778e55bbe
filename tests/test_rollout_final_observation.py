"""Terminal observations recorded by the fused rollout (``enable_trajectory(steps, final_observation=True)``,
``dexsim_rollout_record_final``).

On every row where ``finished`` is set, ``final_observation`` holds the observation that ended the episode, before the
auto-reset: the ``next_obs`` of that transition, which the ``obs`` row (the next episode's first observation) is not.
The yardstick is a same-step auto-reset twin built with ``final_observation=True``, stepped with the same actions and
noise: at every finished env the recorded terminal observation must equal the twin's ``info["final_observation"]`` bit
for bit, every other trajectory field must equal what the twin's ``step()`` returned, and entries of envs that did not
finish must not be written (the buffer is pre-filled with NaN)."""
import ctypes as C

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
         "_ep_return", "_ep_stats")
MAX_STEPS = 20
NAN = float("nan")


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


def _pair(n, reward="dense", respawn=True, loop=None, seed=5):
    """The recording env and its step() twin: same-step auto-reset with final_observation=True and the rollout's episode
    bound (rollout() defaults loop_max_steps to max_episode_steps, step() does not)."""
    common = dict(max_episode_steps=MAX_STEPS, reward_type=reward, track_episodes=True, seed=seed, respawn=respawn,
                  groups=_ranged_groups())
    rec = dx.BatchedManipulationEnv(n, "cuda", **common)
    twin = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True,
                                     loop_max_steps=MAX_STEPS if loop is None else loop, **common)
    rec.reset(seed=seed); twin.reset(seed=seed)
    return rec, twin


def _assert_rows_equal_twin(twin, tr, actions, dyn_noise, where):
    """Step the twin through the recorded rows: every field must be what its step() returns, the terminal observation
    what its info["final_observation"] holds at the finished envs, and the other entries still NaN."""
    for t in range(tr["obs"].shape[0]):
        extra = {} if dyn_noise is None else {"dyn_noise": dyn_noise[t]}
        obs, rew, term, trunc, info = twin.step(actions[t].contiguous(), **extra)
        fin = info["finished"]
        assert torch.equal(tr["obs"][t], obs), (where, t, "obs")
        assert torch.equal(tr["reward"][t], rew), (where, t, "reward")
        assert torch.equal(tr["terminated"][t], term), (where, t, "terminated")
        assert torch.equal(tr["truncated"][t], trunc), (where, t, "truncated")
        assert torch.equal(tr["finished"][t], fin), (where, t, "finished")
        fo = tr["final_observation"][t]
        assert torch.equal(fo[fin], info["final_observation"][fin]), (where, t, "final_observation")
        assert bool(fo[~fin].isnan().all()), (where, t, "final_observation of unfinished envs written")


def _assert_same_end(a, b):
    n = a.num_envs
    for k in STATE:
        assert torch.equal(getattr(a, k)[..., :n], getattr(b, k)[..., :n]), k
    assert torch.equal(a.counters, b.counters)
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0.0)


def _nan_fill(env):
    env._traj["final_observation"].fill_(NAN)


# (n, reward, respawn, loop bound, pre-drawn dynamics noise), the cases of the plain recording's twin test
EXTERNAL_CASES = [
    (100, "dense", True, None, False),
    (4096 + 77, "sparse", False, 6, True),
    (4096 + 77, "dense", True, 6, False),
    (70_001, "dense", False, None, True),
    (70_001, "sparse", True, 6, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,reward,respawn,loop,noise", EXTERNAL_CASES)
def test_external_actions_final_observation_equals_step_twin(gpu, n, reward, respawn, loop, noise):
    K = 12
    rec, twin = _pair(n, reward, respawn, loop)
    rec.enable_trajectory(2 * K, final_observation=True)
    gen = torch.Generator(device="cuda").manual_seed(n)
    finished = loop_ended = 0
    for call in range(2):                      # the second call starts at step_base K and still writes rows 0 .. K-1
        _nan_fill(rec)
        act = torch.rand(K, n, 15, device="cuda", generator=gen) * 2 - 1
        nz = torch.randn(K, n, 15, device="cuda", generator=gen) * 0.1 if noise else None
        rec.rollout(K, policy="external", actions=act, dyn_noise=nz, respawn=respawn, loop_max_steps=loop)
        tr = rec.trajectory
        assert "action" not in tr and tr["final_observation"].shape == (K, n, 45)
        _assert_rows_equal_twin(twin, tr, act, nz, call)
        finished += int(tr["finished"].sum())
        loop_ended += int((tr["finished"] & ~tr["terminated"] & ~tr["truncated"]).sum())
    _assert_same_end(rec, twin)
    assert finished > 0
    assert loop_ended > 0 or not respawn       # episodes the loop bound ended have their terminal observation too


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
def test_in_kernel_policy_final_observation_replays_on_step_twin(gpu, policy, n, noise):
    K = 15
    rec, twin = _pair(n, "dense", True, None)
    rec.enable_trajectory(K, final_observation=True)
    gen = torch.Generator(device="cuda").manual_seed(7)
    finished = 0
    for call in range(2):
        _nan_fill(rec)
        nz = torch.randn(K, n, 15, device="cuda", generator=gen) * 0.1 if noise else None
        rec.rollout(K, policy=policy, dyn_noise=nz)
        tr = rec.trajectory
        _assert_rows_equal_twin(twin, tr, tr["action"], nz, call)
        finished += int(tr["finished"].sum())
    _assert_same_end(rec, twin)
    assert finished > 0


@pytest.mark.gpu
@pytest.mark.parametrize("policy,n,respawn", [("random", 4096 + 77, False), ("heuristic", 70_001, True),
                                              ("learner", 5000, False)])
def test_final_observation_changes_nothing_else(gpu, policy, n, respawn):
    """Two envs run the same rollouts, one recording terminal observations too: state, counters, return sums, episode
    log, history, learner arrays and every field of the plain recording come out identical."""
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=MAX_STEPS, reward_type="dense", track_episodes=True, seed=9,
              groups=[CC.easy(), CC.medium(), CC.hard()])
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    for e in (a, b):
        e.reset(seed=9)
        e.enable_episode_log(60 * n)            # room for an episode per env-step: an overflow drops records in atomic order
        e.enable_history(60)
    a.enable_trajectory(25, final_observation=True)
    b.enable_trajectory(25)
    for k in (25, 20, 15):
        a.rollout(k, policy=policy, respawn=respawn)
        b.rollout(k, policy=policy, respawn=respawn)
        ta, tb = a.trajectory, b.trajectory
        assert "final_observation" not in tb and set(ta) == set(tb) | {"final_observation"}
        for name, v in tb.items():
            assert torch.equal(ta[name], v), (k, name)
    _assert_same_end(a, b)
    la, lb = a.read_episode_log(), b.read_episode_log()
    assert a.episode_log_overflow == 0 and len(la) > n and np.array_equal(la, lb)
    assert torch.equal(a._hist, b._hist)
    if policy == "learner":
        assert torch.equal(a._learner_mean, b._learner_mean) and torch.equal(a._learner_best, b._learner_best)


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["heuristic", "external"])
def test_one_episode_final_observation_is_the_ending_row(gpu, policy):
    """one_episode=True: the ending row's terminal observation equals its obs row and the env's final observation (it
    was not reset); every other entry, later rows included, stays NaN."""
    n, K = 4096 + 77, MAX_STEPS + 6
    rec, _ = _pair(n, "dense", False, None)
    rec.enable_trajectory(K, final_observation=True)
    _nan_fill(rec)
    act = torch.rand(K, n, 15, device="cuda") * 2 - 1
    rec.rollout(K, policy=policy, actions=act if policy == "external" else None, one_episode=True, respawn=False)
    tr, cols = rec.trajectory, torch.arange(n, device="cuda")
    fin = tr["finished"].to(torch.uint8)
    assert bool((fin.sum(0) == 1).all())                                    # every env ended exactly once
    end = fin.argmax(0)
    fo = tr["final_observation"]
    assert torch.equal(fo[end, cols], tr["obs"][end, cols])
    assert torch.equal(fo[end, cols], rec._obs[:, :n].t())
    others = torch.ones(K, n, dtype=torch.bool, device="cuda")
    others[end, cols] = False
    assert bool(fo[others].isnan().all())


@pytest.mark.gpu
def test_truncation_wave_at_full_size(gpu):
    """1,048,576 envs whose episodes all truncate on the same step, twice inside a recorded 8-step rollout: every env's
    terminal observation at both wave rows equals the twin's."""
    n, K, T = 1 << 20, 8, 3
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=T, reward_type="dense", track_episodes=True, seed=21, curriculum_config=CC.hard())
    rec = dx.BatchedManipulationEnv(n, "cuda", **kw)
    twin = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, final_observation=True, respawn=True,
                                     loop_max_steps=T, **kw)
    for e in (rec, twin):
        e._params.success_threshold = 6          # five fingers: no episode terminates, every one ends at the bound
        e.reset(seed=21)
    rec.enable_trajectory(K, final_observation=True)
    _nan_fill(rec)
    rec.rollout(K, policy="random")
    tr = rec.trajectory
    waves = [t for t in range(K) if bool(tr["finished"][t].all())]
    assert waves == [T - 1, 2 * T - 1] and int(tr["finished"].sum()) == 2 * n
    assert not bool(tr["final_observation"][waves].isnan().any())
    _assert_rows_equal_twin(twin, tr, tr["action"], None, "wave")
    _assert_same_end(rec, twin)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [130, 70_001])
def test_no_writes_outside_n_columns_and_k_rows(gpu, n):
    """The buffers sit between guard bands, filled with a byte pattern: nothing is written outside them, past column n,
    past row k, or into the terminal observation of an env that did not finish."""
    cap, k, guard = 16, 10, 4096
    rec, _ = _pair(n, "dense", True, None)
    rec.enable_trajectory(cap, final_observation=True)
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
        unfinished = rec._traj["finished"][:k, :n] != 1
        fo, fo_was = rec._traj["final_observation"], pattern["final_observation"]
        assert bool(unfinished.any())
        assert torch.equal(fo[:k, :, :n].transpose(1, 2)[unfinished], fo_was[:k, :, :n].transpose(1, 2)[unfinished])

    # a loop bound of 4 ends episodes inside the k rows
    rec.rollout(k, policy="heuristic", loop_max_steps=4)
    check(True)
    for name, t in rec._traj.items():                  # back to the pattern, then a call with the caller's actions
        t.copy_(pattern[name])
    rec.rollout(k, policy="external", actions=torch.rand(k, n, 15, device="cuda") * 2 - 1, loop_max_steps=4)
    check(False)
    with pytest.raises(_lib.DexsimError) as err:       # k beyond the capacity: refused before anything runs
        rec.rollout(cap + 1, policy="heuristic")
    assert err.value.code == -1002
    check(False)


def test_record_final_errors_before_any_device_call():
    """Each documented error of dexsim_rollout_record_final comes back before the device is touched (no GPU needed)."""
    L = _lib.lib()
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
    call = lambda k=5, kind=_lib.POLICY_RANDOM, traj=tr, fo=ptr: L.dexsim_rollout_record_final(
        C.byref(st), C.byref(p), ptr, None, k, kind, C.byref(rio), None if traj is None else C.byref(traj), fo, None)
    assert call() == 0
    assert call(fo=None) == -1001                           # DEXSIM_E_NULL: no terminal-observation buffer
    assert call(fo=ptr + 4) == -1003                        # DEXSIM_E_ALIGN: a misaligned one
    assert call(traj=None) == -1001                         # DEXSIM_E_NULL: no trajectory
    assert call(k=6) == -1002                               # DEXSIM_E_SIZE: more steps than rows
    assert call(k=0) == -1002
    for name in ("obs", "action", "reward", "terminated", "truncated", "finished"):
        setattr(tr, name, None)
        assert call() == -1001, name                        # DEXSIM_E_NULL: a missing array
        setattr(tr, name, ptr + 4)
        assert call() == -1003, name                        # DEXSIM_E_ALIGN: a misaligned array
        setattr(tr, name, ptr)
    assert call(kind=7) == -1004                            # DEXSIM_E_PARAM: no such policy
    rio.actions = ptr
    tr.action = None
    assert call(kind=_lib.POLICY_EXTERNAL) == 0             # the caller's actions need not be recorded
    assert call() == -1001
    tr.action = ptr
    try:
        _lib.set_rollout_impl("split")
        assert call() == -1004                              # DEXSIM_E_PARAM: the 5-lanes-per-env kernel forced
        assert call(fo=ptr + 4) == -1003                    # the buffer's own errors come first
        assert call(kind=_lib.POLICY_EXTERNAL) == 0         # not eligible for it: recorded by one thread per env
    finally:
        _lib.set_rollout_impl("auto")
    assert call() == 0
