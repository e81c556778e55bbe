"""Generalized advantage estimation on the device (``dexsim_gae``, ``env.gae``).

``gae_reference`` restates the kernel's float32 arithmetic (include/dexsim.h) in NumPy, one rounding per operation; the
kernel must equal it bit for bit on real recordings.  The reference itself is checked against a float64 textbook
computation that walks each episode on its own, on hand-built rows covering termination, truncation, the loop bound,
terminated && truncated and back-to-back one-step episodes."""
import ctypes as C

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

U = 2.0 ** -24


def gae_reference(reward, terminated, finished, values, final_values, gamma, lam):
    """float32 GAE of include/dexsim.h: reward / terminated / finished / final_values [k, n], values [k+1, n]."""
    f32 = np.float32
    reward, values, final_values = (np.asarray(a, f32) for a in (reward, values, final_values))
    term, fin = np.asarray(terminated, bool), np.asarray(finished, bool)
    k, n = reward.shape
    g = f32(gamma)
    gl = f32(g * f32(lam))
    adv, ret = np.empty((k, n), f32), np.empty((k, n), f32)
    a_next = np.zeros(n, f32)
    with np.errstate(all="ignore"):
        for t in range(k - 1, -1, -1):
            nv = np.where(fin[t], np.where(term[t], f32(0.0), final_values[t]), values[t + 1])
            delta = (reward[t] + g * nv) - values[t]
            a = np.where(fin[t], delta, delta + gl * a_next)
            adv[t], ret[t] = a, a + values[t]
            a_next = a
    return adv, ret


def gae_textbook(reward, terminated, finished, values, final_values, gamma, lam):
    """float64, per env and per episode: A_t = sum_l (gamma lam)^l delta_{t+l} over the rest of the episode, each
    episode's last delta bootstrapping from 0 (terminated), final_values (finished otherwise) or values[k] (cut by the
    end of the recording).  Also the discounted return sum_l gamma^l r_{t+l} + gamma^L bootstrap."""
    r, v, fv = (np.asarray(a, np.float64) for a in (reward, values, final_values))
    term, fin = np.asarray(terminated, bool), np.asarray(finished, bool)
    k, n = r.shape
    adv, disc = np.zeros((k, n)), np.zeros((k, n))
    for i in range(n):
        start = 0
        for end in range(k):
            if not (fin[end, i] or end == k - 1):
                continue
            boot = 0.0 if (fin[end, i] and term[end, i]) else fv[end, i] if fin[end, i] else v[k, i]
            for t in range(start, end + 1):
                a = d = 0.0
                for l, s in enumerate(range(t, end + 1)):
                    nxt = boot if s == end else v[s + 1, i]
                    a += (gamma * lam) ** l * (r[s, i] + gamma * nxt - v[s, i])
                    d += gamma ** l * r[s, i]
                adv[t, i] = a
                disc[t, i] = d + gamma ** (end - t + 1) * boot
            start = end + 1
    return adv, disc


def _case(k, n, seed, p_fin=0.2, p_term=0.5):
    rng = np.random.default_rng(seed)
    reward = rng.normal(0.0, 1.0, (k, n)).astype(np.float32)
    values = rng.normal(0.0, 5.0, (k + 1, n)).astype(np.float32)
    final_values = rng.normal(0.0, 5.0, (k, n)).astype(np.float32)
    finished = rng.random((k, n)) < p_fin
    terminated = finished & (rng.random((k, n)) < p_term)
    return reward, terminated, finished, values, final_values


def _hand_cases():
    """Columns: (0) a termination mid-way, (1) a truncation, (2) the loop bound (finished only), (3) terminated and
    truncated on the same row, (4) one-step episodes back to back, (5) nothing finished, (6) finished on the last row."""
    k, n = 6, 7
    reward, terminated, finished, values, final_values = _case(k, n, 1)
    terminated[:] = False
    finished[:] = False
    finished[2, 0] = terminated[2, 0] = True
    finished[3, 1] = True                           # truncated: bootstraps from final_values
    finished[1, 2] = True                           # the loop bound: bootstraps from final_values
    finished[4, 3] = terminated[4, 3] = True        # terminated && truncated: terminated wins
    finished[:, 4] = True
    terminated[::2, 4] = True
    finished[k - 1, 6] = True
    return reward, terminated, finished, values, final_values


def _tol(reward, values, final_values):
    """|float32 recursion - float64| bound: each of the at most k steps of the recursion adds a few roundings of
    quantities bounded by the largest |reward|, |value| and |A|."""
    k = reward.shape[0]
    scale = float(np.abs(reward).max() + 3 * max(np.abs(values).max(), np.abs(final_values).max()))
    return 8 * k * k * U * scale


# ---- CPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (0.9, 0.0), (1.0, 1.0), (0.97, 1.0)])
def test_reference_equals_textbook_on_hand_cases(gamma, lam):
    case = _hand_cases()
    adv, ret = gae_reference(*case, gamma, lam)
    want, disc = gae_textbook(*case, gamma, lam)
    tol = _tol(case[0], case[3], case[4])
    assert np.all(np.abs(adv - want) <= tol)
    if lam == 1.0:                                  # lam = 1: A + V is the discounted, bootstrapped return
        assert np.all(np.abs(ret.astype(np.float64) - disc) <= tol)


@pytest.mark.parametrize("seed", range(4))
def test_reference_equals_textbook_on_random_rows(seed):
    case = _case(23, 40, seed)
    for gamma, lam in ((0.99, 0.95), (0.95, 1.0)):
        adv, ret = gae_reference(*case, gamma, lam)
        want, disc = gae_textbook(*case, gamma, lam)
        tol = _tol(case[0], case[3], case[4])
        assert np.all(np.abs(adv - want) <= tol)
        if lam == 1.0:
            assert np.all(np.abs(ret.astype(np.float64) - disc) <= tol)


def test_hand_cases_bootstrap_where_they_should():
    """Bootstrap values reach the advantage only through the rows that may use them."""
    reward, terminated, finished, values, final_values = _hand_cases()
    base, _ = gae_reference(reward, terminated, finished, values, final_values, 0.99, 0.95)
    for col, row, used in ((0, 2, False), (1, 3, True), (2, 1, True), (3, 4, False)):
        fv = final_values.copy()
        fv[row, col] += 100.0
        adv, _ = gae_reference(reward, terminated, finished, values, fv, 0.99, 0.95)
        assert (not np.array_equal(adv[:, col], base[:, col])) == used, col
        assert np.array_equal(adv[row + 1:, col], base[row + 1:, col])
    # values[t+1] of a finished row is never read
    v = values.copy()
    v[3, 0] = np.nan                                # row 2 of column 0 terminated: values[3] is not its next value
    adv, _ = gae_reference(reward, terminated, finished, v, final_values, 0.99, 0.95)
    assert np.array_equal(adv[:3, 0], base[:3, 0]) and np.isnan(adv[3, 0])


def test_non_finite_advantage_stays_in_its_episode():
    reward, terminated, finished, values, final_values = _hand_cases()
    reward = reward.copy()
    reward[3, 0] = np.inf                           # after column 0's termination at row 2
    reward[0, 4] = np.nan                           # column 4 ends an episode on every row
    adv, ret = gae_reference(reward, terminated, finished, values, final_values, 0.99, 0.95)
    assert np.all(np.isfinite(adv[:3, 0])) and not np.isfinite(adv[3, 0])
    assert np.isnan(adv[0, 4]) and np.all(np.isfinite(adv[1:, 4]))


def test_errors_before_any_device_call():
    L = _lib.lib()
    buf = (C.c_char * 512)()
    ptr = (C.addressof(buf) + 15) & ~15
    tr = _lib.DexsimTrajectory(ptr, None, ptr, ptr, None, ptr, 5)

    def call(traj=tr, n=0, ld=32, k=5, v=ptr, fv=ptr, a=ptr, r=ptr):
        return L.dexsim_gae(None if traj is None else C.byref(traj), n, ld, k, v, fv, C.c_float(0.99), C.c_float(0.95),
                            a, r, None)

    assert call() == 0                              # n == 0: nothing to do, obs / action / truncated not needed
    assert call(traj=None) == -1001
    for name in ("reward", "terminated", "finished"):
        setattr(tr, name, None)
        assert call() == -1001, name
        setattr(tr, name, ptr + 4)
        assert call() == -1003, name
        setattr(tr, name, ptr)
    for kw in ("v", "fv", "a", "r"):
        assert call(**{kw: None}) == -1001, kw
        assert call(**{kw: ptr + 8}) == -1003, kw
    assert call(n=-1) == -1002 and call(n=33, ld=32) == -1002 and call(n=5, ld=40) == -1002
    assert call(k=0) == -1002 and call(k=6) == -1002


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


def _values_for(env, k, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = env.num_envs
    values = torch.randn(k + 1, n, generator=g, device="cuda") * 5
    final_values = torch.randn(k, n, generator=g, device="cuda") * 5
    return values, final_values


def _check_env_gae(env, seed, gamma=0.99, lam=0.95):
    tr = env.trajectory
    k = tr["reward"].shape[0]
    values, final_values = _values_for(env, k, seed)
    adv, ret = env.gae(values, final_values, gamma, lam)
    want_a, want_r = gae_reference(tr["reward"].cpu().numpy(), tr["terminated"].cpu().numpy(),
                                   tr["finished"].cpu().numpy(), values.cpu().numpy(), final_values.cpu().numpy(),
                                   gamma, lam)
    assert np.array_equal(adv.cpu().numpy().view(np.uint32), want_a.view(np.uint32))
    assert np.array_equal(ret.cpu().numpy().view(np.uint32), want_r.view(np.uint32))
    return tr


@pytest.mark.gpu
def test_gae_equals_reference_truncation_wave(gpu):
    """1 Mi envs x 50 steps, 200-step episodes with no early termination: every env truncates on row 24."""
    n = 1 << 20
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=200, reward_type="dense", track_episodes=True, seed=3,
                                    curriculum_config=dx.CurriculumConfig.hard())
    env._params.success_threshold = 6               # five fingers: no episode terminates
    env.reset(seed=3)
    env.enable_trajectory(50)
    for k in (25, 50, 50, 50, 50):                  # steps 176 .. 225: the bound (200) falls on row 24
        env.rollout(k, policy="random")
    tr = _check_env_gae(env, 1)
    assert [t for t in range(50) if bool(tr["finished"][t].all())] == [24]
    assert not bool(tr["terminated"].any())


@pytest.mark.gpu
@pytest.mark.parametrize("loop", [None, 7])
def test_gae_equals_reference_short_episodes(gpu, loop):
    """15-step episodes (with the shipped threshold some terminate early), and a loop bound of 7."""
    env = dx.BatchedManipulationEnv(70_001, "cuda", max_episode_steps=15, reward_type="dense", track_episodes=True,
                                    seed=4)
    env.reset(seed=4)
    env.enable_trajectory(50)
    env.rollout(50, policy="heuristic", loop_max_steps=loop)
    tr = _check_env_gae(env, 2)
    frac = float(tr["finished"].float().mean())
    assert frac > 1 / 16 and bool(tr["terminated"].any())
    if loop is not None:                            # rows ended by the loop bound alone
        assert bool((tr["finished"] & ~tr["terminated"] & ~tr["truncated"]).any())
    for gamma, lam in ((1.0, 1.0), (0.9, 0.0)):
        _check_env_gae(env, 3, gamma, lam)


@pytest.mark.gpu
def test_gae_argument_checks(gpu):
    env = dx.BatchedManipulationEnv(100, "cuda", max_episode_steps=15, reward_type="dense", track_episodes=True, seed=4)
    env.reset(seed=4)
    v, fv = _values_for(env, 10, 0)
    with pytest.raises(RuntimeError):
        env.gae(v, fv, 0.99, 0.95)                  # no recording
    env.enable_trajectory(10)
    env.rollout(10, policy="random")
    env.gae(v, fv, 0.99, 0.95)
    for bad_v, bad_fv, exc in ((v[:-1], fv, ValueError), (v, fv[:, :-1], ValueError), (v.double(), fv, TypeError),
                               (v, fv.cpu(), ValueError)):
        with pytest.raises(exc):
            env.gae(bad_v, bad_fv, 0.99, 0.95)
    env.rollout(10, policy="random", one_episode=True, respawn=False)
    with pytest.raises(RuntimeError):
        env.gae(v, fv, 0.99, 0.95)                  # rows after a one_episode stop are not written


@pytest.mark.gpu
def test_gae_no_writes_outside_outputs(gpu):
    """advantages / returns between guard bands: nothing outside them, past column n or past row k is written."""
    n, k, cap, guard = 130, 10, 12, 4096
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=4, reward_type="dense", track_episodes=True, seed=5)
    env.reset(seed=5)
    env.enable_trajectory(cap)
    env.rollout(k, policy="random")
    ld = env.ld
    v, fv = torch.zeros(k + 1, ld, device="cuda"), torch.zeros(k, ld, device="cuda")
    vv, ff = _values_for(env, k, 6)
    v[:, :n], fv[:, :n] = vv, ff
    outs = []
    for _ in range(2):
        nbytes = cap * ld * 4
        big = torch.full((nbytes + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
        outs.append((big, big[guard:guard + nbytes].view(torch.float32).view(cap, ld)))
    tr = env._traj
    traj = _lib.DexsimTrajectory(tr["obs"].data_ptr(), None, tr["reward"].data_ptr(), tr["terminated"].data_ptr(),
                                 None, tr["finished"].data_ptr(), cap)
    pattern = outs[0][1].clone()
    _lib.check(_lib.lib().dexsim_gae(C.byref(traj), n, ld, k, v.data_ptr(), fv.data_ptr(), C.c_float(0.99),
                                     C.c_float(0.95), outs[0][1].data_ptr(), outs[1][1].data_ptr(), None), "dexsim_gae")
    torch.cuda.synchronize()
    for big, inner in outs:
        assert bool((big[:guard] == 0xA5).all()) and bool((big[-guard:] == 0xA5).all())
        assert torch.equal(inner[k:], pattern[k:]) and torch.equal(inner[:, n:], pattern[:, n:])
    adv, ret = env.gae(vv, ff, 0.99, 0.95)
    assert torch.equal(outs[0][1][:k, :n], adv) and torch.equal(outs[1][1][:k, :n], ret)
    assert int(env.trajectory["finished"].sum()) > 0
