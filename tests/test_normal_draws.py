"""The library's Gaussian draws (csrc/dexsim_core.cuh normal_pair / normal_rows: Box-Muller on Philox words) against a
float64 restatement of the same spec (oracle.normal_pair_ref / normal_rows_ref, DESIGN.md "RNG").

The device evaluates Box-Muller in float32 with the hardware log / sin / cos (__logf, __sinf, __cosf), so its draws are
compared with the float64 spec within a per-element bound derived from the published accuracy of those intrinsics
(CUDA C++ Programming Guide, "Intrinsic Functions") and from the float32 roundings the compiled code performs between
them: the product 6.2831855f·(u2 - 1/2), the correctly rounded sqrtf and the two final products.  Every input value of
each of the two words is swept exhaustively through a probe kernel that includes dexsim_core.cuh unchanged."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import oracle

PROBE_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "normal_pair_probe.cu")

U = 2.0 ** -24                          # unit roundoff of float32 (round to nearest)
TWO_PI_F = float(np.float32(2 * np.pi))  # 6.2831855f, the constant of the device's angle product
LN2 = math.log(2.0)
A_LOG = 2.0 ** -21.41                   # __logf: absolute error on [0.5, 2] ...
ULP_LOG = 3.0                           # ... and at most 3 ulp elsewhere
A_SIN = 2.0 ** -21.41                   # __sinf on [-pi, pi], absolute
A_COS = 2.0 ** -21.19                   # __cosf on [-pi, pi], absolute
A_TRIG = max(A_SIN, A_COS)
F64 = 2.0 ** -50                        # float64 evaluation of the reference and of the error measures (generous)
R_MAX = math.sqrt(48 * LN2)             # largest radius: u1 = 2^-24, sqrt(-2 ln 2^-24) ~ 5.77
# (c^2 + s^2) of the hardware cosine / sine is 1 within 2|(e_c, e_s)| + |(e_c, e_s)|^2; sqrtf and the two products
# each add one rounding of relative size <= U to the radius, hence four to the squared radius
EPS_R2 = (1 + U) ** 4 * (1 + 2 * math.hypot(A_COS, A_SIN) + A_COS ** 2 + A_SIN ** 2) - 1


def _log_err(R2, xp):
    """Bound on |__logf(u1) - ln u1| for u1 = exp(-R2 / 2): absolute on [0.5, 1], 3 ulp (<= 3·2^-23·|ln u1|) below."""
    return xp.where(R2 <= 2 * LN2 * (1 + 1e-12), A_LOG, ULP_LOG * 2.0 ** -23 * (R2 / 2))


def _theta_err(theta, xp):
    """|theta_f - theta| for theta_f = fl(6.2831855f·d), theta = 2·pi·d, d = u2 - 1/2 (exact in float32)."""
    d = xp.abs(theta) / (2 * math.pi)
    return d * abs(TWO_PI_F - 2 * math.pi) + U * TWO_PI_F * d


def r2_bound(R2, xp):
    """Bound on |z0^2 + z1^2 - R^2|, R^2 = -2 ln u1: relative EPS_R2 plus twice the log error."""
    return EPS_R2 * R2 + 2 * _log_err(R2, xp) * (1 + EPS_R2) + F64 * R2


def angle_bound(theta, xp):
    """Bound on |atan2(z1, z0) - theta| (mod 2 pi): the angle product, a point within |(e_c, e_s)| of the unit circle
    seen from the origin, and the two final products rounded independently (tan scaled by (1 + d1) / (1 + d0))."""
    return _theta_err(theta, xp) + math.asin(math.hypot(A_COS, A_SIN)) + U * (1 + U) / (1 - U) + F64


def z_bound(R, theta, xp):
    """Bound on |z0 - R cos(theta)| and |z1 - R sin(theta)|."""
    eL = _log_err(R * R, xp)
    # |sqrt(-2 L) - R| = |2 (L - ln u1)| / (sqrt(-2 L) + R) <= min(2 eL / R, sqrt(2 eL))
    dr = xp.minimum(2 * eL / xp.where(R > 0, R, 1e-300), xp.sqrt(2 * eL))
    drad = dr + U * (R + dr)                                             # + the rounding of sqrtf
    return drad * (1 + A_TRIG) * (1 + U) + R * (A_TRIG + _theta_err(theta, xp)) + U * R * (1 + A_TRIG) + F64 * (1 + R)


# ---- the reference itself (CPU) ----------------------------------------------------------------------------------

def _words(hi24, low8=0):
    return (np.asarray(hi24, np.uint64) << np.uint64(8) | np.uint64(low8)).astype(np.uint32)


def test_normal_pair_ref_known_answers():
    r = np.sqrt(-2 * np.log((np.arange(0, 1 << 24, 99_991, dtype=np.float64) + 1) * U))
    wa = _words(np.arange(0, 1 << 24, 99_991), 0x5A)
    z0, z1 = oracle.normal_pair_ref(_words(2 ** 24 - 1, 0xFF), _words([0, 2 ** 22, 2 ** 23, 2 ** 24 - 1]))
    assert np.all(z0 == 0) and np.all(z1 == 0)                          # u1 = 1: radius 0 at every angle
    z0, z1 = oracle.normal_pair_ref(wa, _words(2 ** 23, 0x33))           # u2 = 1/2: theta = 0
    np.testing.assert_allclose(z0, r, rtol=1e-15)
    assert np.all(z1 == 0)
    z0, z1 = oracle.normal_pair_ref(wa, _words(2 ** 22))                 # u2 = 1/4: theta = -pi/2
    np.testing.assert_allclose(z0, 0, atol=1e-15)
    np.testing.assert_allclose(z1, -r, rtol=1e-15)
    z0, z1 = oracle.normal_pair_ref(_words(0), _words(2 ** 23))          # the truncation point: u1 = 2^-24
    assert z0[()] == pytest.approx(R_MAX, rel=1e-15) and z1 == 0


def test_normal_rows_ref_uses_philox_block_words_in_order():
    seed, gid, ep, step = 0x9E3779B97F4A7C15, 2 ** 32 - 3, 7, 11
    for stream, rows in ((2, 15), (3, 45), (4, 15), (5, 15)):
        got = oracle.normal_rows_ref(seed, gid, ep, step, stream, rows, 0.5)[0]
        exp = []
        for b in range((rows + 3) // 4):
            x, y, z, w = oracle.philox([gid, ep, step, stream | b << 8], [seed & 0xFFFFFFFF, seed >> 32])
            exp += [*oracle.normal_pair_ref(x, y), *oracle.normal_pair_ref(z, w)]
        assert np.array_equal(got, 0.5 * np.asarray(exp[:rows]))


def test_normal_rows_ref_distribution():
    import scipy.stats
    n = 1 << 17
    gid = np.arange(n)
    z = oracle.normal_rows_ref(12345, gid, gid % 7, gid % 13, 2, 8, 1.0)      # 8 rows = two blocks: 1,048,576 draws
    ks = scipy.stats.kstest(z.ravel(), "norm")
    assert ks.pvalue > 1e-3, ks
    assert abs(z.mean()) < 5e-3 and abs(z.std() - 1) < 5e-3
    pairs = z.reshape(n, 4, 2)                                           # (z0, z1) of one Box-Muller pair
    rho = np.corrcoef(pairs[..., 0].ravel(), pairs[..., 1].ravel())[0, 1]
    assert abs(rho) < 5 / math.sqrt(pairs[..., 0].size), rho
    assert np.abs(z).max() <= R_MAX


# ---- the device's normal_pair, every input value ------------------------------------------------------------------

@pytest.fixture(scope="session")
def probe(tmp_path_factory):
    """normal_pair compiled exactly as the library compiles it (build.NVCC_FLAGS), callable on device tensors."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from dexterous_rl_manipulation_b200 import build
    out = str(tmp_path_factory.mktemp("normal_pair_probe") / "normal_pair_probe.so")
    proc = subprocess.run([build.nvcc_path()] + build.NVCC_FLAGS + ["-o", out, PROBE_SRC],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert proc.returncode == 0, proc.stdout
    lib = C.CDLL(out)
    lib.normal_pair_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.normal_pair_probe.restype = C.c_int

    def run(wa, wb):
        """wa, wb: int32 device tensors holding the uint32 words; returns float32 (z0, z1)."""
        z0, z1 = torch.empty_like(wa, dtype=torch.float32), torch.empty_like(wa, dtype=torch.float32)
        rc = lib.normal_pair_probe(wa.data_ptr(), wb.data_ptr(), z0.data_ptr(), z1.data_ptr(), wa.numel(),
                                   torch.cuda.current_stream().cuda_stream)
        assert rc == 0, rc
        return z0, z1
    return run


def _dev_words(hi24, low8=0):
    """uint32 words (hi24 << 8 | low8) as int32 device tensors (same bits)."""
    w = (hi24.to(torch.int64) << 8) | low8
    return (w - (w >= 2 ** 31).to(torch.int64) * 2 ** 32).to(torch.int32)


def _spec(a24, b24):
    """Float64 spec on the device from the 24-bit fields: R^2, R, theta, Z0, Z1."""
    u1 = (a24.to(torch.float64) + 1) * U
    R2 = -2 * torch.log(u1)
    R = torch.sqrt(R2)
    theta = 2 * math.pi * (b24.to(torch.float64) * U - 0.5)
    return R2, R, theta, R * torch.cos(theta), R * torch.sin(theta)


@pytest.mark.gpu
def test_normal_pair_exhaustive_sweeps(probe):
    """Sweep A: all 2^24 values of wa >> 8 at five angles (theta = -pi, -pi/2, 0, pi/2, ~pi).  Sweep B: all 2^24 values
    of wb >> 8 at four radii (u1 = 2^-24, 1/2 - 2^-24, 1 - 2^-24, 1).  Every output finite, and per element within the
    bounds derived above for the squared radius, the angle and each coordinate."""
    full = torch.arange(1 << 24, device="cuda", dtype=torch.int64)
    cases = [("A", full, torch.full_like(full, b)) for b in (0, 2 ** 22, 2 ** 23, 3 * 2 ** 22, 2 ** 24 - 1)] + \
            [("B", torch.full_like(full, a), full) for a in (0, 2 ** 23 - 1, 2 ** 24 - 2, 2 ** 24 - 1)]
    worst = dict(r2_abs_hi=0.0, r2_rel_lo=0.0, angle=0.0, z=0.0, r2_ratio=0.0, angle_ratio=0.0, z_ratio=0.0)
    nonfinite, n_nonfinite = [], 0
    checked_oracle = False
    for name, a24, b24 in cases:
        z0, z1 = probe(_dev_words(a24), _dev_words(b24))
        bad = ~(torch.isfinite(z0) & torch.isfinite(z1))
        if bool(bad.any()):
            n_nonfinite += int(bad.sum())
            nonfinite += [(name, a, b) for a, b in zip(a24[bad][:64].tolist(), b24[bad][:64].tolist())]
        ok = ~bad
        R2, R, theta, Z0, Z1 = _spec(a24, b24)
        if not checked_oracle:          # the device-side float64 spec is the oracle's, on a random subset
            pick = torch.randint(0, 1 << 24, (4096,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
            o0, o1 = oracle.normal_pair_ref(_words(a24[pick].cpu().numpy()), _words(b24[pick].cpu().numpy()))
            np.testing.assert_allclose(Z0[pick].cpu().numpy(), o0, rtol=1e-14, atol=1e-15)
            np.testing.assert_allclose(Z1[pick].cpu().numpy(), o1, rtol=1e-14, atol=1e-15)
            checked_oracle = True
        x0, x1 = z0.to(torch.float64)[ok], z1.to(torch.float64)[ok]
        R2, R, theta, Z0, Z1 = R2[ok], R[ok], theta[ok], Z0[ok], Z1[ok]
        e_r2 = (x0 * x0 + x1 * x1 - R2).abs()
        hi = R2 <= 2 * LN2                                               # u1 in [0.5, 1]: absolute log error
        if bool(hi.any()):
            worst["r2_abs_hi"] = max(worst["r2_abs_hi"], float(e_r2[hi].max()))
        if bool((~hi).any()):
            worst["r2_rel_lo"] = max(worst["r2_rel_lo"], float((e_r2[~hi] / R2[~hi]).max()))
        worst["r2_ratio"] = max(worst["r2_ratio"], float((e_r2 / r2_bound(R2, torch)).max()))
        nz = (x0 != 0) | (x1 != 0)                                       # the angle of a zero radius is undefined
        e_ang = torch.remainder(torch.atan2(x1, x0) - theta + math.pi, 2 * math.pi) - math.pi
        e_ang = e_ang[nz].abs()
        if e_ang.numel():
            worst["angle"] = max(worst["angle"], float(e_ang.max()))
            worst["angle_ratio"] = max(worst["angle_ratio"], float((e_ang / angle_bound(theta[nz], torch)).max()))
        e_z = torch.maximum((x0 - Z0).abs(), (x1 - Z1).abs())
        worst["z"] = max(worst["z"], float(e_z.max()))
        worst["z_ratio"] = max(worst["z_ratio"], float((e_z / z_bound(R, theta, torch)).max()))
        del z0, z1, R2, R, theta, Z0, Z1, x0, x1, e_r2, e_ang, e_z
    print("\nnormal_pair sweeps: max |r^2 - R^2| (u1 >= 1/2) %.3e, max |r^2 - R^2| / R^2 (u1 < 1/2) %.3e, "
          "max angle error %.3e rad, max |z - Z| %.3e; largest error / bound: r^2 %.3f, angle %.3f, z %.3f; "
          "non-finite outputs: %d, at wa >> 8 in %s" % (worst["r2_abs_hi"], worst["r2_rel_lo"], worst["angle"], worst["z"],
                                                        worst["r2_ratio"], worst["angle_ratio"], worst["z_ratio"],
                                                        n_nonfinite, sorted({a for _, a, _ in nonfinite})[:16]))
    assert not nonfinite, "non-finite normal_pair outputs at (sweep, wa >> 8, wb >> 8): %s" % nonfinite[:32]
    assert worst["r2_ratio"] <= 1.0 and worst["angle_ratio"] <= 1.0 and worst["z_ratio"] <= 1.0, worst


@pytest.mark.gpu
def test_normal_pair_ignores_the_low_byte(probe):
    """Only the top 24 bits of each word are used: random words give bit-identical output with the low bytes cleared."""
    g = torch.Generator(device="cuda").manual_seed(7)
    wa = torch.randint(-2 ** 31, 2 ** 31, (1 << 22,), device="cuda", dtype=torch.int64, generator=g).to(torch.int32)
    wb = torch.randint(-2 ** 31, 2 ** 31, (1 << 22,), device="cuda", dtype=torch.int64, generator=g).to(torch.int32)
    assert int(((wa & 0xFF) != 0).sum()) > (1 << 21) and int(((wb & 0xFF) != 0).sum()) > (1 << 21)
    a0, a1 = probe(wa, wb)
    b0, b1 = probe(wa & ~0xFF, wb & ~0xFF)
    assert torch.equal(a0.view(torch.int32), b0.view(torch.int32)) and torch.equal(a1.view(torch.int32), b1.view(torch.int32))


# ---- what the library's entry points draw ----------------------------------------------------------------------------

@pytest.fixture(scope="module")
def dx():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import dexterous_rl_manipulation_b200 as d
    return d


SEED = 0x9E3779B97F4A7C15               # non-zero high word: both key words matter


def _fill_normal(env, stream, rows, sigma, out):
    from dexterous_rl_manipulation_b200 import _lib
    _lib.check(env._lib.dexsim_fill_normal(C.byref(env._state), C.byref(env._params), stream, rows, C.c_float(sigma),
                                           out.data_ptr(), env._stream()), "dexsim_fill_normal")
    return out


def _check_against_reference(got, ref, sigma):
    """got [n, rows] float32 from the device, ref [n, rows4] float64 sigma·Z of the spec (rows4 = rows rounded up to a
    whole Philox block, so every coordinate has its Box-Muller partner for R and theta)."""
    n, rows = got.shape
    pair = ref.reshape(n, -1, 2) / sigma
    R = np.repeat(np.hypot(pair[..., 0], pair[..., 1]), 2, axis=1)[:, :rows]
    theta = np.repeat(np.arctan2(pair[..., 1], pair[..., 0]), 2, axis=1)[:, :rows]
    tol = sigma * z_bound(R, theta, np) + np.spacing(np.abs(got)).astype(np.float64) / 2
    err = np.abs(got.astype(np.float64) - ref[:, :rows])
    assert np.all(err <= tol), (float((err / tol).max()), np.unravel_index(np.argmax(err / tol), err.shape))


@pytest.mark.gpu
@pytest.mark.parametrize("n,gid0", [(1, 2 ** 31 - 1), (33, 2 ** 32 - 20), (4097, 2 ** 31 - 100), (4097, 2 ** 32 - 20)])
def test_fill_normal_matches_reference(dx, n, gid0):
    """dexsim_fill_normal for every stream it exposes (2 dynamics, 3 observation, 4 learner exploration, 5 learner
    update), both row counts and three sigmas, with distinct (episode, step) words per env and env ids that cross 2^31
    or wrap past 2^32 inside the batch: element by element within sigma × the per-draw bound + half an ulp, and nothing
    written past column n of the [rows, ld] output."""
    env = dx.BatchedManipulationEnv(n, "cuda", seed=SEED, env_gid0=gid0)
    env.reset(seed=SEED)
    rng = np.random.default_rng(n + gid0)
    ep = rng.integers(1, 2 ** 32, n, dtype=np.int64)
    sc = rng.integers(1, 2 ** 32, n, dtype=np.int64)
    env._episode[:n] = torch.from_numpy((ep - (ep >= 2 ** 31) * 2 ** 32).astype(np.int32)).cuda()
    env._step_count[:n] = torch.from_numpy((sc - (sc >= 2 ** 31) * 2 ** 32).astype(np.int32)).cuda()
    gid = gid0 + np.arange(n)
    sentinel = -1234.5
    for stream in (2, 3, 4, 5):
        for rows in (15, 45):
            for sigma in (1.0, 0.05, 3.0):
                out = torch.full((rows, env.ld), sentinel, dtype=torch.float32, device="cuda")
                _fill_normal(env, stream, rows, sigma, out)
                s = float(np.float32(sigma))
                ref = oracle.normal_rows_ref(SEED, gid, ep, sc, stream, (rows + 3) // 4 * 4, s)
                _check_against_reference(out[:, :n].t().cpu().numpy(), ref, s)
                assert bool((out[:, n:] == sentinel).all())
    with pytest.raises(dx.DexsimError):
        _fill_normal(env, 6, 15, 1.0, torch.zeros(15, env.ld, device="cuda"))


@pytest.mark.gpu
def test_philox_learner_draws_streams_4_and_5(dx):
    """rollout(policy="learner") without pre-drawn noise draws exploration from stream 4 and the update from stream 5,
    both keyed by the step count BEFORE the step: K one-step launches fed with dexsim_fill_normal(4 | 5) draws equal
    one K-step Philox launch bit for bit (auto-resets included), and the recorded draws replayed through the oracle's
    SimpleLearner give the same trajectories, learner state and counters."""
    CC = dx.CurriculumConfig
    n, K, seed, lr, expl = 2000, 150, 21, 0.01, 0.3
    cfg = CC.medium()
    kw = dict(max_episode_steps=40, reward_type="dense", curriculum_config=cfg, track_episodes=True, seed=seed)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    for e in (a, b):
        e.enable_learner(lr, expl, 0.5)
        e.reset(seed=seed)
    ob = oracle.OracleBatch(n, dense=True, max_episode_steps=40)
    ob.reset_predrawn(a._obs[:15, :n].t().cpu().numpy(), a._size[:n].cpu().numpy(), a._mass[:n].cpu().numpy(),
                      a._friction[:n].cpu().numpy(), a._obs[30:33, :n].t().cpu().numpy())
    run = dict(policy="learner", respawn=False, loop_max_steps=40, success_is_terminated=False)
    act_buf, upd_buf = torch.empty(15, a.ld, device="cuda"), torch.empty(15, a.ld, device="cuda")
    acts, upds = [], []
    for t in range(K):
        act = _fill_normal(a, 4, 15, expl, act_buf)[:, :n].t().contiguous()
        upd = _fill_normal(a, 5, 15, lr, upd_buf)[:, :n].t().to(torch.float64).contiguous()
        acts.append(act); upds.append(upd)
        a.rollout(1, learner_act_noise=act[None], learner_upd_noise=upd[None], **run)
    b.rollout(K, **run)
    assert int(b.counters[0, 0]) > n                                     # every env finished at least one episode
    for name in ("_obs", "_op64", "_episode", "_step_count", "_learner_mean", "_learner_best"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert torch.equal(a.counters, b.counters)
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0)
    assert int((b.learner_mean != 0).any(1).sum()) > n // 2              # the update draw moved most learners
    mean = np.zeros((n, 15), np.float32); best = np.full(n, -np.inf)
    cnt, rs = oracle.rollout_learner(ob, oracle.make_group(cfg), K, seed, mean, best, torch.stack(acts).cpu().numpy(),
                                     torch.stack(upds).cpu().numpy(), respawn=False, loop_max_steps=40)
    assert np.array_equal(b.counters.cpu().numpy()[:, :16], cnt[:, :16])
    assert np.array_equal(b.learner_mean.cpu().numpy(), mean)
    gb = b.learner_best.cpu().numpy()              # best holds float64 rewards: CUDA and glibc exp differ by <= 1 ulp
    assert np.array_equal(np.isinf(gb), np.isinf(best))
    np.testing.assert_allclose(gb[np.isfinite(gb)], best[np.isfinite(best)], rtol=1e-14)
    assert np.array_equal(b._obs[:, :n].t().cpu().numpy(), ob.observation())
    np.testing.assert_allclose(b.ret_sums.cpu().numpy(), rs, rtol=1e-9)


@pytest.mark.gpu
def test_full_size_noisy_paths_stay_finite(dx):
    """1,048,576 envs through the product's noisy paths: API steps with sigma_obs 0.05 and sigma_dyn 0.1 drawn in the
    step kernel (auto-reset, counts-only tracking), then a 200-step fused learner rollout with per-group sigma_dyn.
    Every observation, noisy observation, position, reward and learner value stays finite."""
    CC = dx.CurriculumConfig
    N, seed = 1 << 20, 42
    env = dx.BatchedManipulationEnv(N, "cuda", max_episode_steps=8, reward_type="dense", seed=seed, curriculum_config=CC.hard(),
                                    observation_noise_std=0.05, dynamics_noise_std=0.1, auto_reset=True, respawn=True,
                                    loop_max_steps=8, track_episodes=False)
    env.reset(seed=seed)
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(20):
        obs, rew, te, tr, info = env.step(torch.rand(N, 15, device="cuda", generator=gen) * 2 - 1)
        assert bool(torch.isfinite(obs).all()) and bool(torch.isfinite(rew).all()), t
    assert int(env.counters[:, 0].sum()) >= N                             # every env was auto-reset at least once
    for name in ("_obs", "_noisy_obs", "_op64"):
        assert bool(torch.isfinite(getattr(env, name)[:, :N]).all()), name
    del env
    env = dx.BatchedManipulationEnv(N, "cuda", max_episode_steps=50, reward_type="dense", seed=seed, track_episodes=True,
                                    groups=[CC.easy(), CC.hard()], group_sigma_dyn=[0.1, 0.3])
    env.enable_learner(0.01, 0.3, 0.5)
    env.reset(seed=seed)
    env.rollout(200, policy="learner")
    assert int(env.counters[:, 0].sum()) >= N
    for name in ("_obs", "_op64"):
        assert bool(torch.isfinite(getattr(env, name)[:, :N]).all()), name
    assert bool(torch.isfinite(env.learner_mean).all()) and not bool(torch.isnan(env.learner_best).any())
    assert bool(torch.isfinite(env.ret_sums).all())
