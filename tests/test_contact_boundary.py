"""The contact decision on the exact size * 1.5 boundary, in every kernel that makes it.

The reference decides contact with ``RN(sqrt(sq)) < size * 1.5`` in float64 (envs/manipulation_env.py:309-310).  The
kernels compare ``sq`` with ``thr^2 (1 -+ 2^-50)`` and take the square root only inside that tie band
(``finger_contact`` in dexsim_core.cuh; the fused 5-lanes-per-env rollout has its own copy, ``split_contact``).  Random
inputs land in a band of relative width 2^-49 about once in 10^15 finger-steps, so these tests put fingers there on
purpose: they take a state, compute the fingertip distance exactly as the reference does, and choose the object size
whose threshold lies a few ulps around it (``d == thr`` included).  Contacts never feed back into the dynamics, so a
trajectory is the same for every size as long as no episode ends early: sizes tuned on one oracle pre-run are hit by the
replay, and every case asserts how many finger-steps landed in the band (decided either way) and exactly on the tie.

Domain of the shortcut.  Fingertips are float32 values and object positions stay on the float32 grid (float64 sums of
float32 values: multiples of 2^-149), so a squared distance is 0 or at least 2^-298.  On that domain, for every
threshold (0, negative, tiny enough that thr^2 underflows, huge enough that it overflows, inf, NaN), the kernel's
decision equals the reference's; ``test_shortcut_equals_reference_on_constructed_boundaries`` checks it on millions of
constructed cases."""
import numpy as np
import pytest
import torch

from oracle import oracle

SQ_MIN = 2.0 ** -298          # smallest non-zero squared distance of two points on the float32 grid


# ---- the decision, restated ------------------------------------------------------------------------------------------
def shortcut_contact(sq, thr):
    """finger_contact / split_contact operation by operation (float64, round to nearest)."""
    with np.errstate(over="ignore", invalid="ignore"):
        thr2 = thr * thr
        lo2, hi2 = thr2 * (1.0 - 2.0 ** -50), thr2 * (1.0 + 2.0 ** -50)
        below, above = sq < lo2, sq > hi2
        c = np.where(below | above, below, np.sqrt(sq) < thr)
        return c & (thr > 0.0)


def reference_contact(sq, thr):
    with np.errstate(invalid="ignore"):
        return np.sqrt(sq) < thr


def in_band(sq, thr):
    with np.errstate(over="ignore", invalid="ignore"):
        thr2 = thr * thr
        return ~((sq < thr2 * (1.0 - 2.0 ** -50)) | (sq > thr2 * (1.0 + 2.0 ** -50)))


def finger_sq(jp, op):
    """Squared fingertip-object distances [..., 5] as the reference computes them: float32 sequential joint sums times
    0.1f widened to float64, then (dx*dx + dy*dy) + dz*dz in float64.  jp [..., 15] float32, op [..., 3] float64."""
    jp = np.asarray(jp, np.float32)
    s = (jp[..., 0::3] + jp[..., 1::3]) + jp[..., 2::3]
    tip = (s * np.float32(0.1)).astype(np.float64)
    op = np.asarray(op, np.float64)
    dx, dy, dz = tip - op[..., 0:1], tip - op[..., 1:2], tip - op[..., 2:3]
    return (dx * dx + dy * dy) + dz * dz


def nudge(x, k):
    """x moved by k float64 ulps (k may be an array)."""
    x = np.array(x, np.float64, copy=True)
    k = np.broadcast_to(np.asarray(k), x.shape)
    with np.errstate(over="ignore"):
        for s in range(int(np.abs(k).max(initial=0))):
            up, dn = k > s, -k > s
            x[up] = np.nextafter(x[up], np.inf)
            x[dn] = np.nextafter(x[dn], -np.inf)
    return x


def size_for(thr):
    """A float64 size with size * 1.5 == thr, NaN where no float64 gives exactly thr."""
    thr = np.asarray(thr, np.float64)
    c, out = thr / 1.5, np.full(thr.shape, np.nan)
    for j in (0, 1, -1, 2, -2, 3, -3):
        cand = nudge(c, j)
        ok = np.isnan(out) & (cand * 1.5 == thr)
        out[ok] = cand[ok]
    return out


def draw_offsets(rng, n):
    """Ulp offsets of the threshold from the distance: mostly inside the band (|k| <= 2, k == 0 is the exact tie),
    the rest out to 8 ulps."""
    k = rng.integers(-2, 3, n)
    wide = rng.random(n) < 0.2
    k[wide] = rng.integers(-8, 9, int(wide.sum()))
    return k


def tuned_sizes(sq, k):
    """Sizes whose threshold sits k ulps from sqrt(sq); where that threshold is not reachable, the nearest reachable
    offset (k+1, k-1, k+2, ...)."""
    d = np.sqrt(np.asarray(sq, np.float64))
    out = np.full(d.shape, np.nan)
    for j in (0, 1, -1, 2, -2, 3, -3):
        cand = size_for(nudge(d, np.asarray(k) + j))
        fill = np.isnan(out)
        out[fill] = cand[fill]
    assert not np.isnan(out).any()
    return out


def coverage(sq, thr, contact):
    """Finger-steps in the tie band decided "contact" / "no contact", and finger-steps with d == thr exactly; asserts the
    decision given is the reference's."""
    sq, thr, contact = np.asarray(sq), np.asarray(thr), np.asarray(contact, bool)
    assert np.array_equal(contact, reference_contact(sq, thr))
    band = in_band(sq, thr)
    return {"band_contact": int((band & contact).sum()), "band_free": int((band & ~contact).sum()),
            "tie": int((np.sqrt(sq) == thr).sum())}


def assert_coverage(cov, minimum):
    print("coverage", cov)
    for key, m in minimum.items():
        assert cov[key] >= m, (key, cov)


# ---- CPU: the shortcut against the reference, and the oracle against the reference ----------------------------------
def _boundary_sweep(rng):
    """(sq, thr) pairs on and around the boundary: yields arrays, about 8 million pairs in all."""
    ks = np.arange(-8, 9)
    # states the simulator can produce: joints in [-1, 1], positions in the workspace, float32 and float64 positions
    m = 40_000
    jp = rng.uniform(-1, 1, (m, 15)).astype(np.float32)
    op = np.stack([rng.uniform(-0.2, 0.2, m), rng.uniform(-0.2, 0.2, m), rng.uniform(0.0, 0.3, m)], 1)
    op[::2] = op[::2].astype(np.float32)
    sq = finger_sq(jp, op).ravel()
    for k in ks:
        thr = nudge(np.sqrt(sq), k)
        yield sq, thr                                        # every target threshold
        s = size_for(thr)
        ok = ~np.isnan(s)
        yield sq[ok], s[ok] * 1.5                           # the reachable ones, through a size
    # thresholds across binades: sq = mantissa * 2^e over the whole domain above 2^-298
    e = rng.integers(-298, 1023, 100_000)
    sq = np.ldexp(rng.uniform(1.0, 2.0, e.size), e)
    sq = sq[np.isfinite(sq)]
    for k in ks:
        yield sq, nudge(np.sqrt(sq), k)
    # the bottom of the domain, and squares near the top of the float64 range (thr^2 rounds close to overflow)
    for sq in (np.full(1000, SQ_MIN) * rng.integers(1, 1 << 20, 1000), np.nextafter(np.finfo(np.float64).max, 0) / rng.uniform(1, 4, 1000)):
        for k in ks:
            yield sq, nudge(np.sqrt(sq), k)
    # thresholds that are 0, negative, tiny (thr^2 underflows to 0 or a subnormal), huge (thr^2 overflows), inf, NaN;
    # squared distances 0, the smallest on the grid, ordinary, huge, inf and NaN
    sqs = np.concatenate([[0.0, SQ_MIN, 2 * SQ_MIN, 1e-80, 1e-20, 0.0123, 1.0, 1e300, np.finfo(np.float64).max, np.inf, np.nan],
                          rng.uniform(0, 0.5, 200)])
    thrs = np.concatenate([[0.0, -0.0, -1e-300, -0.05, -np.inf, 1e-300 * 1.5, 5e-324, 1e-200, 2.0 ** -537, 2.0 ** -511,
                            1e-160, 1e154, 1.4e154, 1e155, 1e200, np.finfo(np.float64).max, np.inf, np.nan],
                           np.sqrt(sqs[np.isfinite(sqs)])])
    S, T = np.meshgrid(sqs, thrs)
    for k in (-2, -1, 0, 1, 2):
        yield S.ravel(), nudge(T.ravel(), k)


def test_shortcut_equals_reference_on_constructed_boundaries():
    rng = np.random.default_rng(20261021)
    total = band = 0
    for sq, thr in _boundary_sweep(rng):
        assert ((sq == 0) | (sq >= SQ_MIN) | ~np.isfinite(sq)).all()          # the domain the shortcut is proven on
        got, want = shortcut_contact(sq, thr), reference_contact(sq, thr)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, [(float(sq[i]), float(thr[i]), bool(got[i])) for i in bad[:5]]
        total += sq.size
        band += int(in_band(sq, thr).sum())
    print(f"{total} boundary cases, {band} in the tie band")
    assert total >= 1_000_000 and band >= 300_000


def _reset_cases(rng, n):
    jp0 = rng.uniform(-0.1, 0.1, (n, 15)).astype(np.float32)
    p = np.stack([rng.uniform(-0.1, 0.1, n), rng.uniform(-0.1, 0.1, n), rng.uniform(0.05, 0.2, n)], 1).astype(np.float32)
    return jp0, p


def test_oracle_decides_the_reference_way_at_reset():
    rng = np.random.default_rng(1)
    n = 6000
    jp0, pos = _reset_cases(rng, n)
    sq = finger_sq(jp0, pos.astype(np.float64))
    size = tuned_sizes(sq[np.arange(n), np.arange(n) % 5], draw_offsets(rng, n))
    ob = oracle.OracleBatch(n)
    obs = ob.reset_predrawn(jp0, size, 0.1, 0.5, pos)
    cov = coverage(sq, (size * 1.5)[:, None], obs[:, 40:45] > 0.5)
    assert_coverage(cov, {"band_contact": 1000, "band_free": 1500, "tie": 700})


def test_oracle_decides_the_reference_way_after_steps():
    rng = np.random.default_rng(2)
    n, K = 3000, 6
    jp0, pos = _reset_cases(rng, n)
    acts = rng.uniform(-1.2, 1.2, (K, n, 15)).astype(np.float32)
    pre = oracle.OracleBatch(n)
    pre.reset_predrawn(jp0, 0.05, 0.1, 0.5, pos)
    sqs = []
    for t in range(K):
        o = pre.step(acts[t])[0]
        sqs.append(finger_sq(o[:, :15], pre.env["op"]))
    t_of, f_of = rng.integers(0, K, n), rng.integers(0, 5, n)
    size = tuned_sizes(np.stack(sqs)[t_of, np.arange(n), f_of], draw_offsets(rng, n))
    ob = oracle.OracleBatch(n)
    ob.reset_predrawn(jp0, size, 0.1, 0.5, pos)
    cov = {"band_contact": 0, "band_free": 0, "tie": 0}
    for t in range(K):
        o = ob.step(acts[t])[0]
        c = coverage(finger_sq(o[:, :15], ob.env["op"]), (size * 1.5)[:, None], o[:, 40:45] > 0.5)
        cov = {k: cov[k] + c[k] for k in cov}
    for k in ("jp", "jv", "op", "ov"):                  # the trajectory does not depend on the size
        assert np.array_equal(ob.env[k], pre.env[k]), k
    assert_coverage(cov, {"band_contact": 500, "band_free": 800, "tie": 350})


def test_single_step_oracle_rollouts_resume_where_they_stopped():
    """The GPU rollout cases take per-step oracle states from repeated one-step rollouts: K of them must leave the same
    state and counters as one K-step rollout."""
    G, n, K, M, seed = 7, 200, 25, 6, 5
    groups = np.concatenate([oracle.make_group(None, object_size=0.03 + 0.01 * g) for g in range(G)])
    a, b = oracle.OracleBatch(n, max_episode_steps=M), oracle.OracleBatch(n, max_episode_steps=M)
    for ob in (a, b):
        _oracle_initial_reset(ob, groups, seed)
    ca, ra = a.rollout(groups, K, seed, policy_kind=2, loop_max_steps=M)
    cb = rb = None
    for _ in range(K):
        cb, rb = b.rollout(groups, 1, seed, policy_kind=2, loop_max_steps=M, counters=cb, ret_sums=rb)
    assert np.array_equal(a.env, b.env) and np.array_equal(ca, cb) and int(ca[:, 0].sum()) >= 3 * n
    np.testing.assert_allclose(ra, rb, rtol=1e-12)


# ---- oracle side of the GPU cases --------------------------------------------------------------------------------------
def _oracle_initial_reset(ob, groups, seed):
    G = groups.shape[0]
    draws = [oracle.reset_draws(seed, i, 0, groups[i % G:i % G + 1]) for i in range(ob.n)]
    return ob.reset_predrawn(np.stack([d[0] for d in draws]), np.array([d[1] for d in draws]),
                             np.array([d[2] for d in draws]), np.array([d[3] for d in draws]), np.stack([d[4] for d in draws]))


def _decisions(obs, op, size):
    """(sq [n, 5], thr [n, 1], contact [n, 5]) of a state given by its observation and float64 object position."""
    return finger_sq(obs[:, :15], op), (np.asarray(size, np.float64) * 1.5)[:, None], obs[:, 40:45] > 0.5


def _cov_sum(points):
    cov = {"band_contact": 0, "band_free": 0, "tie": 0}
    for sq, thr, c in points:
        x = coverage(sq, np.broadcast_to(thr, sq.shape), c)
        cov = {k: cov[k] + x[k] for k in cov}
    return cov


class PlainRun:
    """Per-env sizes through reset_from_draws, then K external-action steps without auto-reset.  Every env's size is
    tuned to one finger at the reset state or at one step of a pre-run."""

    def __init__(self, n, K, dense, success_threshold, seed, max_steps=200):
        rng = np.random.default_rng(seed)
        self.n, self.K = n, K
        self.jp0, self.pos = _reset_cases(rng, n)
        self.mass, self.fric = rng.uniform(0.05, 0.3, n), rng.uniform(0.0, 1.0, n)
        self.acts = rng.uniform(-1.2, 1.2, (K, n, 15)).astype(np.float32)
        pre = oracle.OracleBatch(n, dense=dense, max_episode_steps=max_steps)
        o = pre.reset_predrawn(self.jp0, 0.05, self.mass, self.fric, self.pos)
        sqs = [finger_sq(o[:, :15], pre.env["op"])]
        for t in range(K):
            o = pre.step(self.acts[t])[0]
            sqs.append(finger_sq(o[:, :15], pre.env["op"]))
        t_of, f_of = rng.integers(0, K + 1, n), rng.integers(0, 5, n)
        self.size = tuned_sizes(np.stack(sqs)[t_of, np.arange(n), f_of], draw_offsets(rng, n))
        ob = oracle.OracleBatch(n, dense=dense, max_episode_steps=max_steps)
        ob.params["success_threshold"] = success_threshold
        self.obs0 = ob.reset_predrawn(self.jp0, self.size, self.mass, self.fric, self.pos)
        points = [_decisions(self.obs0, ob.env["op"], self.size)]
        self.steps = []
        for t in range(K):
            oo, rr, cc, te, tr, nc = ob.step(self.acts[t])
            self.steps.append((oo, rr, cc, te, tr, nc, ob.env["op"].copy()))
            points.append(_decisions(oo, ob.env["op"], self.size))
        self.coverage = _cov_sum(points)
        self.flips = sum(int(((in_band(sq, thr) & ((c.sum(1) == success_threshold) | (c.sum(1) == success_threshold - 1))[:, None])).sum())
                         for sq, thr, c in points[1:])


def _group_table(sizes):
    return np.concatenate([oracle.make_group(None, object_size=float(s)) for s in sizes])


class GroupRun:
    """Env i belongs to group i % G, every group has its own fixed size; auto-reset after M steps (the loop bound) or on
    success.  Per-step oracle records from one-step rollouts: the step's own outputs (a copy of the pre-step state stepped
    without reset) and the state after the step and a possible reset."""

    def __init__(self, n, G, K, M, seed, success_threshold, policy_kind=0, sizes=None, acts=None):
        self.n, self.G, self.K, self.M, self.seed, self.kind = n, G, K, M, seed, policy_kind
        self.sizes = np.full(G, 0.05) if sizes is None else sizes
        self.groups = _group_table(self.sizes)
        self.acts = acts
        ob = oracle.OracleBatch(n, dense=True, max_episode_steps=M)
        ob.params["success_threshold"] = success_threshold
        self.obs0 = _oracle_initial_reset(ob, self.groups, seed)
        size_env = self.sizes[np.arange(n) % G]
        self.points = [_decisions(self.obs0, ob.env["op"], size_env)]
        self.reset_points = {}                  # (env, episode) -> squared distances at that episode's reset
        sq0 = self.points[0][0]
        for i in range(min(n, G)):
            self.reset_points[(i, 0)] = sq0[i]
        cnt = rs = None
        self.steps = []
        for t in range(K):
            pre = ob.env.copy()
            if policy_kind == 0:
                a = acts[t]
            else:
                a = np.stack([oracle.policy_action(seed, i, int(pre["episode"][i]), int(pre["step_count"][i]), policy_kind)
                              for i in range(n)])
            scratch = oracle.OracleBatch(n, dense=True, max_episode_steps=M)
            scratch.env, scratch.params = pre, ob.params
            so, sr, sc, ste, stru, snc = scratch.step(a)
            cnt, rs = ob.rollout(self.groups, 1, seed, policy_kind=policy_kind, actions=a if policy_kind == 0 else None,
                                 respawn=True, loop_max_steps=M, counters=cnt, ret_sums=rs)
            fin = ob.env["episode"] != pre["episode"]
            post = ob.observation()
            self.steps.append(dict(final=so, term_op=scratch.env["op"].copy(), reward=sr, comps=sc, terminated=ste,
                                   truncated=stru, nc=snc, finished=fin, obs=post, op=ob.env["op"].copy(), episode=ob.env["episode"].copy(),
                                   step_count=ob.env["step_count"].copy()))
            self.points.append(_decisions(so, scratch.env["op"], size_env))
            if fin.any():
                d = _decisions(post[fin], ob.env["op"][fin], size_env[fin])
                self.points.append(d)
                for j, i in enumerate(np.flatnonzero(fin)):
                    if i < G:
                        self.reset_points[(int(i), int(ob.env["episode"][i]))] = d[0][j]
        self.counters, self.ret_sums = cnt, rs
        self.coverage = _cov_sum(self.points)


def tuned_group_run(n, G, K, M, seed, success_threshold, policy_kind=0):
    """Pre-run with every size 0.05 and no early success, tune group g's size to env g (the first env of the group):
    a third of the groups to the state of an in-kernel reset, a third to the initial reset, a third to a step; then the
    run with the tuned sizes at ``success_threshold``."""
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-1.0, 1.0, (K, n, 15)).astype(np.float32) if policy_kind == 0 else None
    pre = GroupRun(n, G, K, M, seed, 6, policy_kind, acts=acts)
    sq = np.empty(G)
    for g in range(G):
        f = int(rng.integers(0, 5))
        later = [ep for (i, ep) in pre.reset_points if i == g and ep > 0]
        if g % 3 == 0 and later:
            sq[g] = pre.reset_points[(g, int(rng.choice(later)))][f]
        elif g % 3 == 1:
            sq[g] = pre.reset_points[(g, 0)][f]
        else:
            s = pre.steps[int(rng.integers(0, K))]
            sq[g] = finger_sq(s["final"][g, :15], s["term_op"][g])[f]
    sizes = tuned_sizes(sq, draw_offsets(rng, G))
    return GroupRun(n, G, K, M, seed, success_threshold, policy_kind, sizes=sizes, acts=acts)



PLAIN_MIN = {"band_contact": 700, "band_free": 1000, "tie": 300}
GROUP_MIN = {"band_contact": 40, "band_free": 60, "tie": 20}


# ---- GPU: every kernel that decides contact, bit for bit against the oracle ---------------------------------------------
@pytest.fixture(scope="module")
def dx():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import dexterous_rl_manipulation_b200 as d
    return d


@pytest.fixture
def kernels():
    """Pin the step kernel ('register', 'tma' narrow tiles, 'tma_wide') and the rollout kernel ('thread', 'split');
    restored afterwards."""
    from dexterous_rl_manipulation_b200 import _lib

    def choose(step="auto", rollout="auto"):
        _lib.set_step_impl("tma" if step == "tma_wide" else step)
        _lib.set_step_tile("wide" if step == "tma_wide" else "narrow" if step == "tma" else "auto")
        _lib.set_rollout_impl(rollout)
    yield choose
    choose()


def _np(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _check_exact_components(got, want):
    """Contact and stability rewards are exact functions of the contact bits: float32 of the oracle's, not a tolerance."""
    assert np.array_equal(_np(got["contact"]), want[:, 1].astype(np.float32))
    assert np.array_equal(_np(got["stability"]), want[:, 3].astype(np.float32))
    for k, j in (("distance", 0), ("closure", 2)):
        np.testing.assert_allclose(_np(got[k]), want[:, j], rtol=1e-6, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("success_threshold", [6, 3])
@pytest.mark.parametrize("n,dense,comps,impl", [(4096 + 77, True, True, "register"), (4096 + 77, True, True, "tma"),
                                                (4096 + 77, False, False, "tma"), (224 * 19 + 3, True, False, "tma_wide"),
                                                (224 * 19 + 3, False, True, "tma_wide"), (4096 + 77, True, False, "register"),
                                                (1, True, True, "auto")])
def test_reset_and_step_on_the_boundary(dx, kernels, n, dense, comps, impl, success_threshold):
    """reset_from_draws and step() without auto-reset: every env's size tuned to one finger at its reset state or at one
    step; observations, flags, counts, object positions and the contact-derived rewards bit for bit."""
    kernels(impl)
    K = 10
    run = PlainRun(max(n, 64), K, dense, success_threshold, seed=n + success_threshold)
    sel = slice(0, n)
    if n > 1:
        assert_coverage(run.coverage, PLAIN_MIN)
        if success_threshold == 3:
            assert run.flips >= 100
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=200, reward_type="dense" if dense else "sparse",
                                    reward_components=comps)
    env._params.success_threshold = success_threshold
    o0, _ = env.reset_from_draws(run.jp0[sel], run.size[sel], run.mass[sel], run.fric[sel], run.pos[sel])
    assert np.array_equal(_np(o0).reshape(n, 45), run.obs0[sel])
    for t in range(K):
        oo, rr, cc, te, tr, nc, op = run.steps[t]
        a = run.acts[t][sel]
        if n == 1:
            obs, rew, ter, tru, info = env.step(a[0])
            assert np.array_equal(obs, oo[0]) and ter == te[0] and tru == tr[0] and info["num_contacts"] == nc[0], t
            assert rew == pytest.approx(rr[0], rel=1e-6, abs=1e-7)
            assert np.array_equal(info["object_position"], op[0])
            comp = info["reward_components"]
            assert np.float32(comp["contact"]) == np.float32(cc[0, 1]), t
            assert np.float32(comp["stability"]) == np.float32(cc[0, 3]), t
            continue
        obs, rew, ter, tru, info = env.step(torch.from_numpy(a).cuda())
        assert np.array_equal(_np(obs), oo[sel]), t
        assert np.array_equal(_np(ter), te[sel]) and np.array_equal(_np(tru), tr[sel]), t
        assert np.array_equal(_np(info["num_contacts"]), nc[sel]), t
        assert np.array_equal(_np(info["object_position"]), op[sel]), t
        np.testing.assert_allclose(_np(rew), rr[sel], rtol=1e-6, atol=1e-7)
        if comps:
            _check_exact_components(info["reward_components"], cc[sel])


@pytest.mark.gpu
@pytest.mark.parametrize("success_threshold", [6, 3])
@pytest.mark.parametrize("zero_copy", [False, True])
def test_step_host_on_the_boundary(dx, kernels, zero_copy, success_threshold):
    """step_host() through the pipelined kernel's host epilogue, with the download copies and zero-copy."""
    kernels("tma")
    n, K = 4096 + 77, 10
    run = PlainRun(n, K, True, success_threshold, seed=77 + success_threshold)
    assert_coverage(run.coverage, PLAIN_MIN)
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=200, reward_type="dense")
    env._params.success_threshold = success_threshold
    env.host_zero_copy = zero_copy
    env.reset_from_draws(run.jp0, run.size, run.mass, run.fric, run.pos)
    for t in range(K):
        oo, rr, _, te, tr, nc, op = run.steps[t]
        obs, rew, ter, tru, info = env.step_host(run.acts[t])
        assert np.array_equal(_np(obs), oo) and np.array_equal(_np(ter), te) and np.array_equal(_np(tru), tr), t
        assert np.array_equal(_np(info["num_contacts"]), nc), t
        np.testing.assert_allclose(_np(rew), rr, rtol=1e-6, atol=1e-7)
    assert np.array_equal(_np(env._op64[:, :n].t()), run.steps[-1][6])


def _group_env(dx, run, success_threshold, **kw):
    cfgs = [dx.CurriculumConfig(object_size=float(s)) for s in run.sizes]
    env = dx.BatchedManipulationEnv(run.n, "cuda", max_episode_steps=run.M, reward_type="dense", respawn=True,
                                    loop_max_steps=run.M, seed=run.seed, groups=cfgs, **kw)
    env._params.success_threshold = success_threshold
    o0, _ = env.reset(seed=run.seed)
    assert np.array_equal(_np(o0), run.obs0)
    return env


def _check_final_state(dx, env, run, full):
    from dexterous_rl_manipulation_b200 import _lib
    n = run.n
    assert np.array_equal(_np(env._op64[:, :n].t()), run.steps[-1]["op"])
    assert np.array_equal(_np(env._episode[:n]).astype(np.uint32), run.steps[-1]["episode"])
    assert np.array_equal(_np(env._step_count[:n]), run.steps[-1]["step_count"])
    cnt = _np(env.counters)
    cols = (list(range(16)) + [_lib.CNT_SUM_STEPS_SQ] if full else
            [_lib.CNT_EPISODES, _lib.CNT_SUCCESSES, _lib.CNT_SUM_STEPS, _lib.CNT_SUM_FINAL_CONTACTS, _lib.CNT_SUM_STEPS_SQ])
    assert np.array_equal(cnt[:, cols], run.counters[:, cols])
    if full:
        np.testing.assert_allclose(_np(env.ret_sums), run.ret_sums, rtol=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("success_threshold", [6, 3])
@pytest.mark.parametrize("impl,mode,track", [("register", "same", "counts"), ("register", "same", "full"),
                                             ("tma", "same", "counts"), ("tma", "same", "full"),
                                             ("tma_wide", "same", "counts"), ("register", "final", "full"),
                                             ("tma", "final", "counts")])
def test_auto_reset_step_on_the_boundary(dx, kernels, impl, mode, track, success_threshold):
    """Same-step auto-reset (in-kernel reset of both step kernels), counts-only and full tracking, and the two-pass
    final_observation step: 256 groups, each size tuned to an in-kernel reset state, the initial reset or a step."""
    kernels(impl)
    run = tuned_group_run(4096 + 77, 256, 16, 6, 11, success_threshold)
    assert_coverage(run.coverage, GROUP_MIN)
    env = _group_env(dx, run, success_threshold, auto_reset=True, track_episodes=track == "full", reward_components=True,
                     final_observation=mode == "final")
    for t, s in enumerate(run.steps):
        obs, rew, ter, tru, info = env.step(torch.from_numpy(run.acts[t]).cuda())
        assert np.array_equal(_np(obs), s["obs"]), t
        assert np.array_equal(_np(ter), s["terminated"]) and np.array_equal(_np(tru), s["truncated"]), t
        assert np.array_equal(_np(info["num_contacts"]), s["nc"]), t
        assert np.array_equal(_np(info["finished"]), s["finished"]), t
        np.testing.assert_allclose(_np(rew), s["reward"], rtol=1e-6, atol=1e-7)
        _check_exact_components(info["reward_components"], s["comps"])
        if mode == "final":
            fin = s["finished"]
            assert np.array_equal(_np(info["final_observation"])[fin], s["final"][fin]), t
    _check_final_state(dx, env, run, track == "full")


@pytest.mark.gpu
@pytest.mark.parametrize("success_threshold", [6, 3])
@pytest.mark.parametrize("impl", ["register", "tma"])
def test_next_step_reset_on_the_boundary(dx, kernels, impl, success_threshold):
    """autoreset_mode="next_step": a step that ends an episode returns its terminal observation, the env's next call
    resets it (the NEXT step instantiations and the reset they defer)."""
    kernels(impl)
    run = tuned_group_run(4096 + 77, 256, 16, 6, 11, success_threshold)
    assert_coverage(run.coverage, GROUP_MIN)
    env = _group_env(dx, run, success_threshold, auto_reset=True, autoreset_mode="next_step", track_episodes=True,
                     reward_components=True)
    n = run.n
    ptr = np.zeros(n, np.int64)                 # physical step each env takes next
    pending = np.zeros(n, bool)
    rows = np.arange(n)
    calls = 0
    while ptr.min() < run.K:
        a = run.acts[np.minimum(ptr, run.K - 1), rows]
        out = env.step(torch.from_numpy(a).cuda())
        obs, rew, ter, tru = (_np(x) for x in out[:4])
        info = out[4]
        live = ~pending & (ptr < run.K)
        p = np.minimum(ptr, run.K - 1)
        final = np.stack([run.steps[p[i]]["final"][i] for i in range(n)])
        reward = np.array([run.steps[p[i]]["reward"][i] for i in range(n)])
        want = {k: np.array([run.steps[p[i]][k][i] for i in range(n)]) for k in ("terminated", "truncated", "nc", "finished")}
        comps = np.stack([run.steps[p[i]]["comps"][i] for i in range(n)])
        assert np.array_equal(obs[live], final[live]), calls
        assert np.array_equal(ter[live], want["terminated"][live]) and np.array_equal(tru[live], want["truncated"][live]), calls
        assert np.array_equal(_np(info["num_contacts"])[live], want["nc"][live]), calls
        assert np.array_equal(_np(info["finished"])[live], want["finished"][live]), calls
        np.testing.assert_allclose(rew[live], reward[live], rtol=1e-6, atol=1e-7)
        rc = {k: _np(v)[live] for k, v in info["reward_components"].items()}
        _check_exact_components(rc, comps[live])
        # the reset call: the first observation of the next episode, reward 0, both flags False
        reset = pending
        post = np.stack([run.steps[max(ptr[i] - 1, 0)]["obs"][i] for i in range(n)])
        assert np.array_equal(obs[reset], post[reset]), calls
        assert not ter[reset].any() and not tru[reset].any() and (rew[reset] == 0).all(), calls
        pending = live & want["finished"]
        ptr[live] += 1
        calls += 1
    assert calls > run.K


@pytest.mark.gpu
@pytest.mark.parametrize("success_threshold", [6, 3])
@pytest.mark.parametrize("policy,rollout_impl", [("random", "thread"), ("heuristic", "thread"), ("random", "split"),
                                                 ("heuristic", "split")])
def test_rollout_on_the_boundary(dx, kernels, policy, rollout_impl, success_threshold):
    """The fused rollout, one thread per env (rollout_kernel) and 5 lanes per env (rollout_split_kernel, split_contact):
    one-step launches compared with the oracle's one-step rollouts after every step, then counters and returns."""
    kernels(rollout=rollout_impl)
    kind = 1 if policy == "random" else 2
    run = tuned_group_run(4096 + 77, 256, 16, 6, 13, success_threshold, policy_kind=kind)
    assert_coverage(run.coverage, GROUP_MIN)
    env = _group_env(dx, run, success_threshold, track_episodes=True)
    n = run.n
    for t, s in enumerate(run.steps):
        env.rollout(1, policy=policy, respawn=True, loop_max_steps=run.M)
        assert np.array_equal(_np(env._obs[:, :n].t()), s["obs"]), t
        assert np.array_equal(_np(env._op64[:, :n].t()), s["op"]), t
    _check_final_state(dx, env, run, True)


@pytest.mark.gpu
@pytest.mark.parametrize("success_threshold", [6, 3])
def test_recorded_rollout_on_the_boundary(dx, kernels, success_threshold):
    """enable_trajectory + rollout(): every recorded row's observation (contact rows included), reward, flags and
    terminal observation against the oracle's per-step record."""
    kernels()
    run = tuned_group_run(4096 + 77, 256, 16, 6, 17, success_threshold, policy_kind=2)
    assert_coverage(run.coverage, GROUP_MIN)
    env = _group_env(dx, run, success_threshold, track_episodes=True)
    env.enable_trajectory(run.K, final_observation=True)
    env.rollout(run.K, policy="heuristic", respawn=True, loop_max_steps=run.M)
    tr = {k: _np(v) for k, v in env.trajectory.items()}
    for t, s in enumerate(run.steps):
        assert np.array_equal(tr["obs"][t], s["obs"]), t
        assert np.array_equal(tr["terminated"][t], s["terminated"]) and np.array_equal(tr["truncated"][t], s["truncated"]), t
        assert np.array_equal(tr["finished"][t], s["finished"]), t
        fin = s["finished"]
        assert np.array_equal(tr["final_observation"][t][fin], s["final"][fin]), t
        np.testing.assert_allclose(tr["reward"][t], s["reward"], rtol=1e-6, atol=1e-7)
    _check_final_state(dx, env, run, True)
