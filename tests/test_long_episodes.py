"""Tracked episodes up to the longest the library accepts (5,242 steps) against an oracle that keeps every count.

The packed per-env summary EpStats (csrc/dexsim_core.cuh) holds a 16-bit sum of the per-step contact counts, a 17-bit
sum of squares (5,242 steps of five contacts give 131,050 of 131,071), a 5-bit sum of the first five counts, a 3-bit
maximum and a 15-bit ring of the last five, and saturates when a tracked env is stepped past the limit without a
reset.  Every failure label of such an episode comes from it; an exact variance tie is decided on the recorded
history by resolve_ties_kernel, whose pairwise sum recurses 7 frames deep at these lengths.  These tests drive every
field to its edge and compare it with counts the test records itself.

CPU tests need no device; the GPU tests share one oracle rollout per configuration (module-scoped)."""
import ctypes as C

import numpy as np
import pytest

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib
from oracle import oracle

LONGEST = 5242                                  # EPSTATS_MAX_STEPS: the longest tracked episode the library accepts
# (max_episode_steps, loop_max_steps): truncation ends the 5,242nd step, or only the caller's loop bound does
BOUNDS = {"truncation": (5241, LONGEST), "loop": (100000, LONGEST)}
# (success_threshold, success_is_terminated): (a) no episode can terminate, every one runs to the bound and the sums
# grow large; (b) five contacts end an episode early as a failure, so long episodes reach the variance / trend branches
REGIMES = {"a": (6, True), "b": (5, False)}
CHECKPOINTS = (1023, 1024, 1025, 4096, 5241, 5242, 5542)
N_GPU = 4096 + 77                               # ragged, at least two 224-env wide tiles; <= 8192: split rollout eligible
SEED, GID0 = 1, 3

# multisets of counts with n * sum(c^2) - sum(c)^2 == 2 n^2 (np.var exactly 2) and a mean that is not a dyadic
# rational (tests/test_cpu_abi_and_host.py); repetition keeps them exact ties
M18 = [0, 0, 0, 0, 0, 1, 1, 1, 2, 2, 2, 2, 2, 2, 3, 3, 4, 5]
M27 = [0, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 3, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5]


def _multiset(k):
    """Counts of 0..5 taken k[j] times each."""
    return [j for j in range(6) for _ in range(k[j])]


# exact variance-2 ties at the lengths around the 1,024 and 4,096 boundaries.  1,023 is square-free, so the mean is an
# integer; 1,024 and 4,096 are powers of two, so the mean is dyadic (17/16, 33/32): np.var is exact there and only
# "not above 2" occurs.  1,025's mean is 6/5 and NumPy's rounding decides.
TIES = {
    "m27x5": M27 * 5, "m27x7": M27 * 7,                                  # 135, 189: both sides (the existing test)
    "m18x57": M18 * 57, "m27x38": M27 * 38,                              # 1,026
    "m18x100": M18 * 100, "m27x100": M27 * 100, "m18x200": M18 * 200,   # 1,800, 2,700, 3,600
    "m18x291": M18 * 291, "m27x194": M27 * 194,                          # 5,238: the longest below the limit
    "n1023": _multiset((680, 3, 2, 337, 0, 1)), "n1024": _multiset((650, 1, 34, 338, 0, 1)),
    "n1025": _multiset((585, 1, 94, 340, 4, 1)), "n4096": _multiset((2666, 1, 66, 1362, 0, 1)),
}
# multisets whose random permutations land on both sides of the threshold (seed 5, 120 permutations each; at 1,026
# entries about 1 in 200 lands above).  The others only ever give "not above 2": the repeated m18 (mean 5/3) above 1,000
# entries in 2,000 permutations each, and the exact 1,023 / 1,024 / 4,096.
TIES_BOTH_SIDES = {"m27x5", "m27x7", "m27x38", "m27x100", "m27x194", "n1025"}


def _code(label):
    return 255 if label < 0 else int(label)


def _labels(counts, steps, final, max_steps, thr, success=False):
    a, b, _ = oracle.classify(success, steps, final, final, counts, max_steps=max_steps, threshold=thr)
    return _code(a), _code(b)


def _summary_kw(c):
    c = np.asarray(c, np.int64)
    return dict(hist_len=len(c), max_count=int(c.max()), sum_counts=int(c.sum()), sum_sq_counts=int((c * c).sum()),
                first5_sum=int(c[:5].sum()), last5_sum=int(c[-5:].sum()))


def _epstats_expected(counts, start, now):
    """EpStats fields of every env's current episode from the recorded counts: counts[t, i] is the count of step t,
    env i's episode began at step start[i], and `now` steps have run.  Exact (no saturation)."""
    n = counts.shape[1]
    idx = np.arange(n)
    c = np.where(np.arange(now)[:, None] >= start[None, :], counts[:now], 0)         # uint8: [now, n] stays small
    hits = [(c == v).sum(0, dtype=np.int64) for v in range(6)]
    out = dict(sum=sum(v * hits[v] for v in range(6)), sq=sum(v * v * hits[v] for v in range(6)), max=c.max(0))
    first5 = np.zeros(n, np.int64)
    ring = np.zeros(n, np.int64)
    for k in range(5):
        first = start + k
        first5 += np.where(first < now, counts[np.minimum(first, now - 1), idx], 0)
        last = now - 1 - k
        ring |= np.where(last >= start, counts[max(last, 0), idx].astype(np.int64) << (3 * k), 0)
    out.update(first5=first5, ring=ring)
    return out


def _epstats_decode(ep_stats, n):
    w = ep_stats[:, :n].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    return dict(sum=w[0] & 0xFFFF, first5=(w[0] >> 16) & 0x1F, max=(w[0] >> 21) & 0x7, sq=w[1] & 0x1FFFF, ring=w[1] >> 17)


class OracleRun:
    """The oracle's auto-reset rollout with the in-kernel random policy, one step per call, with one counter group per
    env: the counter deltas of a step attribute each finished episode (steps, final contacts, labels, return) to its
    env.  The per-step contact counts are recorded here -- num_contacts for an env that goes on, the final contacts for
    one that finished (the oracle has reset it already) -- so nothing below relies on the oracle's own history."""

    def __init__(self, n, steps, thr, sit, max_episode_steps, loop_max, checkpoints=(), seed=SEED, gid0=GID0):
        self.n, self.steps, self.thr, self.loop_max = n, steps, thr, loop_max
        grp = oracle.make_group(dx.CurriculumConfig())
        ob = oracle.OracleBatch(n, dense=True, max_episode_steps=max_episode_steps)
        ob.params["success_threshold"] = thr
        draws = [oracle.reset_draws(seed, gid0 + i, 0, grp) for i in range(n)]
        self.obs0 = ob.reset_predrawn(np.stack([d[0] for d in draws]), np.array([d[1] for d in draws]),
                                      np.array([d[2] for d in draws]), np.array([d[3] for d in draws]),
                                      np.stack([d[4] for d in draws]))
        groups, goe = np.repeat(grp, n), np.arange(n, dtype=np.uint16)
        cnt, rs = np.zeros((n, oracle.NCOUNTERS), np.int64), np.zeros((n, 2))
        self.counts = np.zeros((steps, n), np.uint8)
        start = np.zeros(n, np.int64)
        counters, ret_sums = np.zeros(oracle.NCOUNTERS, np.int64), np.zeros(2)
        eps, self.snap, self.hist_matches = [], {}, {}
        for t in range(steps):
            episode = ob.env["episode"].copy()
            cnt[:] = 0
            rs[:] = 0
            ob.rollout(groups, 1, seed, policy_kind=1, respawn=True, success_is_terminated=sit, loop_max_steps=loop_max,
                       env_gid0=gid0, group_of_env=goe, counters=cnt, ret_sums=rs, threads=8)
            done = cnt[:, 0] > 0
            assert cnt[:, 0].max() <= 1
            self.counts[t] = np.where(done, cnt[:, 3], ob.env["num_contacts"])
            i = np.nonzero(done)[0]
            if len(i):
                la, lb = cnt[i, 4:10], cnt[i, 10:16]
                eps.append(dict(env=i, episode=episode[i], steps=cnt[i, 2], success=cnt[i, 1], final=cnt[i, 3],
                                la=np.where(la.any(1), la.argmax(1), 255), lb=np.where(lb.any(1), lb.argmax(1), 255),
                                ret=rs[i, 0], t_end=np.full(len(i), t), start=start[i]))
                assert np.array_equal(start[i] + cnt[i, 2], np.full(len(i), t + 1))
                start[i] = t + 1
            counters += cnt.sum(0)
            ret_sums += rs.sum(0)
            if t + 1 in checkpoints:
                assert np.array_equal(ob.env["ep_steps"], t + 1 - start)
                self.snap[t + 1] = dict(obs=ob.observation(), op=ob.env["op"].copy(), step_count=ob.env["step_count"].copy(),
                                        episode=ob.env["episode"].copy(), ep_return=ob.env["ep_return"].copy(),
                                        start=start.copy(), counters=counters.copy(), ret_sums=ret_sums.copy(),
                                        stats=_epstats_expected(self.counts, start, t + 1))
                self.hist_matches[t + 1] = self._hist_matches(ob, start, t + 1)
        self.eps = {k: np.concatenate([e[k] for e in eps]) for k in eps[0]} if eps else {}
        self.counters, self.ret_sums, self.start = counters, ret_sums, start
        # reference labels of every finished episode: the oracle's classifiers on its full recorded history
        self.eps["ref"] = np.array([_labels(self.episode_counts(q), int(self.eps["steps"][q]), int(self.eps["final"][q]),
                                            loop_max, thr, bool(self.eps["success"][q])) for q in range(len(self.eps["env"]))])

    def episode_counts(self, q):
        return self.counts[self.eps["start"][q]:self.eps["t_end"][q] + 1, self.eps["env"][q]]

    def _hist_matches(self, ob, start, now):
        return all(np.array_equal(ob.env["hist"][i, :now - start[i]], self.counts[start[i]:now, i]) for i in range(self.n))

    def long_early(self):
        """Finished episodes longer than 1,024 steps that ended before the bound."""
        return int(((self.eps["steps"] > 1024) & (self.eps["steps"] < self.loop_max)).sum())


# ---------------------------------------------------------------------------------------------------- CPU, no device
def test_oracle_labels_long_episodes_use_the_whole_history():
    """The oracle's labels of episodes up to 5,242 steps are those of both classifiers on every count of the episode,
    and its history is the episode's counts.  The configuration contains episodes whose labels from their first 1,024
    counts differ from those on the full history: an oracle that cut its history there fails this test by a label."""
    n, steps, thr = 4096, 6000, 5
    run = OracleRun(n, steps, thr, False, *BOUNDS["truncation"], checkpoints=(1024, 4096, steps))
    e = run.eps
    assert np.array_equal(e["la"], e["ref"][:, 0]) and np.array_equal(e["lb"], e["ref"][:, 1])
    assert all(run.hist_matches.values())
    cut = 0
    for q in np.nonzero(e["steps"] > 1024)[0]:
        c = run.episode_counts(q)
        steps_q, fin = int(e["steps"][q]), int(e["final"][q])
        assert _lib.classify_counts(False, steps_q, fin, fin, c, max_steps=LONGEST, success_threshold=thr) == tuple(e["ref"][q])
        cut += _labels(c[:1024], steps_q, fin, LONGEST, thr) != tuple(e["ref"][q])
    assert run.long_early() >= 24, run.long_early()
    assert cut >= 1                       # the history past 1,024 steps decides some label
    assert (e["steps"] == LONGEST).sum() > 1000


def test_variance_ties_follow_numpy_rounding_at_long_lengths():
    """Exact variance-2 ties of up to 5,238 counts (NumPy's pairwise sum recurses 6 levels): on random permutations
    the host classifier with the history and the oracle's np.var land on the side of 2.0 that np.var of the
    Python-int list lands on, and give the reference labels."""
    rng = np.random.default_rng(5)
    thr = 6
    for name, base in TIES.items():
        n_ = len(base)
        seen = set()
        for _ in range(120):
            c = rng.permutation(np.array(base, np.int64))
            if c[-1] == 0:                         # keep "object dropped" from deciding before the variance
                j = np.flatnonzero(c)[-1]
                c[[j, -1]] = c[[-1, j]]
            S, Q = int(c.sum()), int((c * c).sum())
            assert n_ * Q - S * S == 2 * n_ * n_
            v = float(np.var([int(x) for x in c]))
            assert (oracle.np_var_counts(c) > 2.0) == (v > 2.0), (name, v)
            fin = int(c[-1])
            a, b, tie = dx.classify_summary(False, n_, fin, fin, max_steps=10 ** 6, success_threshold=thr, counts=c,
                                            **_summary_kw(c))
            assert tie == 2
            assert (a, b) == _labels(c, n_, fin, 10 ** 6, thr), name
            assert (dx.LABELS_METRICS[a] == "unstable_contacts") == (v > 2.0), (name, v)
            seen.add(v > 2.0)
        assert seen == ({False, True} if name in TIES_BOTH_SIDES else {False}), (name, n_, seen)


def test_all_five_history_of_the_longest_episode():
    """5,242 steps of five contacts (sum 26,210, sum of squares 131,050 of the 17-bit field's 131,071): the summary
    path gives the labels of the history path, at the bound and one step before it."""
    c = np.full(LONGEST, 5, np.uint8)
    kw = _summary_kw(c)
    assert kw["sum_counts"] == 26210 and kw["sum_sq_counts"] == 131050
    for max_steps in (LONGEST, LONGEST + 1):
        for fin in (5, 0):
            want = _labels(c, LONGEST, fin, max_steps, 6)
            assert dx.classify_summary(False, LONGEST, fin, fin, max_steps=max_steps, success_threshold=6, **kw)[:2] == want
            assert dx.classify_counts(False, LONGEST, fin, fin, c, max_steps=max_steps, success_threshold=6) == want


def test_oracle_refuses_an_episode_longer_than_its_history():
    ob = oracle.OracleBatch(2, dense=True, max_episode_steps=100000)
    ob.params["success_threshold"] = 6                # never terminates
    with pytest.raises(RuntimeError, match="history"):
        ob.rollout(oracle.make_group(None), oracle.HIST_MAX + 1, 1, policy_kind=1, loop_max_steps=100000)


# -------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch


@pytest.fixture(scope="module")
def oracle_runs():
    """One oracle rollout per (bound, regime), shared by the API-mode and fused-rollout tests."""
    cache = {}

    def get(bound, regime):
        if (bound, regime) not in cache:
            thr, sit = REGIMES[regime]
            cache[bound, regime] = OracleRun(N_GPU, CHECKPOINTS[-1], thr, sit, *BOUNDS[bound], checkpoints=CHECKPOINTS)
        return cache[bound, regime]
    return get


@pytest.fixture
def step_kernel():
    """Pin dexsim_step to one kernel: 'register', 'tma' (128-env tiles) or 'tma_wide' (224-env tiles)."""
    def choose(impl):
        _lib.set_step_impl("tma" if impl == "tma_wide" else impl)
        _lib.set_step_tile("wide" if impl == "tma_wide" else "narrow" if impl == "tma" else "auto")
    yield choose
    _lib.set_step_impl("auto")
    _lib.set_step_tile("auto")


def _env(cuda, bound, regime, **kw):
    mes, loop_max = BOUNDS[bound]
    thr, sit = REGIMES[regime]
    env = dx.BatchedManipulationEnv(N_GPU, "cuda", max_episode_steps=mes, reward_type="dense", loop_max_steps=loop_max,
                                    success_is_terminated=sit, track_episodes=True, groups=[dx.CurriculumConfig()],
                                    seed=SEED, env_gid0=GID0, **kw)
    env._params.success_threshold = thr
    env.reset(seed=SEED)
    return env


def _check_checkpoint(env, run, t):
    n = run.n
    s = run.snap[t]
    assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), s["obs"]), t
    assert np.array_equal(env._op64[:, :n].t().cpu().numpy(), s["op"]), t
    assert np.array_equal(env._step_count[:n].cpu().numpy(), s["step_count"]), t
    assert np.array_equal(env._episode[:n].cpu().numpy().astype(np.uint32), s["episode"]), t
    np.testing.assert_allclose(env._ep_return[:n].cpu().numpy(), s["ep_return"], rtol=1e-12, atol=1e-12)
    got, want = _epstats_decode(env._ep_stats, n), s["stats"]
    for field in ("sum", "sq", "first5", "max", "ring"):
        assert np.array_equal(got[field], want[field]), (t, field)
    cols = [k for k in range(dx.NCOUNTERS) if k != dx.CNT_VAR_TIES]      # the oracle does not keep the tie counter
    assert np.array_equal(env.counters.cpu().numpy().sum(0)[cols], s["counters"][cols]), t
    np.testing.assert_allclose(env.ret_sums.cpu().numpy().sum(0), s["ret_sums"], rtol=1e-9)
    return int(want["sq"].max())


def _check_edges(run, regime, max_sq):
    if regime == "a":
        assert max_sq >= 1 << 16, max_sq                 # the 17th bit of the sum of squares is in use
        assert (run.eps["steps"] == LONGEST).all() and len(run.eps["steps"]) >= run.n
    else:
        assert run.long_early() >= 24, run.long_early()  # long episodes that end early take the history's branches


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["a", "b"])
@pytest.mark.parametrize("bound", ["truncation", "loop"])
@pytest.mark.parametrize("impl", ["register", "tma", "tma_wide"])
def test_api_stepping_long_tracked_episodes(cuda, oracle_runs, step_kernel, impl, bound, regime):
    """Auto-reset stepping with full tracking, fed with the exposed Philox policy, against the oracle at steps 1,023 ..
    5,242 and 300 steps past the bound: every EpStats field, the state, the counters."""
    run = oracle_runs(bound, regime)
    step_kernel(impl)
    env = _env(cuda, bound, regime, auto_reset=True, respawn=True)
    n = run.n
    assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), run.obs0)
    act = cuda.zeros(15, env.ld, device="cuda")
    max_sq = 0
    for t in range(1, CHECKPOINTS[-1] + 1):
        _lib.check(env._lib.dexsim_fill_policy_actions(C.byref(env._state), C.byref(env._params), 1, act.data_ptr(),
                                                       env._stream()), "dexsim_fill_policy_actions")
        env.step(act[:, :n].t().contiguous())
        if t in run.snap:
            max_sq = max(max_sq, _check_checkpoint(env, run, t))
    _check_edges(run, regime, max_sq)


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["a", "b"])
@pytest.mark.parametrize("bound", ["truncation", "loop"])
@pytest.mark.parametrize("kernel", ["thread", "split"])
def test_fused_rollout_long_tracked_episodes(cuda, oracle_runs, kernel, bound, regime):
    """Both fused-rollout kernels, launched in chunks that end at the checkpoints (episodes straddle launches and the
    1,024-step boundary): history rows, every episode record and the counters against the oracle."""
    run = oracle_runs(bound, regime)
    env = _env(cuda, bound, regime)
    n, K = run.n, CHECKPOINTS[-1]
    env.enable_episode_log(4 * n)
    env.enable_history(K)
    max_sq, done = 0, 0
    try:
        _lib.set_rollout_impl(kernel)
        for t in CHECKPOINTS:
            env.rollout(t - done, policy="random", respawn=True, loop_max_steps=BOUNDS[bound][1],
                        success_is_terminated=REGIMES[regime][1])
            done = t
            max_sq = max(max_sq, _check_checkpoint(env, run, t))
    finally:
        _lib.set_rollout_impl("auto")
    assert np.array_equal(env._hist[:K, :n].cpu().numpy(), run.counts)
    log = env.read_episode_log()
    assert env.episode_log_overflow == 0
    e = run.eps
    order = np.lexsort((e["env"], e["t_end"]))                   # read_episode_log's order: (t_end, env_gid)
    assert len(log) == len(order)
    assert np.array_equal(log["env_gid"], (e["env"][order] + GID0).astype(np.uint32))
    assert np.array_equal(log["episode"], e["episode"][order])
    assert np.array_equal(log["steps"], e["steps"][order]) and np.array_equal(log["t_end"], e["t_end"][order])
    assert np.array_equal(log["final_contacts"], e["final"][order]) and np.array_equal(log["success"], e["success"][order])
    assert np.array_equal(log["label_metrics"], e["ref"][order, 0]) and np.array_equal(log["label_taxonomy"], e["ref"][order, 1])
    np.testing.assert_allclose(log["episode_reward"], e["ret"][order], rtol=1e-12)
    assert not np.any(log["var_tie"] == 1)
    _check_edges(run, regime, max_sq)


@pytest.mark.gpu
def test_device_resolves_variance_ties_of_long_histories(cuda):
    """Episode records flagged with an exact variance tie (var_tie == 1) over histories of 135 .. 5,238 counts,
    injected into the log and history of a rollout: resolve_ties_kernel (a 7-frame-deep pairwise sum at 5,238) decides
    each one with np.var's arithmetic, moves the label counters by exactly the relabelled records, and leaves the one
    record whose history was not recorded alone."""
    rng = np.random.default_rng(11)
    thr, hist_steps, max_steps = 6, 5300, 5241
    picks = []                                               # (name, counts): one permutation per side where both exist
    for name, base in TIES.items():
        want = {True, False} if name in TIES_BOTH_SIDES else {False}
        got = {}
        while set(got) != want:
            c = rng.permutation(np.array(base, np.uint8))
            if c[-1] != 0:
                got.setdefault(float(np.var([int(x) for x in c])) > 2.0, c)
        picks += [(name, got[k]) for k in sorted(got)]
    n = len(picks) + 1
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense", track_episodes=True,
                                    seed=3, env_gid0=GID0)
    env._params.success_threshold = thr
    env.reset(seed=3)
    env.enable_episode_log(n)
    env.enable_history(hist_steps)
    hist = np.zeros((hist_steps, env.ld), np.uint8)
    rec = np.zeros(n, _lib.EPISODE_RECORD_DTYPE)
    before = np.zeros((1, dx.NCOUNTERS), np.int64)
    expect = []
    for i, (name, c) in enumerate(picks + [("unrecorded", picks[-1][1])]):
        L, fin = len(c), int(c[-1])
        t_end = L - 1 if i < len(picks) else hist_steps     # the last record's episode ended past the recorded rows
        if i < len(picks):
            hist[:L, i] = c
        a0, b0, tie = dx.classify_summary(False, L, fin, fin, max_steps=max_steps, success_threshold=thr, **_summary_kw(c))
        assert tie == 1                                      # what the rollout kernel would have logged and counted
        rec[i] = (GID0 + i, 0, L, 0, fin, a0, b0, 0.0, t_end, 1)
        before[0, dx.CNT_LABEL_METRICS + a0] += 1
        before[0, dx.CNT_LABEL_TAXONOMY + b0] += 1
        before[0, dx.CNT_VAR_TIES] += 1
        expect.append(_labels(c, L, fin, max_steps, thr) if i < len(picks) else (a0, b0))
    env._hist.copy_(cuda.from_numpy(hist))
    env._ep_log.copy_(cuda.from_numpy(rec.view(np.uint8)))
    env._ep_log_count.fill_(n)
    env.counters.copy_(cuda.from_numpy(before))
    env._rollout_steps = hist_steps                          # the rollout's own step writes no history row
    env.rollout(1, policy="random")                          # no episode ends in one step
    out = env.read_episode_log(sort=False)
    assert len(out) == n
    assert np.array_equal(out["var_tie"], [2] * len(picks) + [1])
    assert [tuple(int(x) for x in r) for r in out[["label_metrics", "label_taxonomy"]]] == expect
    for i, (name, c) in enumerate(picks):
        v = float(np.var([int(x) for x in c]))
        assert (dx.LABELS_METRICS[out["label_metrics"][i]] == "unstable_contacts") == (v > 2.0), name
    after = before.copy()
    for i in range(len(picks)):
        for base, old, new in ((dx.CNT_LABEL_METRICS, rec["label_metrics"][i], out["label_metrics"][i]),
                               (dx.CNT_LABEL_TAXONOMY, rec["label_taxonomy"][i], out["label_taxonomy"][i])):
            after[0, base + old] -= 1
            after[0, base + new] += 1
        after[0, dx.CNT_VAR_TIES] -= 1
    assert np.array_equal(env.counters.cpu().numpy(), after)
    flipped = [name for i, (name, c) in enumerate(picks) if out["label_metrics"][i] != rec["label_metrics"][i]]
    assert any(len(TIES[name]) > 1024 for name in flipped), flipped    # ties longer than the old history, resolved up


@pytest.mark.gpu
def test_epstats_saturate_instead_of_wrapping(cuda):
    """A tracked env stepped far past the limit without a reset: the sum of squares stops at 0x1FFFF and the sum at
    0xFFFF, the ring, maximum and first five stay exact.  Env 0 holds five contacts from the first step (a large object
    and a zero action), so it reaches 131,050 exactly at step 5,242 and both saturations later."""
    n, thr, steps = 4096, 6, 13200
    checkpoints = (5242, 5243, 7000, 13107, 13108, steps)
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=5241, reward_type="dense", auto_reset=False,
                                    track_episodes=True, seed=SEED, env_gid0=GID0)
    env._params.success_threshold = thr
    env.reset(seed=SEED)
    jp0 = env._obs[:15, :n].t().cpu().numpy().copy()
    size, mass, fric = (a[:n].cpu().numpy().copy() for a in (env._size, env._mass, env._friction))
    pos = env._obs[30:33, :n].t().cpu().numpy().copy()
    jp0[0], size[0] = 0.0, 0.4                               # every point of the workspace is within 1.5 * 0.4 of the tips
    env.reset_from_draws(jp0, size, mass, fric, pos)
    ob = oracle.OracleBatch(n, dense=True, max_episode_steps=5241)
    ob.params["success_threshold"] = thr
    assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), ob.reset_predrawn(jp0, size, mass, fric, pos))
    act = cuda.zeros(15, env.ld, device="cuda")
    counts = np.zeros((steps, n), np.uint8)
    for t in range(steps):
        _lib.check(env._lib.dexsim_fill_policy_actions(C.byref(env._state), C.byref(env._params), 1, act.data_ptr(),
                                                       env._stream()), "dexsim_fill_policy_actions")
        act[:, 0] = 0.0
        a = act[:, :n].t().contiguous()
        env.step(a)
        counts[t] = ob.step(a.cpu().numpy(), threads=8)[5]
        if t + 1 in checkpoints:
            now = t + 1
            assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), ob.observation()), now
            want = _epstats_expected(counts, np.zeros(n, np.int64), now)
            got = _epstats_decode(env._ep_stats, n)
            assert np.array_equal(got["sq"], np.minimum(want["sq"], 0x1FFFF)), now
            assert np.array_equal(got["sum"], np.minimum(want["sum"], 0xFFFF)), now
            for field in ("ring", "max", "first5"):
                assert np.array_equal(got[field], want[field]), (now, field)
            if now == LONGEST:
                assert want["sq"][0] == 131050 and got["sq"][0] == 131050
            if now == 13107:
                assert want["sum"][0] == 0xFFFF
    assert (want["sq"] > 0x1FFFF).sum() > 1 and want["sum"][0] > 0xFFFF, (int(want["sq"].max()), int(want["sum"][0]))
