"""Group tables of 5 to 256 rows and explicit env -> group maps, through every kernel that reads them.

Every kernel that resets an env or counts an episode reads the group table ``DexsimGroup[num_groups]`` at the env's
row: ``group_of_env[i]``, or ``(uint32)(env_gid0 + i) % num_groups`` without a map.  The kernels switch code paths on
the group count: the pipelined step kernel stages its counters in shared memory up to 16 groups, the register step
kernel, ``finish_reset_kernel`` and the fused rollout up to 64 (the rollout stages the table too, and its MLP weights
sit behind that staged area), and the 5-lane rollout, ``resolve_ties_kernel`` and ``reset_philox_kernel`` always work
in global memory with their own copy of the index formula.  The tables here make every row distinguishable (size,
mass, friction, ranges, spawn box, dynamics noise on rows either side of the thresholds), so a kernel that reads or
counts into the wrong row changes the state or the counters.

Group counts 5, 16, 17, 64, 65, 255 and 256 sit either side of both staging limits, at the ABI maximum, and at 255,
where the 2^32 wrap of the global id changes ``gid % G``.  Maps: the default map with ``env_gid0 = 2^32 - n/2`` (the
batch crosses the wrap), a random explicit map, and a skewed one (most envs in the last group, several groups empty).

The references: the oracle's rollout (``oracle/dexsim_oracle.c``) given the same table, map and ``env_gid0``; the
oracle's reset draws; and a derived bound on the float64 return sums (``_sum_bound``) against the exact ``math.fsum``
of the logged episode returns.

CPU tests need no device: the map validation, the bound helper and the oracle's own sums."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib
from dexterous_rl_manipulation_b200.env import BatchedManipulationEnv, check_group_of_env
from oracle import oracle

U = 2.0 ** -53                    # unit roundoff of float64
M32 = 0xFFFFFFFF
GS = (5, 16, 17, 64, 65, 255, 256)
MAPS = ("default", "random", "skewed")
SIZES = (130, 4096 + 77, 70_001)  # CTAs shrunk to 32 threads; ragged and split-eligible; many CTAs and tiles
EPISODES, SUCCESSES = dx.CNT_EPISODES, dx.CNT_SUCCESSES
STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode")


# ---- tables, maps and the bound ------------------------------------------------------------------------------------
def _noisy_rows(G):
    """Rows with dynamics noise: either side of the 16 and 64 thresholds, and the last."""
    return sorted({r for r in (3, 16, 63, 64, G - 1) if r < G})


def _cfgs(G):
    """G rows that differ in every field a reset reads: fixed size, mass and friction, some ranged, and spawn boxes."""
    CC = dx.CurriculumConfig
    out = []
    for k in range(G):
        f = k / G
        kw = dict(object_size=0.02 + 0.1 * f, object_mass=0.05 + 0.4 * f, friction_coefficient=0.1 + 0.8 * f,
                  spawn_x_range=(-0.1 + 0.05 * f, 0.1), spawn_z_range=(0.05, 0.1 + 0.1 * f))
        if k % 3 == 1:
            kw["object_size_range"] = (0.02 + 0.05 * f, 0.07 + 0.05 * f)
        if k % 5 == 2:
            kw["object_mass_range"] = (0.05 + 0.1 * f, 0.3 + 0.1 * f)
            kw["friction_range"] = (0.2 * f, 0.5 + 0.2 * f)
        out.append(CC(**kw))
    return out


def _sigma_dyn(G, on=True):
    return [0.05 if on and k in _noisy_rows(G) else 0.0 for k in range(G)]


def _oracle_table(cfgs, sigma_obs=0.0, sigma_dyn=0.0):
    """The oracle's group array holding the bytes the env uploads."""
    return np.frombuffer(bytes(dx.group_table(cfgs, sigma_obs, sigma_dyn)), oracle.GROUP_DTYPE).copy()


def _map(kind, n, G, seed=0):
    """(env_gid0, group_of_env or None, group of every env)."""
    if kind == "default":
        gid0 = 2 ** 32 - n // 2
        return gid0, None, ((gid0 + np.arange(n, dtype=np.int64)) & M32) % G
    rng = np.random.default_rng(seed + 1000 * G + n)
    if kind == "random":
        goe = rng.integers(0, G, n)
    else:                                    # most envs in G-1; only every third other group is used at all
        goe = np.full(n, G - 1)
        few = rng.random(n) < 0.2
        goe[few] = rng.choice(np.arange(0, G - 1, 3), int(few.sum()))
    return 7, goe.astype(np.uint16), goe.astype(np.int64)


def _gamma(k):
    return k * U / (1.0 - k * U)


def _sum_bound(values, extra_rounding=False):
    """Bound on |computed - exact| of a float64 sum of `values` in any order: gamma_{m-1} * sum |v| (Higham, Accuracy
    and Stability of Numerical Algorithms, 2nd ed., (4.4)); gamma_m when every term was rounded once before it was
    added (the squares)."""
    m = len(values)
    k = m if extra_rounding else m - 1
    return _gamma(max(k, 0)) * math.fsum(abs(v) for v in values)


def _assert_sums_within_bound(ret_sums, per_group, where=""):
    """ret_sums [G, 2] against the exact sums of the episode returns `per_group` (list of lists) and of their squares."""
    for g, r in enumerate(per_group):
        s, s2 = math.fsum(r), math.fsum(x * x for x in r)
        assert abs(ret_sums[g, 0] - s) <= _sum_bound(r), (where, g, ret_sums[g, 0], s)
        assert abs(ret_sums[g, 1] - s2) <= _sum_bound([x * x for x in r], extra_rounding=True), (where, g)


def _returns_by_group(log, gid0, groups, G):
    """Logged episode returns grouped by the env's group (env = (env_gid - env_gid0) mod 2^32)."""
    env = ((log["env_gid"].astype(np.int64) - gid0) & M32)
    out = [[] for _ in range(G)]
    for e, r in zip(env, log["episode_reward"]):
        out[groups[e]].append(float(r))
    return out


# ---- CPU: validation ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad,why", [
    (np.zeros(9, np.int64), "shape"),
    (np.zeros((10, 1), np.int64), "shape"),
    (np.array([0] * 9 + [-1]), r"\[0, 17\)"),
    (np.array([0] * 9 + [17]), r"\[0, 17\)"),
    (np.array([0] * 9 + [40000]), r"\[0, 17\)"),
    (np.array([0] * 9 + [2 ** 40]), r"\[0, 17\)"),
    (np.zeros(10, np.float32), "integers"),
    (np.zeros(10, bool), "integers"),
    ([0.0] * 10, "integers"),
    (torch.full((10,), 32768, dtype=torch.int32), r"\[0, 17\)"),
])
def test_map_validation_rejects(bad, why):
    with pytest.raises(ValueError, match=why):
        check_group_of_env(bad, 10, 17)


def test_map_validation_accepts_and_keeps_values():
    for src in (np.arange(10) % 17, list(range(10)), torch.arange(10, dtype=torch.int16), np.full(10, 16, np.uint8)):
        out = check_group_of_env(src, 10, 17)
        assert out.dtype == np.uint16 and np.array_equal(out, np.asarray(src.numpy() if isinstance(src, torch.Tensor) else src))
    assert np.array_equal(check_group_of_env(np.full(10, 255), 10, 256), np.full(10, 255))


def _bare_env(n, G, goe=None):
    """A BatchedManipulationEnv with only what set_groups reads before it would touch a device."""
    env = object.__new__(BatchedManipulationEnv)
    env.num_envs, env._group_cfgs = n, [dx.CurriculumConfig()] * G
    env._goe = env._goe_host = None
    env._goe_max = -1
    if goe is not None:
        env._goe = env._goe_host = check_group_of_env(goe, n, G)
        env._goe_max = int(env._goe_host.max())
    return env


def test_set_groups_rejects_a_table_the_kept_map_does_not_fit():
    env = _bare_env(10, 17, np.arange(10) + 7)                          # names group 16
    with pytest.raises(ValueError, match="group 16"):
        env.set_groups([dx.CurriculumConfig()] * 16)
    assert len(env._group_cfgs) == 17                                   # a refused call changes nothing
    with pytest.raises(ValueError, match=r"\[0, 5\)"):
        env.set_groups([dx.CurriculumConfig()] * 5, group_of_env=np.arange(10))


def test_set_groups_rejects_more_than_256_configs():
    env = _bare_env(10, 4)
    with pytest.raises(ValueError, match="1..256"):
        env.set_groups([dx.CurriculumConfig()] * 257)
    with pytest.raises(ValueError, match="1..256"):
        env.set_groups([])


def test_config_of_env_wraps_the_global_id_at_2_32():
    """rng="numpy" resets pick each env's config on the host; the kernels count it in (uint32)(env_gid0 + i) % G."""
    env = object.__new__(BatchedManipulationEnv)
    env._group_cfgs, env._goe = list(range(5)), None
    for gid0 in (2 ** 32 - 3, 2 ** 33 + 11, -4):
        env.env_gid0 = gid0
        assert [env._config_of_env(i) for i in range(8)] == [((gid0 + i) & M32) % 5 for i in range(8)]


# ---- CPU: the bound and the oracle's own sums -----------------------------------------------------------------------
def test_sum_bound_holds_and_is_tight_enough():
    rng = np.random.default_rng(3)
    for m in (1, 2, 7, 1000, 20000):
        v = list(rng.normal(0.0, 10.0, m) * np.exp(rng.uniform(-20, 20, m)))
        exact = math.fsum(v)
        for order in (v, sorted(v), sorted(v, key=abs, reverse=True)):
            s = 0.0
            for x in order:
                s += x
            assert abs(s - exact) <= _sum_bound(v)
        assert _sum_bound(v) <= 1.01 * (m - 1) * U * math.fsum(abs(x) for x in v)
    assert _sum_bound([3.5]) == 0.0 and _gamma(1) > U


@pytest.mark.parametrize("G,kind", [(17, "random"), (65, "skewed"), (255, "default")])
def test_oracle_sums_within_bound_of_exact_episode_sums(G, kind):
    """The oracle's sequential return sums against math.fsum of every episode return.  The returns come from a twin
    run that puts every env in a group of its own (table row i = the coarse row of env i, so the dynamics are the
    same) and steps one call at a time: then each group's sum holds one return, exactly."""
    n, K, max_steps, seed = 200, 24, 5, 17
    cfgs = _cfgs(G)
    table = _oracle_table(cfgs, 0.0, _sigma_dyn(G))
    gid0, goe, groups = _map(kind, n, G)
    fine = table[groups]
    starts = []
    for i in range(n):
        starts.append(oracle.reset_draws(seed, (gid0 + i) & M32, 0, table[groups[i]:groups[i] + 1]))
    batches = []
    for _ in range(2):
        ob = oracle.OracleBatch(n, dense=True, max_episode_steps=max_steps)
        ob.reset_predrawn(np.stack([d[0] for d in starts]), [d[1] for d in starts], [d[2] for d in starts],
                          [d[3] for d in starts], np.stack([d[4] for d in starts]))
        batches.append(ob)
    cnt, rs = batches[0].rollout(table, K, seed, policy_kind=2, env_gid0=gid0, group_of_env=goe, loop_max_steps=max_steps)
    per_group = [[] for _ in range(G)]
    cnt_fine = np.zeros((n, oracle.NCOUNTERS), np.int64)
    for t in range(K):
        c1, r1 = batches[1].rollout(fine, 1, seed, policy_kind=2, env_gid0=gid0, group_of_env=np.arange(n, dtype=np.uint16),
                                    loop_max_steps=max_steps)
        cnt_fine += c1
        for i in np.nonzero(c1[:, EPISODES])[0]:
            assert c1[i, EPISODES] == 1 and r1[i, 1] == r1[i, 0] * r1[i, 0]
            per_group[groups[i]].append(float(r1[i, 0]))
    assert np.array_equal(batches[0].env, batches[1].env)
    summed = np.zeros_like(cnt)
    np.add.at(summed, groups, cnt_fine)
    assert np.array_equal(summed, cnt)                                  # the map routes every counter
    assert [len(r) for r in per_group] == list(cnt[:, EPISODES]) and cnt[:, EPISODES].sum() >= 3 * n
    _assert_sums_within_bound(rs, per_group)


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


def _env(n, G, kind, max_steps=6, sigma_dyn=None, sigma_obs=0.0, seed=11, **kw):
    gid0, goe, groups = _map(kind, n, G)
    cfgs = _cfgs(G)
    sd = _sigma_dyn(G) if sigma_dyn is None else sigma_dyn
    kw.setdefault("track_episodes", True)
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense", groups=cfgs, seed=seed,
                                    env_gid0=gid0, group_of_env=goe, group_sigma_dyn=sd, group_sigma_obs=sigma_obs, **kw)
    return env, _oracle_table(cfgs, sigma_obs, sd), gid0, goe, groups


def _oracle_from(env):
    """An oracle batch in the env's current state (fresh after a reset)."""
    n = env.num_envs
    ob = oracle.OracleBatch(n, dense=True, max_episode_steps=env.max_episode_steps)
    ob.reset_predrawn(env._obs[:15, :n].t().cpu().numpy(), env._size[:n].cpu().numpy(), env._mass[:n].cpu().numpy(),
                      env._friction[:n].cpu().numpy(), env._obs[30:33, :n].t().cpu().numpy())
    return ob


def _drawn_dyn_noise(aux, ob, noisy):
    """The dynamics noise the kernels draw for every env at the oracle's current (episode, step): dexsim_fill_normal on
    stream 2 at the noisy rows' sigma (checked against the in-kernel draw by tests/test_gpu_parity.py), 0 elsewhere.
    The oracle itself has no noise generator."""
    n = aux.num_envs
    aux._episode[:n] = torch.from_numpy(ob.env["episode"].view(np.int32).copy())
    aux._step_count[:n] = torch.from_numpy(ob.env["step_count"].copy())
    out = torch.zeros(15, aux.ld, dtype=torch.float32, device=aux.device)
    _lib.check(aux._lib.dexsim_fill_normal(C.byref(aux._state), C.byref(aux._params), _lib.RNG_STREAM_DYN, 15,
                                           C.c_float(0.05), out.data_ptr(), aux._stream()), "dexsim_fill_normal")
    z = out[:, :n].t().cpu().numpy()
    return np.where(noisy[:, None], z, np.float32(0.0))[None]


def _rollout_cases():
    """Every (G, map) pair once, with the size, policy, noise and kernel rotating so that each of them meets group
    counts on both sides of every threshold.  The 5-lane kernel runs without dynamics noise, and only up to 8,192 envs."""
    cases = []
    for a, G in enumerate(GS):
        for b, kind in enumerate(MAPS):
            k = a + b
            n = SIZES[k % 3]
            policy = ("random", "heuristic")[(a + 2 * b) % 2]
            split = n <= 8192 and (a + b) % 2 == 1
            cases.append((G, kind, n, policy, "split" if split else "thread", not split and (a * 3 + b) % 4 != 3))
    # the rotation gives the 5-lane kernel the default map only at 16 and 64 groups, where the 2^32 wrap leaves gid % G
    # unchanged: two more cases across the wrap at group counts where it does not
    return cases + [(17, "default", 130, "random", "split", False), (255, "default", 4096 + 77, "heuristic", "split", False)]


ROLLOUT_CASES = _rollout_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("G,kind,n,policy,impl,noise", ROLLOUT_CASES)
def test_fused_rollout_matches_oracle(gpu, G, kind, n, policy, impl, noise):
    """Two launches of the fused rollout against the oracle's rollout with the same table, map and env_gid0: every
    state array bit for bit, every counter of every row (empty rows included) exactly, and the return sums within
    the derived bound of the exact sums of the logged episode returns."""
    max_steps, K = 6, 20
    env, table, gid0, goe, groups = _env(n, G, kind, max_steps, sigma_dyn=None if noise else 0.0)
    env.reset(seed=11)
    env.enable_episode_log(n * K)
    ob = _oracle_from(env)
    aux = _env(n, G, kind, max_steps)[0] if noise else None
    noisy = np.isin(groups, _noisy_rows(G))
    cnt_o = rs_o = None
    kw = dict(policy_kind=1 if policy == "random" else 2, env_gid0=gid0, group_of_env=goe, loop_max_steps=max_steps,
              threads=8)
    try:
        _lib.set_rollout_impl(impl)
        for chunk in (K // 2, K - K // 2):
            env.rollout(chunk, policy=policy)
            if not noise:
                cnt_o, rs_o = ob.rollout(table, chunk, 11, counters=cnt_o, ret_sums=rs_o, **kw)
            for _ in range(chunk if noise else 0):   # the oracle takes the noise the kernel draws, one step at a time
                cnt_o, rs_o = ob.rollout(table, 1, 11, dyn_noise=_drawn_dyn_noise(aux, ob, noisy), counters=cnt_o,
                                         ret_sums=rs_o, **kw)
    finally:
        _lib.set_rollout_impl("auto")
    cnt = env.counters.cpu().numpy()
    assert np.array_equal(cnt, cnt_o)
    used = np.bincount(groups, minlength=G) > 0
    assert np.all(cnt[used, EPISODES] >= 3 * np.bincount(groups, minlength=G)[used])   # every env reset several times
    assert not cnt[~used].any()
    assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), ob.observation())
    for name, key in (("_op64", "op"), ("_size", "size"), ("_mass", "mass"), ("_friction", "friction"),
                      ("_step_count", "step_count")):
        got = getattr(env, name)
        got = got[:, :n].t() if got.dim() == 2 else got[:n]
        assert np.array_equal(got.cpu().numpy(), ob.env[key]), name
    assert np.array_equal(env._episode[:n].cpu().numpy().astype(np.uint32), ob.env["episode"])
    log = env.read_episode_log()
    assert env.episode_log_overflow == 0
    per_group = _returns_by_group(log, gid0, groups, G)
    assert [len(r) for r in per_group] == list(cnt[:, EPISODES])
    rs = env.ret_sums.cpu().numpy()
    _assert_sums_within_bound(rs, per_group, "kernel")
    _assert_sums_within_bound(rs_o, per_group, "oracle")


def _fill(env, act, kind=2):
    _lib.check(env._lib.dexsim_fill_policy_actions(C.byref(env._state), C.byref(env._params), kind, act.data_ptr(),
                                                   env._stream()), "dexsim_fill_policy_actions")
    return act[:, :env.num_envs].t().contiguous()


STEP_PATHS = ("register", "tma", "tma_wide", "register_counts", "tma_counts", "final_observation", "host_chunks",
              "host_zero_copy")
STEP_CASES = [(path, G, MAPS[(a + b) % 3]) for a, path in enumerate(STEP_PATHS) for b, G in enumerate((16, 17, 64, 65, 256))]


@pytest.mark.gpu
@pytest.mark.parametrize("path,G,kind", STEP_CASES)
def test_step_paths_equal_fused_rollout(gpu, path, G, kind):
    """Auto-reset stepping fed with the in-kernel heuristic policy's actions equals the fused rollout (itself checked
    against the oracle above): counters exactly, state bit for bit, return sums within the bound of the rollout's
    logged returns."""
    n, K, max_steps = 4096 + 77, 20, 6
    counts_only = path.endswith("_counts")
    a, *_ = _env(n, G, kind, max_steps, sigma_dyn=0.0, auto_reset=True, respawn=True, loop_max_steps=max_steps,
                 track_episodes=not counts_only, final_observation=path == "final_observation")
    b, _, gid0, goe, groups = _env(n, G, kind, max_steps, sigma_dyn=0.0)
    a.reset(seed=11); b.reset(seed=11)
    if path.startswith("host"):
        a.host_zero_copy = path == "host_zero_copy"
    act = torch.zeros(15, a.ld, device="cuda")
    impl = path.replace("_counts", "")
    try:
        if impl in ("register", "tma", "tma_wide"):
            _lib.set_step_impl("tma" if impl == "tma_wide" else impl)
            _lib.set_step_tile("wide" if impl == "tma_wide" else "narrow" if impl == "tma" else "auto")
        for t in range(K):
            x = _fill(a, act)
            if path == "host_chunks":
                a.step_host(x.cpu().pin_memory(), chunks=1 + t % 4)
            elif path == "host_zero_copy":
                a.step_host(x.cpu().pin_memory())
            else:
                a.step(x)
    finally:
        _lib.set_step_impl("auto"); _lib.set_step_tile("auto")
    b.enable_episode_log(n * K)
    b.rollout(K, policy="heuristic", respawn=True, loop_max_steps=max_steps)
    torch.cuda.synchronize()
    cols = [0, 1, 2, 3, 17] if counts_only else list(range(dx.NCOUNTERS))
    assert torch.equal(a.counters[:, cols], b.counters[:, cols])
    assert int(b.counters[:, EPISODES].sum()) >= 3 * n
    for name in STATE:
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    if not counts_only:
        per_group = _returns_by_group(b.read_episode_log(), gid0, groups, G)
        _assert_sums_within_bound(a.ret_sums.cpu().numpy(), per_group)


@pytest.mark.gpu
@pytest.mark.parametrize("G,kind,impl", [(17, "random", "tma"), (65, "skewed", "register"), (255, "default", "tma_wide"),
                                         (256, "random", "tma")])
def test_next_step_reset_counts_and_draws_by_group(gpu, G, kind, impl):
    """autoreset_mode="next_step": EPISODES and SUCCESSES equal a host bincount of info["finished"] (and of finished &
    terminated) by each env's group, and every pending reset draws size, mass and friction from its own group's row."""
    n, K, max_steps, seed = 4096 + 77, 20, 5, 11
    env, table, gid0, goe, groups = _env(n, G, kind, max_steps, sigma_dyn=0.0, auto_reset=True, respawn=True,
                                         loop_max_steps=max_steps, autoreset_mode="next_step")
    env.reset(seed=seed)
    act = torch.zeros(15, env.ld, device="cuda")
    want = np.zeros((G, 2), np.int64)
    pending = np.zeros(n, bool)
    checked = 0
    g_t = torch.from_numpy(groups).cuda()
    try:
        _lib.set_step_impl("tma" if impl == "tma_wide" else impl)
        _lib.set_step_tile("wide" if impl == "tma_wide" else "narrow" if impl == "tma" else "auto")
        for t in range(K):
            obs, rew, te, tr, info = env.step(_fill(env, act))
            if pending.any():                        # this step reset them: check their draws against their own row
                idx = np.nonzero(pending)[0][::7]
                ep = env._episode[:n].cpu().numpy()
                got = np.stack([getattr(env, k)[:n].cpu().numpy()[idx] for k in ("_size", "_mass", "_friction")], 1)
                for j, i in enumerate(idx):
                    d = oracle.reset_draws(seed, (gid0 + int(i)) & M32, int(ep[i]), table[groups[i]:groups[i] + 1])
                    assert tuple(got[j]) == (d[1], d[2], d[3]), (t, i)
                checked += len(idx)
            fin = info["finished"]
            want[:, 0] += torch.bincount(g_t[fin], minlength=G).cpu().numpy()
            want[:, 1] += torch.bincount(g_t[fin & te], minlength=G).cpu().numpy()
            pending = fin.cpu().numpy()
    finally:
        _lib.set_step_impl("auto"); _lib.set_step_tile("auto")
    cnt = env.counters.cpu().numpy()
    assert np.array_equal(cnt[:, [EPISODES, SUCCESSES]], want)
    assert want[:, 0].sum() >= 2 * n and checked > n // 4


@pytest.mark.gpu
@pytest.mark.parametrize("G,kind,n", [(5, "default", 130), (17, "random", 4096 + 77), (65, "skewed", 4096 + 77),
                                      (255, "default", 70_001), (256, "random", 130), (64, "skewed", 70_001)])
def test_philox_and_masked_resets_draw_from_each_envs_row(gpu, G, kind, n):
    """reset(seed) and a masked reset: per env, size, mass, friction, joints and position equal the oracle's draws for
    (seed, (env_gid0 + i) mod 2^32, episode, its group's row); envs outside the mask keep their state."""
    seed = 23
    env, table, gid0, goe, groups = _env(n, G, kind, 50, respawn=True)
    sample = np.unique(np.concatenate([np.arange(min(n, 300)), np.random.default_rng(n).integers(0, n, 700), [n - 1]]))

    def check(episode_of, idx):
        size, mass, fric = (getattr(env, k)[:n].cpu().numpy() for k in ("_size", "_mass", "_friction"))
        jp, pos = env._obs[0:15, :n].t().cpu().numpy(), env._obs[30:33, :n].t().cpu().numpy()
        for i in idx:
            d = oracle.reset_draws(seed, (gid0 + int(i)) & M32, int(episode_of[i]), table[groups[i]:groups[i] + 1])
            assert np.array_equal(jp[i], d[0]) and (size[i], mass[i], fric[i]) == (d[1], d[2], d[3]), i
            assert np.array_equal(pos[i], d[4]), i

    env.reset(seed=seed)
    check(np.zeros(n, np.int64), sample)
    gen = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(3):
        env.step(torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1)
    mask = torch.rand(n, device="cuda", generator=gen) < 0.4
    before = {k: getattr(env, k).clone() for k in STATE}
    env.reset(options={"mask": mask})
    m = mask.cpu().numpy()
    check(env._episode[:n].cpu().numpy(), sample[m[sample]])
    assert bool((env._episode[:n][mask] == 1).all())
    keep = ~mask
    for k, v in before.items():
        cur = getattr(env, k)
        assert torch.equal(cur[..., :n][..., keep], v[..., :n][..., keep]), k


@pytest.mark.gpu
def test_numpy_resets_take_each_envs_config_across_the_wrap(gpu):
    """rng="numpy" with the global ids crossing 2^32 and G = 5 (2^32 mod 5 = 1): each env's object comes from the
    configuration of the group the kernels count it in."""
    n, G, gid0 = 64, 5, 2 ** 32 - 32
    CC = dx.CurriculumConfig
    cfgs = [CC(object_size=0.03 + 0.01 * k, object_mass=0.1 + 0.05 * k, friction_coefficient=0.2 + 0.1 * k) for k in range(G)]
    env = dx.BatchedManipulationEnv(n, "cuda", rng="numpy", groups=cfgs, env_gid0=gid0, track_episodes=True,
                                    auto_reset=True, loop_max_steps=3, max_episode_steps=3)
    env.reset(seed=list(range(n)))
    g = ((gid0 + np.arange(n)) & M32) % G
    for name, attr in (("_size", "object_size"), ("_mass", "object_mass"), ("_friction", "friction_coefficient")):
        assert np.array_equal(getattr(env, name)[:n].cpu().numpy(), [getattr(cfgs[k], attr) for k in g]), name
    for _ in range(3):                                    # the kernels count every env's episode in that same group
        env.step(torch.zeros(n, 15, device="cuda"))
    assert np.array_equal(env.counters[:, EPISODES].cpu().numpy(), np.bincount(g, minlength=G))


@pytest.mark.gpu
@pytest.mark.parametrize("G,kind", [(65, "random"), (255, "default")])
def test_tie_resolution_moves_only_the_envs_own_row(gpu, G, kind):
    """Records flagged with an exact variance tie are injected into the log and history of a rollout, as in
    tests/test_long_episodes.py; resolve_ties_kernel must correct the label counters of each env's own group and
    leave every other row unchanged."""
    from test_long_episodes import M27, _labels, _summary_kw
    n, thr, hist_steps, max_steps = 4096 + 77, 6, 200, 200
    env, table, gid0, goe, groups = _env(n, G, kind, max_steps, sigma_dyn=0.0)
    env._params.success_threshold = thr
    env.reset(seed=3)
    rng = np.random.default_rng(G)
    picks = []
    while len(picks) < 24:                              # permutations on both sides of np.var == 2
        c = rng.permutation(np.array(M27 * (5 if len(picks) % 2 else 7), np.uint8))
        if c[-1] != 0:
            picks.append(c)
    envs = rng.choice(n, len(picks), replace=False)
    env.enable_episode_log(len(picks))
    env.enable_history(hist_steps)
    hist = np.zeros((hist_steps, env.ld), np.uint8)
    rec = np.zeros(len(picks), _lib.EPISODE_RECORD_DTYPE)
    before = rng.integers(1000, 2000, (G, dx.NCOUNTERS)).astype(np.int64)     # every row holds something to keep
    after = before.copy()
    flips = 0
    for q, (i, c) in enumerate(zip(envs, picks)):
        L, fin = len(c), int(c[-1])
        hist[:L, i] = c
        a0, b0, tie = dx.classify_summary(False, L, fin, fin, max_steps=max_steps, success_threshold=thr, **_summary_kw(c))
        assert tie == 1
        rec[q] = ((gid0 + int(i)) & M32, 0, L, 0, fin, a0, b0, 0.0, L - 1, 1)
        a1, b1 = _labels(c, L, fin, max_steps, thr)
        g = groups[i]
        for base, old, new in ((dx.CNT_LABEL_METRICS, a0, a1), (dx.CNT_LABEL_TAXONOMY, b0, b1)):
            after[g, base + old] -= 1
            after[g, base + new] += 1
        after[g, dx.CNT_VAR_TIES] -= 1
        flips += a1 != a0
    assert flips > 0
    env._hist.copy_(torch.from_numpy(hist))
    env._ep_log.copy_(torch.from_numpy(rec.view(np.uint8)))
    env._ep_log_count.fill_(len(picks))
    env.counters.copy_(torch.from_numpy(before))
    env._rollout_steps = hist_steps                    # the rollout's own step writes no history row
    env.rollout(1, policy="random")                    # no episode ends in one step
    assert np.array_equal(env.read_episode_log(sort=False)["var_tie"], [2] * len(picks))
    assert np.array_equal(env.counters.cpu().numpy(), after)


def _sigma_of_env(env, goe, sigma):
    return torch.tensor(np.asarray(sigma, np.float32)[goe.astype(np.int64)], device=env.device)


def _rollout_cta_threads(n, sm_count):
    """The CTA size rollout_launch picks: it halves a 256-thread CTA while the batch gives fewer than 4 CTAs per SM."""
    warps, threads = (n + 31) // 32, 256
    while threads > 32 and warps * 32 // threads < sm_count * 4:
        threads = (threads // 2 + 31) // 32 * 32
    return threads


@pytest.mark.gpu
@pytest.mark.parametrize("G", [64, 65])
def test_mlp_rollout_either_side_of_the_staged_table(gpu, G):
    """A (64, 64) MLP with action_std, observation noise on groups above the thresholds and an explicit map, at a batch
    just large enough for 256-thread CTAs (4 CTAs of 256 per SM, plus a ragged tail).  At G = 64 the table is staged
    and the largest weight layout sits behind it: 19,968 B of table and counters, 32,640 B of weights and 65,536 B of
    second-layer scratch (64 floats per thread), 118,144 B of dynamic shared memory by arithmetic.  At G = 65 the
    weights start at offset 0.  Rows, final state and counters equal a step() twin bit for bit
    (tests/test_rollout_mlp.py)."""
    sm = C.c_int()
    _lib.check(_lib.lib().dexsim_device_info(C.byref(sm), C.byref(C.c_int()), C.byref(C.c_int())), "dexsim_device_info")
    n = 4 * sm.value * 256 + 77                      # 151,629 envs on a 148-SM B200
    assert _rollout_cta_threads(n, sm.value) == 256 and _rollout_cta_threads(n // 2, sm.value) == 128
    import test_rollout_mlp as M
    K, max_steps, seed = 12, 6, 5
    so = [0.04 if k in (16, 40, 63, G - 1) else 0.0 for k in range(G)]
    sd = [0.05 if k in (3, 17, 62, G - 1) else 0.0 for k in range(G)]
    common = dict(max_episode_steps=max_steps, reward_type="dense", track_episodes=True, seed=seed, respawn=True,
                  groups=_cfgs(G), group_sigma_obs=so, group_sigma_dyn=sd)
    _, goe, _ = _map("random", n, G)
    rec = dx.BatchedManipulationEnv(n, "cuda", group_of_env=goe, **common)
    twin = dx.BatchedManipulationEnv(n, "cuda", group_of_env=goe, auto_reset=True, final_observation=True,
                                     loop_max_steps=max_steps, **common)
    rec.reset(seed=seed); twin.reset(seed=seed)
    pol = dx.MlpPolicy.from_torch(M._net((64, 64), "relu", G), action_std=M.STD)
    sigma_env = _sigma_of_env(rec, goe, so)
    rec.enable_trajectory(K, final_observation=True)
    finished = 0
    for call in range(2):
        rec.rollout(K, policy=pol)
        tr = rec.trajectory
        M._assert_rows_equal_twin(twin, tr, pol, sigma_env, call)
        finished += int(tr["finished"].sum())
    M._assert_same_end(rec, twin)
    assert finished >= n


def _guard(env, names, guard=4096):
    """Re-home the named device arrays of the env in the middle of larger buffers whose margins hold a byte pattern
    (tests/test_gpu_parity.py::_with_guard_bands, plus the counters, the return sums, the group table and the map)."""
    bands = []
    for name in names:
        t = getattr(env, name, None)
        if t is None:
            continue
        nbytes = t.numel() * t.element_size()
        big = torch.full((nbytes + 2 * guard,), 0xA5, dtype=torch.uint8, device=t.device)
        mid = big[guard:guard + nbytes].view(t.dtype).view(t.shape)
        mid.copy_(t)
        setattr(env, name, mid)
        bands.append((name, big, guard, nbytes))
    n = env.num_envs
    env._refresh_structs()
    env._groups_ptr = env._groups_dev.data_ptr()
    env._goe_ptr = None if env._goe is None else env._goe.data_ptr()
    env._step_final_obs = env._ptr(env._final_obs)
    env._obs_view = env._obs[:, :n].t()
    env._info = None
    env._step_out = (env._obs_view, env._reward[:n], env._terminated[:n].view(torch.bool),
                     env._truncated[:n].view(torch.bool), env._make_info())

    def check():
        torch.cuda.synchronize()
        for name, big, g, nb in bands:
            assert bool((big[:g] == 0xA5).all()) and bool((big[g + nb:] == 0xA5).all()), f"out-of-bounds write around {name}"
    return check


GUARDED = ["_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
           "_ep_return", "_ep_stats", "_reward", "_terminated", "_truncated", "_num_contacts", "_finished", "_action_dev",
           "_final_obs", "counters", "ret_sums", "_groups_dev", "_goe"]


@pytest.mark.gpu
@pytest.mark.parametrize("G", [17, 65, 256])
@pytest.mark.parametrize("kind", ["default", "random"])
def test_no_writes_outside_counters_table_or_map(gpu, G, kind):
    """Every kernel above at G = 17, 65 and 256 with both maps: no byte outside the env's arrays, the counters, the
    return sums, the group table and the map may change."""
    n = {17: 130, 65: 4096 + 77, 256: 70_001}[G]
    gen = torch.Generator(device="cuda").manual_seed(G)
    rnd = lambda: torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
    env, *_ = _env(n, G, kind, 6, sigma_dyn=0.0, auto_reset=True, respawn=True, loop_max_steps=6)   # split-eligible
    fin, *_ = _env(n, G, kind, 6, auto_reset=True, respawn=True, loop_max_steps=6, final_observation=True)
    nxt, *_ = _env(n, G, kind, 6, sigma_dyn=0.0, auto_reset=True, respawn=True, loop_max_steps=6, autoreset_mode="next_step")
    checks = [_guard(e, GUARDED) for e in (env, fin, nxt)]
    check = lambda: [c() for c in checks]
    for e in (env, fin, nxt):
        e.reset(seed=2)
        e.reset(options={"mask": torch.rand(n, device="cuda", generator=gen) < 0.5})
    check()
    try:
        for impl in ("register", "tma", "tma_wide"):
            _lib.set_step_impl("tma" if impl == "tma_wide" else impl)
            _lib.set_step_tile("wide" if impl == "tma_wide" else "narrow" if impl == "tma" else "auto")
            for _ in range(8):
                env.step(rnd()); fin.step(rnd()); nxt.step(rnd())
            check()
        _lib.set_step_impl("auto"); _lib.set_step_tile("auto")
        for zc in (False, True):
            env.host_zero_copy = fin.host_zero_copy = zc
            for chunks in (1, 3):
                env.step_host(rnd().cpu().pin_memory(), chunks=chunks)
                fin.step_host(rnd().cpu().pin_memory(), chunks=chunks)
            check()
        env.enable_episode_log(n * 30)
        env.enable_history(30)
        for impl in ("thread", "split"):
            _lib.set_rollout_impl(impl)
            env.rollout(10, policy="heuristic")
            check()
        _lib.set_rollout_impl("auto")
        import test_rollout_mlp as M
        env.rollout(10, policy=dx.MlpPolicy.from_torch(M._net((64, 64), "relu", 1), action_std=M.STD))
        check()
    finally:
        _lib.set_step_impl("auto"); _lib.set_step_tile("auto"); _lib.set_rollout_impl("auto")
    assert int(env.counters[:, EPISODES].sum()) > n
