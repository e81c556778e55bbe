"""GPU parity tests proper: the CUDA path (through the C ABI, via BatchedManipulationEnv)
against the committed golden fixtures of the UNMODIFIED reference and against the oracle.

Bars (BASELINE.json north_star): done flags, success, contact labels, failure labels and
counters bit-exact; observations bit-exact (they are float32 state computed with the
reference's own roundings); rewards within rtol 1e-6 of the reference's float64 value
(the kernel computes the float64 total and stores it as float32; the stated bar is 1e-5)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

REWARD_RTOL = 1e-6
REWARD_ATOL = 1e-7


def _load(golden_dir, name):
    with np.load(os.path.join(golden_dir, name), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def dx():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import dexterous_rl_manipulation_b200 as d
    return d


class _Shaping:       # weights carrier with the attribute names of rewards/reward_shaping.py:36-39
    def __init__(self, w):
        self.distance_weight, self.contact_weight, self.closure_weight, self.stability_weight = w


def _make_env(dx, n, dense, max_steps, weights=(1.0, 0.5, 0.3, 0.2), **kw):
    return dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=int(max_steps),
                                     reward_type="dense" if dense else "sparse",
                                     reward_shaping=_Shaping(weights) if dense else None,
                                     reward_components=True, **kw)


def test_golden_trajectories_batched(dx, golden_dir):
    """All reference trajectories with equal env parameters run as ONE batch."""
    g = _load(golden_dir, "traj.npz")
    T = g["actions"].shape[1]
    keys = {}
    for i in range(g["actions"].shape[0]):
        if g["keep_pos"][i]:
            continue
        keys.setdefault((bool(g["dense"][i]), int(g["max_steps"][i]), tuple(g["weights"][i])), []).append(i)
    checked = 0
    for (dense, max_steps, weights), idx in keys.items():
        idx = np.asarray(idx)
        n = len(idx)
        env = _make_env(dx, max(n, 2), dense, max_steps, weights)     # >= 2: tensor-returning path
        pad = env.num_envs - n

        def padded(a):
            return np.concatenate([a, np.repeat(a[-1:], pad, 0)]) if pad else a

        def run(sel, pos):
            obs0, _ = env.reset_from_draws(padded(g["jp0"][sel]), padded(g["size"][sel]), padded(g["mass"][sel]),
                                           padded(g["friction"][sel]), pos)
            assert np.array_equal(obs0.cpu().numpy()[:n], g["obs"][sel, 0])
            for t in range(T):
                obs, rew, te, tr, info = env.step(torch.from_numpy(padded(g["actions"][sel, t])).cuda())
                assert np.array_equal(obs.cpu().numpy()[:n], g["obs"][sel, t + 1]), t
                assert np.array_equal(te.cpu().numpy()[:n], g["terminated"][sel, t])
                assert np.array_equal(tr.cpu().numpy()[:n], g["truncated"][sel, t])
                assert np.array_equal(info["num_contacts"].cpu().numpy()[:n], g["num_contacts"][sel, t])
                np.testing.assert_allclose(rew.cpu().numpy()[:n], g["reward"][sel, t], rtol=REWARD_RTOL, atol=REWARD_ATOL)
                rc = info["reward_components"]
                comps = np.stack([rc[k].cpu().numpy()[:n] for k in ("distance", "contact", "closure", "stability")], 1)
                np.testing.assert_allclose(comps, g["comps"][sel, t], rtol=REWARD_RTOL, atol=REWARD_ATOL)
            assert np.array_equal(info["object_position"].cpu().numpy()[:n], g["op_final"][sel])   # float64 exact

        run(idx, padded(g["pos"][idx]))
        checked += n
        # second episodes on the reused env objects keep the object where the first one left it
        chained = np.asarray([j for j in range(g["actions"].shape[0]) if g["keep_pos"][j] and g["chain"][j] in idx])
        if len(chained):
            # rebuild an env holding exactly the predecessors, replay them, then reset in place
            pre = g["chain"][chained]
            n = len(pre)
            env = _make_env(dx, max(n, 2), dense, max_steps, weights)
            pad = env.num_envs - n
            run(pre, padded(g["pos"][pre]))
            run(chained, None)
            checked += n
    assert checked == g["actions"].shape[0]


def test_noise_wrapper_golden(dx, golden_dir):
    g = _load(golden_dir, "noise.npz")
    n, T = g["actions"].shape[:2]
    env = _make_env(dx, n, True, int(g["max_steps"]))
    obs0, _ = env.reset_from_draws(g["jp0"], g["size"], g["mass"], g["friction"], g["pos"])
    exp0 = obs0.cpu().numpy() + g["obs_noise"][:, 0]
    assert np.array_equal(exp0, g["obs"][:, 0])
    for t in range(T):
        obs, rew, te, tr, info = env.step(torch.from_numpy(g["actions"][:, t]).cuda(),
                                          dyn_noise=g["dyn_noise"][:, t], obs_noise=g["obs_noise"][:, t + 1])
        assert np.array_equal(obs.cpu().numpy(), g["obs"][:, t + 1]), t
        assert np.array_equal(te.cpu().numpy(), g["terminated"][:, t])
        assert np.array_equal(tr.cpu().numpy(), g["truncated"][:, t])
        assert np.array_equal(info["num_contacts"].cpu().numpy(), g["num_contacts"][:, t])
        np.testing.assert_allclose(rew.cpu().numpy(), g["reward"][:, t], rtol=REWARD_RTOL, atol=REWARD_ATOL)


@pytest.mark.parametrize("kernel,reps", [("tma", 32), ("tma_wide", 48)])
def test_noise_wrapper_golden_on_the_tma_pipeline(dx, golden_dir, kernel, reps):
    """The same golden (CombinedNoiseWrapper with its own normal draws replayed, evaluation/robustness_tests.py:177-207)
    served by the TMA/mbarrier step kernel: the six golden envs are tiled to 192 (288 for the 224-env tile: one full
    and one ragged tile) so that the batch is pipeline-sized, and the register-resident kernel is switched off for the test."""
    from dexterous_rl_manipulation_b200 import _lib
    g = _load(golden_dir, "noise.npz")
    n0, T = g["actions"].shape[:2]
    n = n0 * reps
    tile = lambda a: np.concatenate([a] * reps, axis=0)
    env = _make_env(dx, n, True, int(g["max_steps"]))
    obs0, _ = env.reset_from_draws(tile(g["jp0"]), tile(g["size"]), tile(g["mass"]), tile(g["friction"]), tile(g["pos"]))
    _set_step_kernel(kernel)
    try:
        for t in range(T):
            obs, rew, te, tr, info = env.step(torch.from_numpy(tile(g["actions"][:, t])).cuda(),
                                              dyn_noise=tile(g["dyn_noise"][:, t]), obs_noise=tile(g["obs_noise"][:, t + 1]))
            assert np.array_equal(obs.cpu().numpy(), tile(g["obs"][:, t + 1])), t
            assert np.array_equal(te.cpu().numpy(), tile(g["terminated"][:, t]))
            assert np.array_equal(tr.cpu().numpy(), tile(g["truncated"][:, t]))
            assert np.array_equal(info["num_contacts"].cpu().numpy(), tile(g["num_contacts"][:, t]))
            np.testing.assert_allclose(rew.cpu().numpy(), tile(g["reward"][:, t]), rtol=REWARD_RTOL, atol=REWARD_ATOL)
    finally:
        _set_step_kernel("auto")


def _random_draws(rng, n, ragged=True):
    jp0 = rng.uniform(-0.1, 0.1, (n, 15)).astype(np.float32)
    size = rng.uniform(0.02, 0.12, n)
    mass = rng.uniform(0.05, 0.3, n)
    fric = rng.uniform(0.0, 1.0, n)
    pos = np.stack([rng.uniform(-0.1, 0.1, n), rng.uniform(-0.1, 0.1, n), rng.uniform(0.05, 0.2, n)], 1).astype(np.float32)
    if ragged:
        pos[::97] = [0.25, -0.3, 0.35]           # outside the workspace: exercises the clip + wall logic
        pos[5::101, 2] = 0.0
    return jp0, size, mass, fric, pos


def _set_step_kernel(impl):
    """'auto' | 'register' | 'tma' (narrow 128-env tiles) | 'tma_wide' (224-env tiles where that instantiation exists; full
    tracking always runs on the narrow tile)."""
    from dexterous_rl_manipulation_b200 import _lib
    _lib.set_step_impl("tma" if impl == "tma_wide" else impl)
    _lib.set_step_tile("wide" if impl == "tma_wide" else "narrow" if impl == "tma" else "auto")


@pytest.fixture
def step_impl():
    """Pin dexsim_step to one of its two kernels for a test (the auto choice goes by batch size: small batches take
    the register-resident kernel, large ones the TMA pipeline); restored afterwards."""
    from dexterous_rl_manipulation_b200 import _lib

    def choose(impl):
        # "tma_wide": the pipeline with its 224-env tiles (2 CTAs x 7 compute warps per SM) wherever that instantiation exists
        _lib.set_step_impl("tma" if impl == "tma_wide" else impl)
        _lib.set_step_tile("wide" if impl == "tma_wide" else "narrow" if impl == "tma" else "auto")
    yield choose
    _lib.set_step_impl("auto")
    _lib.set_step_tile("auto")


@pytest.mark.parametrize("n,dense,comps,impl", [(1, True, True, "auto"), (33, False, True, "auto"), (1000, True, True, "register"),
                                                (1000, True, True, "tma"), (4096, True, True, "tma"), (1000, True, False, "tma"),
                                                (4096, False, False, "tma"), (4096, False, False, "register"),
                                                (20000, True, False, "tma"), (20000, True, False, "auto"),
                                                (1000, True, True, "tma_wide"), (224 * 19 + 3, False, False, "tma_wide"),
                                                (20000, True, False, "tma_wide")])
def test_step_matches_oracle(dx, n, dense, comps, impl, step_impl):
    """Ragged batch sizes (1, 33, 1000 are not multiples of the warp / CTA size) vs the oracle, through both step
    kernels (with and without the reward-component outputs)."""
    from oracle import oracle
    step_impl(impl)
    rng = np.random.default_rng(n)
    jp0, size, mass, fric, pos = _random_draws(rng, n)
    ob = oracle.OracleBatch(n, dense=dense, max_episode_steps=60)
    o0 = ob.reset_predrawn(jp0, size, mass, fric, pos)
    env = None
    if n > 1:
        env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=60, reward_type="dense" if dense else "sparse",
                                        reward_components=comps)
    if n == 1:
        env = dx.BatchedManipulationEnv(1, "cuda", max_episode_steps=60, reward_type="dense", reward_components=True)
    g0, _ = env.reset_from_draws(jp0, size, mass, fric, pos)
    g0 = g0 if n == 1 else g0.cpu().numpy()
    assert np.array_equal(np.asarray(g0).reshape(n, 45), o0)
    for t in range(90):
        a = rng.uniform(-1.3, 1.3, (n, 15)).astype(np.float32) if t % 3 else rng.normal(0, 0.4, (n, 15)).astype(np.float32)
        if t == 7:
            a[0, 0] = np.nan                     # NaN actions propagate through np.clip in the reference
        oo, orr, oc, ote, otr, onc = ob.step(a)
        if n == 1:
            obs, rew, te, tr, info = env.step(a[0])
            assert np.array_equal(obs, oo[0], equal_nan=True)
            assert te == ote[0] and tr == otr[0] and info["num_contacts"] == onc[0]
            assert rew == pytest.approx(orr[0], rel=REWARD_RTOL, abs=REWARD_ATOL, nan_ok=True)
            assert np.array_equal(info["object_position"], ob.env["op"][0])
        else:
            obs, rew, te, tr, info = env.step(torch.from_numpy(a).cuda())
            assert np.array_equal(obs.cpu().numpy(), oo, equal_nan=True), t
            assert np.array_equal(te.cpu().numpy(), ote) and np.array_equal(tr.cpu().numpy(), otr)
            assert np.array_equal(info["num_contacts"].cpu().numpy(), onc)
            np.testing.assert_allclose(rew.cpu().numpy(), orr, rtol=REWARD_RTOL, atol=REWARD_ATOL)
            assert np.array_equal(info["object_position"].cpu().numpy(), ob.env["op"])


def _oracle_groups(cfgs, sigma_dyn=0.0):
    from oracle import oracle
    return np.concatenate([oracle.make_group(c, sigma_dyn=sigma_dyn) for c in cfgs])


@pytest.mark.parametrize("policy,dense,respawn,n", [("random", True, True, 4096), ("heuristic", True, True, 3000),
                                                     ("heuristic", False, False, 777), ("random", True, False, 64)])
def test_fused_rollout_matches_oracle(dx, policy, dense, respawn, n):
    """K-step fused kernel (in-kernel Philox policy, auto-reset, counters) vs the oracle's rollout."""
    from oracle import oracle
    CC = dx.CurriculumConfig
    cfgs = [CC.easy(), CC.medium(), CC.hard(),
            CC(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))]
    seed, K, max_steps = 1234, 130, 50
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense" if dense else "sparse",
                                    track_episodes=True, groups=cfgs, seed=seed, env_gid0=5)
    env.reset(seed=seed)
    ob = oracle.OracleBatch(n, dense=dense, max_episode_steps=max_steps)
    groups = _oracle_groups(cfgs)
    draws = [oracle.reset_draws(seed, 5 + i, 0, groups[(5 + i) % 4:(5 + i) % 4 + 1]) for i in range(n)]
    ob.reset_predrawn(np.stack([d[0] for d in draws]), np.array([d[1] for d in draws]), np.array([d[2] for d in draws]),
                      np.array([d[3] for d in draws]), np.stack([d[4] for d in draws]))
    assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), ob.observation())
    kind = 1 if policy == "random" else 2
    cnt_o = rs_o = None
    for chunk in (K // 2, K - K // 2):               # two launches: state must survive the round trip
        env.rollout(chunk, policy=policy, respawn=respawn)
        cnt_o, rs_o = ob.rollout(groups, chunk, seed, policy_kind=kind, respawn=respawn, env_gid0=5,
                                 loop_max_steps=max_steps, counters=cnt_o, ret_sums=rs_o)
    cnt = env.counters.cpu().numpy()
    assert cnt[:, 0].sum() > n, "episodes must have finished and auto-reset"
    assert np.array_equal(cnt[:, :16], cnt_o[:, :16]) and np.array_equal(cnt[:, 17], cnt_o[:, 17])
    assert cnt[:, 16].sum() == 0                     # no variance ties in real rollouts
    np.testing.assert_allclose(env.ret_sums.cpu().numpy(), rs_o, rtol=1e-9)
    assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), ob.observation())
    assert np.array_equal(env._op64[:, :n].t().cpu().numpy(), ob.env["op"])
    assert np.array_equal(env._episode[:n].cpu().numpy().astype(np.uint32), ob.env["episode"])
    assert np.array_equal(env._step_count[:n].cpu().numpy(), ob.env["step_count"])
    np.testing.assert_allclose(env._ep_return[:n].cpu().numpy(), ob.env["ep_return"], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("impl", ["register", "tma", "tma_wide"])
def test_step_autoreset_equals_fused_rollout(dx, impl, step_impl):
    """Stepping with the exposed Philox actions + in-kernel auto-reset == the fused rollout kernel."""
    step_impl(impl)
    from dexterous_rl_manipulation_b200 import _lib
    import ctypes as C
    CC = dx.CurriculumConfig
    n, K, seed = 2048, 75, 99
    kw = dict(max_episode_steps=40, reward_type="dense", track_episodes=True, groups=[CC.easy(), CC.hard()], seed=seed)
    a = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, respawn=True, loop_max_steps=40, **kw)
    b = dx.BatchedManipulationEnv(n, "cuda", **kw)
    a.reset(seed=seed); b.reset(seed=seed)
    act = torch.zeros(15, a.ld, device="cuda")
    fin = 0
    for t in range(K):
        _lib.check(a._lib.dexsim_fill_policy_actions(C.byref(a._state), C.byref(a._params), 2, act.data_ptr(), a._stream()), "fill")
        obs, rew, te, tr, info = a.step(act[:, :n].t().contiguous())
        fin += int(info["finished"].sum())
    b.rollout(K, policy="heuristic", respawn=True, loop_max_steps=40)
    assert fin == int(b.counters[:, 0].sum()) and fin > 0
    assert torch.equal(a.counters, b.counters)
    assert torch.equal(a._obs, b._obs) and torch.equal(a._op64, b._op64) and torch.equal(a._episode, b._episode)
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0)


@pytest.mark.parametrize("impl", ["register", "tma", "tma_wide"])
def test_noisy_step_equals_noisy_fused_rollout(dx, impl, step_impl):
    """Dynamics-noise cells (per-group sigma): API stepping with in-kernel noise == the fused rollout kernel's noise --
    two independent code paths drawing from the same Philox stream keyed by (env, episode, step)."""
    step_impl(impl)
    from dexterous_rl_manipulation_b200 import _lib
    import ctypes as C
    CC = dx.CurriculumConfig
    n, K, seed = 1536, 70, 21
    kw = dict(max_episode_steps=30, reward_type="dense", track_episodes=True, groups=[CC.easy(), CC.medium(), CC.hard()],
              group_sigma_dyn=[0.0, 0.05, 0.2], seed=seed)
    a = dx.BatchedManipulationEnv(n, "cuda", auto_reset=True, respawn=True, loop_max_steps=30, **kw)
    b = dx.BatchedManipulationEnv(n, "cuda", **kw)
    a.reset(seed=seed); b.reset(seed=seed)
    act = torch.zeros(15, a.ld, device="cuda")
    for t in range(K):
        _lib.check(a._lib.dexsim_fill_policy_actions(C.byref(a._state), C.byref(a._params), 1, act.data_ptr(), a._stream()), "fill")
        a.step(act[:, :n].t().contiguous())
    b.rollout(K, policy="random", respawn=True, loop_max_steps=30)
    assert torch.equal(a.counters, b.counters) and int(a.counters[:, 0].sum()) > n
    assert torch.equal(a._obs, b._obs) and torch.equal(a._op64, b._op64) and torch.equal(a._episode, b._episode)
    quiet = dx.BatchedManipulationEnv(n, "cuda", **dict(kw, group_sigma_dyn=0.0))
    quiet.reset(seed=seed); quiet.rollout(K, policy="random", respawn=True, loop_max_steps=30)
    assert torch.equal(quiet._obs[:, 0::3], b._obs[:, 0::3])           # group 0 (sigma 0) is untouched by the others' noise
    assert not torch.equal(quiet._obs[:, 2::3], b._obs[:, 2::3])


def test_sharding_is_gpu_count_independent(dx):
    """Two half shards keyed by global env id reproduce one full shard (SURVEY.md 8e)."""
    CC = dx.CurriculumConfig
    N, K, seed = 6000, 60, 7
    kw = dict(max_episode_steps=30, reward_type="dense", track_episodes=True, seed=seed,
              groups=[CC.easy(), CC.medium(), CC.hard()])
    full = dx.BatchedManipulationEnv(N, "cuda", **kw)
    full.reset(seed=seed); full.rollout(K, policy="random")
    cnt = torch.zeros_like(full.counters)
    obs = []
    for r in range(3):
        lo, hi = dx.distributed.shard_range(N, r, 3)
        sh = dx.BatchedManipulationEnv(hi - lo, "cuda", env_gid0=lo, **kw)
        sh.reset(seed=seed); sh.rollout(K, policy="random")
        cnt += sh.counters
        obs.append(sh._obs[:, :hi - lo])
    assert torch.equal(cnt, full.counters)
    assert torch.equal(torch.cat(obs, 1), full._obs[:, :N])


def test_full_size_properties(dx):
    """BASELINE.json's largest per-GPU size (1,048,576 envs): size-independent invariants plus a
    2,048-env sample replayed through the oracle."""
    from oracle import oracle
    N, seed, T = 1 << 20, 11, 12
    cfg = dx.CurriculumConfig(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))
    env = dx.BatchedManipulationEnv(N, "cuda", max_episode_steps=200, reward_type="dense", curriculum_config=cfg, seed=seed)
    obs, _ = env.reset(seed=seed)
    pick = torch.from_numpy(np.random.default_rng(0).choice(N, 2048, replace=False)).cuda()
    ob = oracle.OracleBatch(2048, dense=True, max_episode_steps=200)
    o0 = ob.reset_predrawn(obs[pick, :15].cpu().numpy(), env._size[pick].cpu().numpy(), env._mass[pick].cpu().numpy(),
                           env._friction[pick].cpu().numpy(), obs[pick, 30:33].cpu().numpy())
    assert np.array_equal(o0, obs[pick].cpu().numpy())
    gen = torch.Generator(device="cuda").manual_seed(3)
    ret = torch.zeros(N, dtype=torch.float64, device="cuda")
    for t in range(T):
        a = torch.rand(N, 15, device="cuda", generator=gen) * 2.4 - 1.2
        obs, rew, te, tr, info = env.step(a)
        ret += rew
        oo, orr, _, ote, otr, onc = ob.step(a[pick].cpu().numpy())
        assert np.array_equal(obs[pick].cpu().numpy(), oo)
        assert np.array_equal(te[pick].cpu().numpy(), ote) and np.array_equal(info["num_contacts"][pick].cpu().numpy(), onc)
        np.testing.assert_allclose(rew[pick].cpu().numpy(), orr, rtol=REWARD_RTOL, atol=REWARD_ATOL)
    assert int(info["step_count"].min()) == T and int(info["step_count"].max()) == T
    assert float(obs[:, :15].abs().max()) <= 1.0
    assert torch.equal(obs[:, 33:37], torch.tensor([1.0, 0, 0, 0], device="cuda").expand(N, 4))
    bits = torch.stack([((env._cmask[:N] >> f) & 1).to(torch.float32) for f in range(5)], 1)
    assert torch.equal(obs[:, 40:45], bits)
    assert torch.equal(info["num_contacts"].to(torch.int64), bits.sum(1).to(torch.int64))
    assert torch.equal(te, info["num_contacts"] >= 3)
    assert float(obs[:, 32].min()) >= 0.0 and float(obs[:, 32].max()) <= 0.3 + 1e-7
    assert torch.equal(obs[:, 30:33], env._op64[:, :N].t().to(torch.float32))
    assert torch.isfinite(ret).all()


def test_philox_and_normal_streams(dx):
    from dexterous_rl_manipulation_b200 import _lib
    from oracle import oracle
    import ctypes as C
    n, seed = 5000, 77
    env = dx.BatchedManipulationEnv(n, "cuda", seed=seed, env_gid0=123)
    env.reset(seed=seed)
    act = torch.zeros(15, env.ld, device="cuda")
    for kind in (1, 2):
        _lib.check(env._lib.dexsim_fill_policy_actions(C.byref(env._state), C.byref(env._params), kind, act.data_ptr(), env._stream()), "fill")
        got = act[:, :64].t().cpu().numpy()
        exp = np.stack([oracle.policy_action(seed, 123 + i, 0, 0, kind) for i in range(64)])
        assert np.array_equal(got, exp)
    z = torch.zeros(45, env.ld, device="cuda")
    _lib.check(env._lib.dexsim_fill_normal(C.byref(env._state), C.byref(env._params), 3, 45, C.c_float(0.5), z.data_ptr(), env._stream()), "fill")
    zz = z[:, :n]
    assert abs(float(zz.mean())) < 0.005 and abs(float(zz.std()) - 0.5) < 0.005
    assert abs(float((zz / 0.5).pow(4).mean()) - 3.0) < 0.1                        # kurtosis of a normal
    assert abs(float(torch.corrcoef(zz[:2])[0, 1])) < 0.05


def test_dropin_under_reference_callers(dx, golden_dir):
    """num_envs == 1 through the Gymnasium API: replay the Evaluator / run_episode goldens with the
    callers' loop shape; when the byte-compiled reference is present, run the UNMODIFIED callers."""
    g = _load(golden_dir, "episodes.npz")
    prev = None
    for i in range(g["kind"].shape[0]):
        if g["keep_pos"][i]:
            env = prev
            obs, info = env.reset_from_draws(g["jp0"][i][None], g["size"][i:i + 1], g["mass"][i:i + 1], g["friction"][i:i + 1], None)
        else:
            env = dx.BatchedManipulationEnv(1, "cuda", max_episode_steps=int(g["max_steps"][i]),
                                            reward_type="dense" if g["dense"][i] else "sparse")
            obs, info = env.reset_from_draws(g["jp0"][i][None], g["size"][i:i + 1], g["mass"][i:i + 1], g["friction"][i:i + 1], g["pos"][i][None])
        total, steps, success = 0.0, 0, False
        for t in range(int(g["loop_max_steps"][i])):
            obs, r, te, tr, info = env.step(g["actions"][i, t])
            total += r; steps += 1
            if te or tr:
                success = te
                break
        assert steps == g["n_steps"][i]
        assert info["num_contacts"] == g["final_contacts"][i]
        if g["kind"][i] == 0:
            assert success == g["success"][i]
        assert total == pytest.approx(g["episode_reward"][i], rel=1e-5)
        prev = env


def test_unmodified_reference_callers_when_available(dx):
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("reference (source or byte-compiled) not present")
    R = ref_harness.load()
    make = lambda **kw: dx.BatchedManipulationEnv(1, "cuda", **kw)
    # run_episode (training/episode_utils.py:13-55) on a reused env, reference vs drop-in
    for cfg in (R.CurriculumConfig.easy(), R.CurriculumConfig.hard()):
        out = []
        for factory in (R.DexterousManipulationEnv, make):
            np.random.seed(3)
            env = factory(curriculum_config=cfg, reward_type="dense", max_episode_steps=60)
            pol = R.policies.HeuristicPolicy(env.action_space)
            res = []
            for ep in range(3):
                if factory is make:
                    env._host_rngs(100 + ep)
                else:
                    env._np_random = np.random.Generator(np.random.PCG64(np.random.SeedSequence(100 + ep)))
                res.append(R.episode_utils.run_episode(env, pol, max_steps=60))
            out.append(res)
        for (s0, n0, r0), (s1, n1, r1) in zip(*out):
            assert (s0, n0) == (s1, n1) and r1 == pytest.approx(r0, rel=1e-5)
    # Evaluator.evaluate_heldout_set (evaluation/evaluator.py:191-271) with the env class swapped
    train = R.CurriculumConfig(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))
    held = R.heldout_objects.HeldOutObjectSet(train_config=train, eval_size_range=(0.03, 0.09), num_heldout_objects=4, seed=5)
    results = []
    orig = R.evaluator.DexterousManipulationEnv
    for factory in (orig, make):
        R.evaluator.DexterousManipulationEnv = factory
        try:
            np.random.seed(0)
            probe = orig()
            ev = R.evaluator.Evaluator(R.policies.HeuristicPolicy(probe.action_space), held, reward_type="dense", max_episode_steps=50)
            results.append(ev.evaluate_heldout_set(num_episodes_per_object=2, seed=42))
        finally:
            R.evaluator.DexterousManipulationEnv = orig
    ref, got = results
    assert ref["metrics"]["grasp_success_rate"] == got["metrics"]["grasp_success_rate"]
    assert ref["metrics"]["failure_type_frequency"] == got["metrics"]["failure_type_frequency"]
    for e0, e1 in zip(ref["all_episodes"], got["all_episodes"]):
        assert e0["success"] == e1["success"] and e0["episode_steps"] == e1["episode_steps"]
        assert e0["contact_history"] == e1["contact_history"] and e0["final_contacts"] == e1["final_contacts"]
        assert e1["episode_reward"] == pytest.approx(e0["episode_reward"], rel=1e-5)
        assert e0["object_size"] == e1["object_size"] and e0["friction_coefficient"] == e1["friction_coefficient"]


@pytest.mark.parametrize("n,track,dense", [(128, False, True), (1000, False, False), (4096 + 77, True, True),
                                            (65536, True, True), (200_000, False, True), (4096 + 77, "counts", True),
                                            (70_000, "counts", False)])
def test_tma_pipeline_equals_register_kernel(dx, n, track, dense):
    """The TMA/mbarrier step kernel and the register-resident one must agree bit for bit on every
    array (full and ragged last tiles, AoS and SoA actions, with and without tracking/auto-reset)."""
    from dexterous_rl_manipulation_b200 import _lib
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=25, reward_type="dense" if dense else "sparse", seed=3, groups=[CC.easy(), CC.hard()])
    if track:       # "counts": auto-reset + counters without the per-env return / history arrays
        kw.update(auto_reset=True, respawn=True, loop_max_steps=25, track_episodes=track != "counts")
    envs = {}
    try:
        for impl in ("register", "tma", "tma_wide"):
            env = dx.BatchedManipulationEnv(n, "cuda", **kw)
            env.reset(seed=3)
            envs[impl] = env
        gen = torch.Generator(device="cuda").manual_seed(5)
        soa = torch.zeros(15, envs["tma"].ld, device="cuda")
        for t in range(60):
            a = torch.rand(n, 15, device="cuda", generator=gen) * 2.6 - 1.3
            outs = {}
            for impl, env in envs.items():
                _set_step_kernel(impl)
                if t % 2:
                    soa[:, :n] = a.t()
                    o = env._step_soa(soa)
                else:
                    o = env.step(a)
                outs[impl] = [x.clone() for x in o[:4]] + [o[4]["num_contacts"].clone()]
            for x, y, z in zip(outs["register"], outs["tma"], outs["tma_wide"]):
                assert torch.equal(x, y) and torch.equal(x, z), t
        a, b, w = envs["register"], envs["tma"], envs["tma_wide"]
        for name in ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode"):
            assert torch.equal(getattr(a, name), getattr(b, name)) and torch.equal(getattr(a, name), getattr(w, name)), name
        if track:
            assert torch.equal(a.counters, b.counters) and torch.equal(a.counters, w.counters) and int(a.counters[:, 0].sum()) > 0
        if track == "counts":
            # same trajectories as full tracking: episodes / successes / lengths agree, labels and returns stay empty
            full = dx.BatchedManipulationEnv(n, "cuda", **dict(kw, track_episodes=True))
            full.reset(seed=3)
            gen = torch.Generator(device="cuda").manual_seed(5)
            for t in range(60):
                full.step(torch.rand(n, 15, device="cuda", generator=gen) * 2.6 - 1.3)
            from dexterous_rl_manipulation_b200._lib import (CNT_EPISODES, CNT_LABEL_METRICS, CNT_SUCCESSES,
                                                             CNT_SUM_FINAL_CONTACTS, CNT_SUM_STEPS, CNT_SUM_STEPS_SQ)
            cols = [CNT_EPISODES, CNT_SUCCESSES, CNT_SUM_STEPS, CNT_SUM_STEPS_SQ, CNT_SUM_FINAL_CONTACTS]
            assert torch.equal(full.counters[:, cols], b.counters[:, cols])
            assert torch.equal(full._obs, b._obs) and torch.equal(full._episode, b._episode)
            assert int(b.counters[:, CNT_LABEL_METRICS:CNT_LABEL_METRICS + 13].sum()) == 0 and float(b.ret_sums.abs().sum()) == 0.0
            assert int(full.counters[:, CNT_LABEL_METRICS:CNT_LABEL_METRICS + 13].sum()) > 0
        elif track:
            assert torch.equal(a._ep_stats, b._ep_stats) and torch.equal(a._ep_return, b._ep_return)
            torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0)
    finally:
        _set_step_kernel("auto")


@pytest.mark.parametrize("n,track,ranged,respawn,predrawn", [(4096 + 77, False, False, True, False), (1000, True, False, True, False),
                                                            (70_000, "counts", True, True, False), (5000, True, True, False, False),
                                                            (3000, "counts", False, True, True)])
def test_tma_pipeline_noise_and_components_equal_register_kernel(dx, n, track, ranged, respawn, predrawn):
    """Noise (Philox in-kernel or pre-drawn), reward components and the float64 reward on the TMA pipeline
    (EXTRA instantiations) against the register-resident kernel: every output and every state array bit for bit,
    across auto-resets in both spawn modes and with ranged size / mass / friction groups (Philox blocks 5-6 of the
    reset draws)."""
    from dexterous_rl_manipulation_b200 import _lib
    CC = dx.CurriculumConfig
    g1 = CC(object_size_range=(0.03, 0.09), object_mass_range=(0.05, 0.3), friction_range=(0.2, 0.9)) if ranged else CC.hard()
    kw = dict(max_episode_steps=20, reward_type="dense", seed=11, groups=[CC.easy(), g1], reward_components=True)
    if not predrawn:
        kw.update(observation_noise_std=0.05, dynamics_noise_std=0.1)
    if track:
        kw.update(auto_reset=True, respawn=respawn, loop_max_steps=20, track_episodes=track != "counts")
    envs = {}
    try:
        for impl in ("register", "tma", "tma_wide"):
            env = dx.BatchedManipulationEnv(n, "cuda", **kw)
            env.reset(seed=11)
            envs[impl] = env
        gen = torch.Generator(device="cuda").manual_seed(8)
        for t in range(50):
            a = torch.rand(n, 15, device="cuda", generator=gen) * 2.6 - 1.3
            extra = {}
            if predrawn:
                extra = dict(dyn_noise=torch.randn(n, 15, device="cuda", generator=gen) * 0.1,
                             obs_noise=torch.randn(n, 45, device="cuda", generator=gen) * 0.05)
            outs = {}
            for impl, env in envs.items():
                _set_step_kernel(impl)
                o = env.step(a, **extra)
                rc = o[4]["reward_components"]
                outs[impl] = [x.clone() for x in o[:4]] + [o[4]["num_contacts"].clone()] + [rc[k].clone() for k in ("distance", "contact", "closure", "stability")]
            for x, y, z in zip(outs["register"], outs["tma"], outs["tma_wide"]):
                assert torch.equal(x, y) and torch.equal(x, z), t
        a, b, w = envs["register"], envs["tma"], envs["tma_wide"]
        for name in ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode", "_noisy_obs"):
            assert torch.equal(getattr(a, name), getattr(b, name)) and torch.equal(getattr(a, name), getattr(w, name)), name
        if track:
            assert torch.equal(a.counters, b.counters) and torch.equal(a.counters, w.counters) and int(a.counters[:, 0].sum()) > n
        if track is True:
            assert torch.equal(a._ep_stats, b._ep_stats) and torch.equal(a._ep_return, b._ep_return)
    finally:
        _set_step_kernel("auto")


@pytest.mark.parametrize("n,track", [(1000, False), (4096 + 5, True)])
@pytest.mark.parametrize("impl", ["register", "tma", "tma_wide"])
def test_in_kernel_noise_equals_separate_noise_kernels(dx, n, track, impl, step_impl):
    """DexsimStepIO.sigma_dyn / sigma_obs (Philox normals drawn inside the step kernel) give exactly what the
    separate dexsim_fill_normal launches + add give: same streams, same counters, also across auto-resets."""
    step_impl(impl)
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=20, reward_type="dense", seed=9, curriculum_config=CC.easy(),
              observation_noise_std=0.05, dynamics_noise_std=0.1)
    if track:
        kw.update(auto_reset=True, respawn=True, loop_max_steps=20, track_episodes=True)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    b.fused_noise = False
    oa, _ = a.reset(seed=9)
    ob, _ = b.reset(seed=9)
    assert torch.equal(oa, ob)
    gen = torch.Generator(device="cuda").manual_seed(2)
    for t in range(50):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2.4 - 1.2
        ra, rb = a.step(act), b.step(act)
        for x, y in zip(ra[:4], rb[:4]):
            assert torch.equal(x, y), t
        assert torch.equal(ra[4]["num_contacts"], rb[4]["num_contacts"])
    assert not torch.equal(ra[0], a._obs[:, :n].t())                  # the returned observation is the noisy one
    for name in ("_obs", "_op64", "_step_count", "_cmask", "_episode", "_noisy_obs"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    if track:
        assert torch.equal(a.counters, b.counters) and int(a.counters[:, 0].sum()) > n


@pytest.mark.parametrize("impl", ["register", "tma", "tma_wide"])
def test_group_noise_cells_in_step(dx, impl, step_impl):
    """Noise cells as groups of one batch (group_sigma_*), stepped through the API with external actions: every
    env behaves like the same env of a batch whose env-level noise is its group's value."""
    step_impl(impl)
    CC = dx.CurriculumConfig
    n, cfg = 2048, CC.medium()
    kw = dict(max_episode_steps=30, reward_type="dense", seed=4)
    cells = dx.BatchedManipulationEnv(n, "cuda", groups=[cfg, cfg], group_sigma_obs=[0.02, 0.0], group_sigma_dyn=[0.0, 0.1], **kw)
    only_obs = dx.BatchedManipulationEnv(n, "cuda", groups=[cfg, cfg], observation_noise_std=0.02, **kw)
    only_dyn = dx.BatchedManipulationEnv(n, "cuda", groups=[cfg, cfg], dynamics_noise_std=0.1, **kw)
    for e in (cells, only_obs, only_dyn):
        e.reset(seed=4)
    gen = torch.Generator(device="cuda").manual_seed(6)
    for t in range(30):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
        rc, ro, rd = cells.step(act), only_obs.step(act), only_dyn.step(act)
        assert torch.equal(rc[0][0::2], ro[0][0::2]) and torch.equal(rc[1][0::2], ro[1][0::2]), t     # group 0: sigma_obs
        assert torch.equal(rc[0][1::2], rd[0][1::2]) and torch.equal(rc[1][1::2], rd[1][1::2]), t     # group 1: sigma_dyn
    assert torch.equal(cells._obs[:, 0:n:2], only_obs._obs[:, 0:n:2])
    assert torch.equal(cells._obs[:, 1:n:2], only_dyn._obs[:, 1:n:2])
    assert not torch.equal(cells._obs[:, 1:n:2], only_obs._obs[:, 1:n:2])       # dynamics noise did change trajectories


def test_c_abi_demo_matches_python_face(dx, tmp_path):
    """examples/c_abi_demo.c drives libdexsim_b200.so from plain C (cudaMalloc buffers, no Python, no torch);
    its counters and observation checksum equal the Python face's on the same configuration."""
    import json
    import shutil
    import subprocess
    from dexterous_rl_manipulation_b200 import _lib
    import ctypes as C
    if not shutil.which("gcc"):
        pytest.skip("gcc not available")
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    exe = str(tmp_path / "c_abi_demo")
    libdir = os.path.join(root, "dexterous_rl_manipulation_b200")
    subprocess.run(["gcc", "-O2", "-std=c99", "-Wall", "-Werror", f"-I{root}/include", f"-I{cuda}/include",
                    os.path.join(root, "examples", "c_abi_demo.c"), "-o", exe, f"-L{libdir}", "-ldexsim_b200",
                    f"-L{cuda}/lib64", "-lcudart", f"-Wl,-rpath,{libdir}", f"-Wl,-rpath,{cuda}/lib64"], check=True)
    n, steps, seed = 5000, 120, 7
    out = json.loads(subprocess.run([exe, str(n), str(steps), str(seed)], check=True, capture_output=True, text=True,
                                    timeout=120).stdout)
    env = dx.BatchedManipulationEnv(n, "cuda", reward_type="dense", max_episode_steps=50, curriculum_config=dx.CurriculumConfig.hard(),
                                    auto_reset=True, respawn=True, loop_max_steps=50, track_episodes=False, seed=seed)
    env.reset(seed=seed)
    act = torch.zeros(15, env.ld, device="cuda")
    for _ in range(steps):
        _lib.check(env._lib.dexsim_fill_policy_actions(C.byref(env._state), C.byref(env._params), _lib.POLICY_RANDOM,
                                                       act.data_ptr(), env._stream()), "fill")
        env._step_soa(act)
    c = env.counters.cpu().numpy()[0]
    assert (out["episodes"], out["successes"], out["sum_steps"]) == (int(c[0]), int(c[1]), int(c[2])) and out["episodes"] >= n
    bits = env._obs[:, :n].t().contiguous().cpu().numpy().view(np.uint32).reshape(-1).copy()
    bits[bits == 0x80000000] = 0
    h = 1469598103934665603
    for byte in bits.view(np.uint8).tolist():                # little-endian bytes, env-major: the demo's order
        h = ((h ^ byte) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    assert out["obs_fnv1a"] == f"{h:016x}"


def test_maximum_size_batch(dx):
    """33.5 M envs in one batch (~11 GB of state, 7.7e9 bytes of observations, a ragged last tile): both step kernels
    agree on every array, and the LAST 1,000 envs equal a 1,000-env batch created with env_gid0 = n - 1000 --
    every index above 2^31 bytes / 2^25 columns goes through the same 64-bit arithmetic as the small ones."""
    from dexterous_rl_manipulation_b200 import _lib
    free, _ = torch.cuda.mem_get_info()
    if free < 40 * 2 ** 30:
        pytest.skip("needs 40 GB of free device memory")
    CC = dx.CurriculumConfig
    n, tail = (1 << 25) + 128 + 77, 1000
    kw = dict(max_episode_steps=3, reward_type="dense", seed=11, groups=[CC.easy(), CC.hard()],
              auto_reset=True, respawn=True, loop_max_steps=3, track_episodes=True)
    try:
        a = torch.rand(n, 15, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)) * 2.4 - 1.2
        small = dx.BatchedManipulationEnv(tail, "cuda", env_gid0=n - tail, **kw)
        small.reset(seed=11)
        for _ in range(5):
            small.step(a[n - tail:])
        ref = None
        for impl in ("register", "tma"):
            _lib.set_step_impl(impl)
            env = dx.BatchedManipulationEnv(n, "cuda", **kw)
            env.reset(seed=11)
            for _ in range(5):                      # episodes are 3 steps long: every env resets at least once
                out = env.step(a)
            assert torch.equal(env._obs[:, n - tail:n], small._obs[:, :tail]), impl
            assert torch.equal(env._step_count[n - tail:n], small._step_count[:tail])
            assert torch.equal(env._episode[n - tail:n], small._episode[:tail])
            assert torch.equal(env._ep_return[n - tail:n], small._ep_return[:tail])
            assert torch.equal(out[1][n - tail:], small._step_out[1])
            assert int(env.counters[:, 0].sum()) >= n
            state = (env._obs, env._op64, env._step_count, env._cmask, env._episode, env._ep_return, env._ep_stats,
                     env._thr, env._size, env.counters.clone(), out[1], out[2], out[3])
            if ref is None:
                ref = state
            else:
                for k, (x, y) in enumerate(zip(ref, state)):
                    assert torch.equal(x, y), k
            del env
    finally:
        _lib.set_step_impl("auto")


@pytest.mark.parametrize("n,chunks", [(40_000 + 77, None), (70_000, 4)])
def test_step_host_on_the_wide_tile(dx, n, chunks):
    """Host transports (zero-copy: the kernel's own bulk stores into the pinned buffers; copy: chunked sub-batches) with the
    224-env tile forced, against the device API stepping a twin env on the 128-env tile."""
    from dexterous_rl_manipulation_b200 import _lib
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=20, reward_type="dense", seed=8, groups=[CC.easy(), CC.hard()],
              auto_reset=True, respawn=True, loop_max_steps=20, track_episodes=False)
    a_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    b_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    a_env.reset(seed=8); b_env.reset(seed=8)
    rng = np.random.default_rng(1)
    try:
        for t in range(45):
            act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
            _set_step_kernel("tma")
            o1, r1, te1, tr1, i1 = a_env.step(torch.from_numpy(act).cuda())
            _set_step_kernel("auto")
            _lib.set_step_tile("wide")
            o2, r2, te2, tr2, i2 = b_env.step_host(torch.from_numpy(act).pin_memory(), chunks=chunks)
            assert torch.equal(o1.cpu(), o2) and torch.equal(r1.cpu(), r2), t
            assert torch.equal(te1.cpu(), te2) and torch.equal(tr1.cpu(), tr2)
            assert torch.equal(i1["num_contacts"].cpu(), i2["num_contacts"])
        assert torch.equal(a_env._obs, b_env._obs) and torch.equal(a_env._op64, b_env._op64)
        assert torch.equal(a_env.counters, b_env.counters) and int(a_env.counters[:, 0].sum()) > n
    finally:
        _set_step_kernel("auto")


@pytest.mark.parametrize("n,chunks,track", [(5000, 3, True), (4096, 1, False), (70_000, 8, True), (100, 1, True)])
def test_step_host_matches_device_step(dx, n, chunks, track):
    """The end-to-end entry (host buffers, chunked copy/compute overlap) equals the device-tensor API."""
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=20, reward_type="dense", seed=8, groups=[CC.easy(), CC.hard()])
    if track:
        kw.update(auto_reset=True, respawn=True, loop_max_steps=20, track_episodes=True)
    a_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    b_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    a_env.reset(seed=8); b_env.reset(seed=8)
    rng = np.random.default_rng(1)
    for t in range(45):
        act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
        o1, r1, te1, tr1, i1 = a_env.step(torch.from_numpy(act).cuda())
        o2, r2, te2, tr2, i2 = b_env.step_host(torch.from_numpy(act).pin_memory(), chunks=chunks)
        assert not o2.is_cuda
        assert torch.equal(o1.cpu(), o2) and torch.equal(r1.cpu(), r2), t
        assert torch.equal(te1.cpu(), te2) and torch.equal(tr1.cpu(), tr2)
        assert torch.equal(i1["num_contacts"].cpu(), i2["num_contacts"])
    assert torch.equal(a_env._obs, b_env._obs) and torch.equal(a_env._op64, b_env._op64)
    assert torch.equal(a_env._episode, b_env._episode)
    if track:
        assert torch.equal(a_env.counters, b_env.counters) and int(a_env.counters[:, 0].sum()) > 0
    # The default transport does not download the rows that only change at a reset (object x, y and their velocities: the
    # step kernel mirrors them into the pinned observation) once the buffer is current; every other entry point that
    # touches the state must make the next call download them again: an explicit reset, a device-side step, a rollout.
    a_env.reset(seed=77); b_env.reset(seed=77)
    for t in range(30):
        act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
        if t in (7, 19):                              # device-side step in between (changes the state behind the host buffer)
            a_env.step(torch.from_numpy(act).cuda()); b_env.step(torch.from_numpy(act).cuda())
            act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
        if t == 13:
            a_env.reset(seed=5); b_env.reset(seed=5)
        o1, r1, te1, tr1, i1 = a_env.step(torch.from_numpy(act).cuda())
        o2, r2, te2, tr2, i2 = b_env.step_host(torch.from_numpy(act).pin_memory(), chunks=chunks)
        assert torch.equal(o1.cpu(), o2) and torch.equal(r1.cpu(), r2), t
        assert b_env._h_primed_slot == 0
    # asynchronous, double-buffered and with the contacts packed into their 1-byte mask: same results
    pins = [torch.empty(n, 15).pin_memory() for _ in range(2)]
    pending = None
    for t in range(12):
        act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
        o1, r1, te1, tr1, i1 = a_env.step(torch.from_numpy(act).cuda())
        expect = (o1.cpu().clone(), r1.cpu().clone(), te1.cpu().clone(), tr1.cpu().clone(), i1["num_contacts"].cpu().clone())
        pins[t % 2].copy_(torch.from_numpy(act))
        out = b_env.step_host(pins[t % 2], chunks=chunks, sync=False, packed_contacts=True, slot=t % 2)
        if pending is not None:                     # the previous step's results (other slot) are still intact
            po, pe = pending
            assert torch.equal(po[1], pe[1]) and torch.equal(po[2], pe[2])
        b_env.host_sync()
        o2 = b_env.expand_contacts_host(slot=t % 2)
        assert torch.equal(o2, expect[0]) and torch.equal(out[1], expect[1]), t
        assert torch.equal(out[2], expect[2]) and torch.equal(out[3], expect[3]) and torch.equal(out[4]["num_contacts"], expect[4])
        assert torch.equal(out[4]["contact_mask"], a_env._cmask[:n].cpu())
        pending = (out, expect)
    assert torch.equal(a_env._obs, b_env._obs)


@pytest.mark.parametrize("n,track,chunks,impl", [
    pytest.param(5000, True, None, "auto", id="5000-True"),
    pytest.param(70_001, True, None, "auto", id="70001-True"),
    pytest.param(4096, False, None, "auto", id="4096-False"),
    # three chunks of 1,024 envs and one of 50: the last one, below a tile, is folded into its neighbour
    pytest.param(3122, True, 4, "auto", id="fold"),
    # the register-resident kernel selected: not eligible, every call takes the copy transport
    pytest.param(5000, True, 3, "register", id="ineligible"),
])
def test_step_host_zero_copy_launch(dx, n, track, chunks, impl):
    """DEXSIM_HOST_ZERO_COPY: once the pinned buffers are current and the actions are pinned too, a synchronous step_host
    uploads the actions with the copy engine and is then ONE kernel launch per chunk that writes every result into host
    memory -- same results as the device-tensor API, entry by entry, through resets, and the device-side state stays
    identical.  A call the pipelined kernel does not take runs the copy transport with the same results."""
    from dexterous_rl_manipulation_b200 import _lib
    L = _lib.lib()
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=15, reward_type="dense", seed=21, groups=[CC.easy(), CC.hard()])
    if track:
        kw.update(auto_reset=True, respawn=True, loop_max_steps=15, track_episodes=True)
    a_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    b_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    a_env.reset(seed=21); b_env.reset(seed=21)
    b_env.host_zero_copy = True                      # (default "auto": on up to 160K envs)
    rng = np.random.default_rng(4)
    pins = [torch.empty(n, 15).pin_memory() for _ in range(2)]
    _lib.set_step_impl(impl)
    try:
        before = int(L.dexsim_host_zero_copy_steps())
        for t in range(50):
            act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
            if t == 23:                                   # a device-side step behind the host buffer: next call re-primes
                a_env.step(torch.from_numpy(act).cuda()); b_env.step(torch.from_numpy(act).cuda())
                act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
            if t == 31:
                a_env.reset(seed=6); b_env.reset(seed=6)
            pins[t % 2].copy_(torch.from_numpy(act))
            o1, r1, te1, tr1, i1 = a_env.step(torch.from_numpy(act).cuda())
            o2, r2, te2, tr2, i2 = b_env.step_host(pins[t % 2], chunks=chunks)
            assert torch.equal(o1.cpu(), o2), (t, (o1.cpu() != o2).nonzero()[:5])
            assert torch.equal(r1.cpu(), r2) and torch.equal(te1.cpu(), te2) and torch.equal(tr1.cpu(), tr2), t
            assert torch.equal(i1["num_contacts"].cpu(), i2["num_contacts"]), t
            assert torch.equal(i2["contact_mask"], a_env._cmask[:n].cpu()), t
        # 50 calls, three of them priming downloads (first call, after the device-side step, after the reset)
        assert int(L.dexsim_host_zero_copy_steps()) - before == (0 if impl == "register" else 47)
        assert torch.equal(a_env._obs, b_env._obs) and torch.equal(a_env._op64, b_env._op64)
        assert torch.equal(a_env._episode, b_env._episode) and torch.equal(a_env._cmask, b_env._cmask)
        if track:
            assert torch.equal(a_env.counters, b_env.counters) and int(a_env.counters[:, 0].sum()) > 0
        # switched off: the copy transport, same results
        b_env.host_zero_copy = False
        before = int(L.dexsim_host_zero_copy_steps())
        for t in range(5):
            act = rng.uniform(-1.2, 1.2, (n, 15)).astype(np.float32)
            pins[t % 2].copy_(torch.from_numpy(act))
            o1, r1, te1, tr1, i1 = a_env.step(torch.from_numpy(act).cuda())
            o2, r2, te2, tr2, i2 = b_env.step_host(pins[t % 2], chunks=chunks)
            assert torch.equal(o1.cpu(), o2) and torch.equal(r1.cpu(), r2), t
        assert int(L.dexsim_host_zero_copy_steps()) == before
    finally:
        _lib.set_step_impl("auto")


class _PatternPolicy:
    """Deterministic, observation-independent policy (step-indexed pattern) usable on both sides."""

    def __init__(self, T):
        t = np.arange(T, dtype=np.float32)[:, None]
        j = np.arange(15, dtype=np.float32)[None, :]
        self.table = (-0.55 + 0.5 * np.sin(0.37 * t + 0.9 * j)).astype(np.float32)
        self.t = 0

    def reset(self):
        self.t = 0

    def select_action(self, obs):
        a = self.table[self.t]
        self.t += 1
        return a


def test_batched_evaluator_front_end_matches_reference(dx):
    """evaluate_heldout_set_batched (one fused launch for all objects x episodes) against the UNMODIFIED
    Evaluator.evaluate_heldout_set, and the reference's metrics code running on the batched output."""
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("reference (source or byte-compiled) not present")
    R = ref_harness.load()
    T, n_eps = 60, 3
    train = R.CurriculumConfig(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))
    held = R.heldout_objects.HeldOutObjectSet(train_config=train, eval_size_range=(0.025, 0.09), num_heldout_objects=6, seed=5)
    pol = _PatternPolicy(T)
    for reward_type in ("dense", "sparse"):
        ref = R.evaluator.Evaluator(pol, held, reward_type=reward_type, max_episode_steps=T).evaluate_heldout_set(n_eps, seed=42)
        n = 6 * n_eps
        actions = np.broadcast_to(pol.table[:, None, :], (T, n, 15)).copy()
        got = dx.evaluation.evaluate_heldout_set_batched(held, policy="external", actions=actions, num_episodes_per_object=n_eps,
                                                         seed=42, reward_type=reward_type, max_episode_steps=T)
        assert len(ref["all_episodes"]) == len(got["all_episodes"]) == n
        assert any(not e["success"] for e in ref["all_episodes"]) and any(e["success"] for e in ref["all_episodes"])
        for e0, e1 in zip(ref["all_episodes"], got["all_episodes"]):
            for k in ("episode_steps", "success", "num_contacts", "final_contacts", "contact_history", "object_size",
                      "object_mass", "friction_coefficient", "object_idx", "episode"):
                assert e0[k] == e1[k], k
            assert e1["episode_reward"] == pytest.approx(e0["episode_reward"], rel=1e-12, abs=1e-12)
        for k, v in ref["metrics"].items():
            assert got["metrics"][k] == (pytest.approx(v) if isinstance(v, float) else v), k
        assert got["overall_stats"]["overall_success_rate"] == ref["overall_stats"]["overall_success_rate"]
        assert got["overall_stats"]["mean_reward"] == pytest.approx(ref["overall_stats"]["mean_reward"], rel=1e-12)
        for o in ref["per_object_results"]:
            assert got["per_object_results"][o]["success_rate"] == ref["per_object_results"][o]["success_rate"]
            assert got["per_object_metrics"][o]["failure_type_frequency"] == ref["per_object_metrics"][o]["failure_type_frequency"]
        # the reference's own analysis code runs unchanged on the batched output
        again = R.metrics.EvaluationMetrics(3).compute_aggregate_metrics(got["all_episodes"], max_steps=T)
        assert again["failure_type_frequency"] == got["metrics"]["failure_type_frequency"]
        assert again["grasp_success_rate"] == got["metrics"]["grasp_success_rate"]
        assert isinstance(R.metrics.format_metrics_report(got["metrics"]), str)
        # one shard per GPU: three slices of the batch merged give the same records as the single batch
        from dexterous_rl_manipulation_b200.evaluation import _heldout_result
        merged = {}
        for r in range(3):
            part = dx.evaluation.evaluate_heldout_set_batched(held, policy="external", actions=actions, num_episodes_per_object=n_eps,
                                                              seed=42, reward_type=reward_type, max_episode_steps=T, shard=(r, 3))
            merged.update(part["shard_records"])
        again3 = _heldout_result(held, merged, n_eps, [42 + e for e in range(n_eps)], "external", 0, reward_type, T)
        assert again3["all_episodes"] == got["all_episodes"] and again3["metrics"] == got["metrics"]


def test_batched_robustness_front_end_matches_reference(dx):
    """evaluate_with_noise_batched with zero noise (deterministic) against RobustnessTester.evaluate_with_noise:
    one reused env object, reset(seed + episode), the object keeps its position after the first episode."""
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("reference (source or byte-compiled) not present")
    R = ref_harness.load()
    T, n_ep = 50, 6
    cfg = R.CurriculumConfig(object_size=0.045, object_mass=0.1, friction_coefficient=0.4)
    pol = _PatternPolicy(T)
    ref = R.robustness_tests.RobustnessTester(pol, cfg, reward_type="dense", max_episode_steps=T).evaluate_with_noise(
        0.0, 0.0, num_episodes=n_ep, seed=7)

    class _Ext:          # the front-end takes fused policies; feed the same table through a tiny shim
        pass

    import dexterous_rl_manipulation_b200.evaluation as ev
    orig = ev._run_one_episode_each
    table = torch.from_numpy(np.broadcast_to(pol.table[:, None, :], (T, 2, 15)).copy())
    ev._run_one_episode_each = lambda env, k, policy, respawn, lm, hist, kw: orig(env, k, "external", respawn, lm, hist,
                                                                                   {"actions": table})
    try:
        got = dx.evaluation.evaluate_with_noise_batched(cfg, "heuristic", 0.0, 0.0, num_episodes=n_ep, seed=7,
                                                        reward_type="dense", max_episode_steps=T)
    finally:
        ev._run_one_episode_each = orig
    assert len(got["episodes"]) == len(ref["episodes"]) == n_ep
    for e0, e1 in zip(ref["episodes"], got["episodes"]):
        for k in ("success", "episode_steps", "num_contacts", "final_contacts", "contact_history"):
            assert e0[k] == e1[k], k
        assert e1["episode_reward"] == pytest.approx(e0["episode_reward"], rel=1e-12, abs=1e-12)
    for k in ("grasp_success_rate", "mean_episode_length", "failure_type_frequency", "total_episodes"):
        assert got["metrics"][k] == ref["metrics"][k]
    # noisy cells: schema + sanity (dynamics noise is Philox, so only statistics are comparable)
    sweep = dx.evaluation.run_robustness_sweep_batched(cfg, [0.0, 0.05], [0.0, 0.1], policy="heuristic", num_episodes=4,
                                                       seed=3, max_episode_steps=T, num_replicas=8)
    assert set(sweep) == {"baseline", "observation_noise", "dynamics_noise", "combined_noise"}
    assert set(sweep["combined_noise"]) == {"obs_0.000_dyn_0.100", "obs_0.050_dyn_0.000", "obs_0.050_dyn_0.100"}
    assert sweep["dynamics_noise"][0.1]["metrics"]["total_episodes"] == 32
    assert sweep["dynamics_noise"][0.1]["noise_levels"] == {"observation_noise_std": 0.0, "dynamics_noise_std": 0.1}
    # replicas spread over ranks: three shards of 8 noisy replicas == the single batch, record for record
    whole = dx.evaluation.evaluate_with_noise_batched(cfg, "heuristic", 0.0, 0.1, num_episodes=4, seed=3, max_episode_steps=T,
                                                      num_replicas=8)
    merged = {}
    for r in range(3):
        merged.update(dx.evaluation.evaluate_with_noise_batched(cfg, "heuristic", 0.0, 0.1, num_episodes=4, seed=3,
                                                                max_episode_steps=T, num_replicas=8, shard=(r, 3))["shard_replicas"])
    assert [merged[r] for r in range(8)] == whole["replicas"]


def test_seed_variance_front_end_feeds_reference_statistics(dx):
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("reference (source or byte-compiled) not present")
    R = ref_harness.load()
    train = R.CurriculumConfig(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))
    held = R.heldout_objects.HeldOutObjectSet(train_config=train, eval_size_range=(0.03, 0.08), num_heldout_objects=5, seed=9)
    per_seed = dx.evaluation.evaluate_seeds_batched(held, [42, 123, 456], policy="heuristic", num_episodes_per_object=3,
                                                    max_episode_steps=80)
    analyzer = R.seed_variance.SeedVarianceAnalyzer(policy=None, heldout_set=held, reward_type="dense", max_episode_steps=80)
    stats = analyzer.compute_variance_statistics(per_seed)          # the reference's statistics, unchanged
    assert isinstance(stats, dict) and len(stats) > 0
    assert set(per_seed) == {42, 123, 456} and all(r["metrics"]["total_episodes"] == 15 for r in per_seed.values())


def test_fused_simple_learner_matches_reference_golden(dx, golden_dir):
    """rollout(policy="learner") with the reference learner's own normal draws replayed as pre-drawn tensors:
    episode length, final contacts, return and the learner's mean action equal run_episode + SimpleLearner."""
    g = _load(golden_dir, "learner.npz")
    K = int(g["loop_max_steps"])
    for c in range(g["dense"].shape[0]):
        env = dx.BatchedManipulationEnv(2, "cuda", max_episode_steps=200, reward_type="dense" if g["dense"][c] else "sparse",
                                        track_episodes=True)
        env.enable_learner(0.01, 0.3, 0.5)
        env.enable_episode_log(64)
        for ep in range(g["steps"].shape[1]):
            n_steps = int(g["steps"][c, ep])
            two = lambda a: np.stack([a, a])
            env.reset_from_draws(two(g["jp0"][c, ep]), two(g["size"][c]), two(g["mass"][c]), two(g["friction"][c]),
                                 two(g["pos"][c, ep]) if ep == 0 else None)
            env._learner_best.fill_(float("-inf"))
            env._ep_log_count.zero_()
            act = np.repeat(g["act_noise"][c, ep, :K][:, None, :], 2, 1)
            upd = np.repeat(g["upd_noise"][c, ep, :K][:, None, :], 2, 1)
            env.rollout(K, policy="learner", respawn=False, loop_max_steps=K, success_is_terminated=False, one_episode=True,
                        learner_act_noise=act, learner_upd_noise=upd)
            log = env.read_episode_log()
            assert len(log) == 2 and all(log["steps"] == n_steps) and all(log["success"] == 0)
            assert all(log["final_contacts"] == g["final_contacts"][c, ep])
            np.testing.assert_allclose(log["episode_reward"], g["reward"][c, ep], rtol=1e-12)
        assert np.array_equal(env.learner_mean[0].cpu().numpy(), g["final_mean"][c])
        assert np.array_equal(env.learner_mean[1].cpu().numpy(), g["final_mean"][c])


def test_fused_simple_learner_matches_oracle_at_scale(dx):
    """2,000 independent learners x 150 steps with auto-reset (reused env objects), pre-drawn normals."""
    from oracle import oracle
    CC = dx.CurriculumConfig
    n, K, seed = 2000, 150, 21
    cfg = CC.medium()
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=40, reward_type="dense", curriculum_config=cfg,
                                    track_episodes=True, seed=seed)
    env.enable_learner(0.01, 0.3, 0.5)
    env.reset(seed=seed)
    ob = oracle.OracleBatch(n, dense=True, max_episode_steps=40)
    grp = oracle.make_group(cfg)
    ob.reset_predrawn(env._obs[:15, :n].t().cpu().numpy(), env._size[:n].cpu().numpy(), env._mass[:n].cpu().numpy(),
                      env._friction[:n].cpu().numpy(), env._obs[30:33, :n].t().cpu().numpy())
    rng = np.random.default_rng(4)
    act = rng.normal(0, 0.3, (K, n, 15)).astype(np.float32)
    upd = rng.normal(0, 0.01, (K, n, 15))
    env.rollout(K, policy="learner", respawn=False, loop_max_steps=40, success_is_terminated=False,
                learner_act_noise=act, learner_upd_noise=upd)
    mean = np.zeros((n, 15), np.float32); best = np.full(n, -np.inf)
    cnt, rs = oracle.rollout_learner(ob, grp, K, seed, mean, best, act, upd, respawn=False, loop_max_steps=40)
    got = env.counters.cpu().numpy()
    assert got[0, 0] > n and np.array_equal(got[:, :16], cnt[:, :16])
    assert np.array_equal(env.learner_mean.cpu().numpy(), mean)
    gb = env.learner_best.cpu().numpy()            # best holds float64 rewards: CUDA and glibc exp differ by <= 1 ulp
    assert np.array_equal(np.isinf(gb), np.isinf(best))
    np.testing.assert_allclose(gb[np.isfinite(gb)], best[np.isfinite(best)], rtol=1e-14)
    assert np.array_equal(env._obs[:, :n].t().cpu().numpy(), ob.observation())
    np.testing.assert_allclose(env.ret_sums.cpu().numpy(), rs, rtol=1e-9)


def test_batched_learner_training_driver(dx):
    out = dx.training.train_learners_batched(64, 6, curriculum_config=dx.CurriculumConfig.hard(), reward_type="dense",
                                             max_episode_steps=50, seed=5)
    assert out["episode_rewards"].shape == (64, 6) and np.isfinite(out["episode_rewards"]).all()
    assert (out["episode_steps"] >= 1).all() and (out["episode_steps"] <= 50).all()
    assert not out["successes"].any()                         # run_episode semantics: success is always False
    assert np.abs(out["mean_action"]).max() <= 0.5 and np.abs(out["mean_action"]).max() > 0.0
    # Philox-drawn learner noise: exploration std 0.3 shows up in the actions' spread
    sched = dx.CurriculumScheduler(dx.CurriculumConfig.easy(), dx.CurriculumConfig.hard(), success_rate_threshold=0.3,
                                   min_episodes_before_progression=20, window_size=15, progression_steps=5)
    out2 = dx.training.train_learners_batched(64, 4, curriculum_config=dx.CurriculumConfig.easy(), max_episode_steps=50, seed=5,
                                              success_is_terminated=True, scheduler=sched)
    assert out2["successes"].any() and sched.current_difficulty_level == 1.0


def test_capture_step_graph_replay_equals_eager(dx):
    CC = dx.CurriculumConfig
    n, steps = 16384, 4
    kw = dict(max_episode_steps=30, reward_type="dense", curriculum_config=CC.easy(), auto_reset=True, respawn=True,
              loop_max_steps=30, track_episodes=True, seed=7)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    a.reset(seed=7); b.reset(seed=7)
    buf = torch.rand(steps, n, 15, device="cuda") * 2 - 1
    replay = b.capture_step(buf, steps=steps)
    for it in range(12):
        buf.copy_(torch.rand(steps, n, 15, device="cuda") * 2 - 1)
        for k in range(steps):
            oa = a.step(buf[k])
        ob = replay()
        assert torch.equal(oa[0], ob[0]) and torch.equal(oa[1], ob[1]) and torch.equal(oa[2], ob[2])
    assert torch.equal(a._obs, b._obs) and torch.equal(a.counters, b.counters) and int(a.counters[:, 0].sum()) > n
    # a sequence of action tensors (two buffers, each used twice per replay) instead of one stacked buffer
    pool = [torch.rand(n, 15, device="cuda") * 2 - 1 for _ in range(2)]
    replay2 = b.capture_step(pool + pool, steps=4)
    for it in range(3):
        for t in pool:
            t.copy_(torch.rand(n, 15, device="cuda") * 2 - 1)
        for k in range(4):
            oa = a.step(pool[k % 2])
        ob = replay2()
        assert torch.equal(oa[0], ob[0]) and torch.equal(oa[1], ob[1])
    assert torch.equal(a._obs, b._obs) and torch.equal(a.counters, b.counters)
    with pytest.raises(ValueError):
        b.capture_step(pool, steps=4)


def test_heldout_noise_sweep_full_size_properties(dx):
    """BASELINE.json configs[2] at full size: 20 held-out objects x 65,536 envs, fused heuristic policy, one group
    per (object, dynamics-noise level) cell.  Size-independent properties: counter bookkeeping closes, the
    two-shard sum equals the single-shard table, larger objects are grasped at least as often."""
    from dexterous_rl_manipulation_b200.config import CurriculumConfig as CC
    rng = np.random.default_rng(123)
    sizes = np.sort(rng.uniform(0.03, 0.12, 20))
    objs = [CC(object_size=float(s), object_mass=float(rng.uniform(0.16, 0.26)), friction_coefficient=float(rng.uniform(0.0, 0.29)))
            for s in sizes]
    N, K, seed = 20 * 65536, 200, 42
    sig = [0.0, 0.05]
    cfgs = [o for o in objs for _ in sig]
    sd = [s for _ in objs for s in sig]
    kw = dict(max_episode_steps=200, reward_type="dense", track_episodes=True, groups=cfgs, group_sigma_dyn=sd, seed=seed)
    full = dx.BatchedManipulationEnv(N, "cuda", **kw)
    full.reset(seed=seed)
    full.rollout(K, policy="heuristic")
    c = full.counters.cpu().numpy()
    assert c[:, 0].min() >= N // 40                      # every env of every cell finished at least one episode
    assert np.array_equal(c[:, 1] + c[:, 4:10].sum(1), c[:, 0])      # success + labelled failures == episodes
    assert np.array_equal(c[:, 4:10].sum(1), c[:, 10:16].sum(1))     # both classifiers label the same episodes
    assert c[:, 16].sum() == 0
    assert (c[:, 2] <= 200 * c[:, 0]).all() and (c[:, 2] >= c[:, 0]).all()
    rate = (c[:, 1] / c[:, 0]).reshape(20, 2)
    assert rate[-1, 0] > rate[0, 0] + 0.3                # the largest object is far easier than the smallest
    assert np.all(np.diff(rate[:, 0]) > -0.02)           # success is (statistically) monotone in object size
    assert np.abs(rate[:, 0] - rate[:, 1]).max() < 0.05  # sigma_dyn = 0.05 barely moves a closing grasp
    del full
    tot = np.zeros_like(c)
    for r in range(2):
        lo, hi = dx.distributed.shard_range(N, r, 2)
        sh = dx.BatchedManipulationEnv(hi - lo, "cuda", env_gid0=lo, **kw)
        sh.reset(seed=seed); sh.rollout(K, policy="heuristic")
        tot += sh.counters.cpu().numpy()
        del sh
    assert np.array_equal(tot, c)


def test_failed_episodes_replay_and_feed_failure_logger(dx, tmp_path):
    """Failure-trajectory capture by deterministic replay: an episode logged by the fused rollout is reproduced
    step by step (same Philox policy stream), and the reference's FailureLogger stores it unchanged."""
    CC = dx.CurriculumConfig

    class _Obj:
        def __init__(self, s, m, f): self.size, self.mass, self.friction = s, m, f

    class _Held:                                   # duck type of evaluation/heldout_objects.py:39-143
        heldout_objects = [_Obj(0.03, 0.2, 0.1), _Obj(0.05, 0.2, 0.2), _Obj(0.09, 0.2, 0.25)]

        def get_eval_config(self, k):
            o = self.heldout_objects[k]
            return CC(object_size=o.size, object_mass=o.mass, friction_coefficient=o.friction)

    held = _Held()
    res = dx.evaluation.evaluate_heldout_set_batched(held, policy="heuristic", num_episodes_per_object=4, seed=42,
                                                     reward_type="dense", max_episode_steps=60, policy_seed=9)
    failed = [e for e in res["all_episodes"] if not e["success"]]
    ok = [e for e in res["all_episodes"] if e["success"]]
    assert failed and ok
    for ep in (failed[0], failed[-1], ok[0]):
        rp = ep["replay"]
        tr = dx.evaluation.replay_episode(held.get_eval_config(rp["object_idx"]), rp["reset_seed"], rp["env_gid"],
                                          rp["philox_episode"], rp["policy"], rp["policy_seed"], rp["reward_type"],
                                          rp["max_episode_steps"])
        assert tr["episode"]["episode_steps"] == ep["episode_steps"] and tr["episode"]["success"] == ep["success"]
        assert tr["episode"]["contact_history"] == ep["contact_history"]
        assert tr["episode"]["episode_reward"] == pytest.approx(ep["episode_reward"], rel=1e-5)
        assert len(tr["states"]) == ep["episode_steps"] + 1 and len(tr["actions"]) == ep["episode_steps"]
        assert all(-0.6001 <= a.min() and a.max() <= -0.3999 for a in tr["actions"])       # heuristic policy range
    from oracle import ref_harness
    if not ref_harness.available():
        return
    R = ref_harness.load()
    flog = importlib_failure_logger(R)(log_dir=str(tmp_path), save_full_trajectories=True)
    n = dx.evaluation.log_failures_batched(res, held, flog)
    assert n == len(failed) == len(flog.logged_episodes)
    for entry, ep in zip(flog.logged_episodes, failed):
        assert entry["failure_mode"] == ep["failure_mode"]              # reference classifier == device label
        assert entry["episode_steps"] == ep["episode_steps"] and len(entry["states"]) == ep["episode_steps"] + 1
        assert entry["metadata"]["seed"] == ep["replay"]["reset_seed"]
    path = flog.save()
    assert os.path.exists(path)


def importlib_failure_logger(R):
    import importlib
    return importlib.import_module("evaluation.failure_logger").FailureLogger


@pytest.mark.parametrize("n,policy,dense,respawn,one_ep", [(7, "random", True, True, False), (100, "heuristic", False, False, False),
                                                           (4096, "random", True, True, False), (5003, "heuristic", True, False, False),
                                                           (1000, "heuristic", True, True, True)])
def test_split_rollout_kernel_equals_thread_rollout_kernel(dx, n, policy, dense, respawn, one_ep):
    """The 5-lanes-per-env small-batch rollout kernel and the one-thread-per-env kernel (itself checked against the
    oracle) must agree on every array, counter, log record and history byte."""
    from dexterous_rl_manipulation_b200 import _lib
    CC = dx.CurriculumConfig
    cfgs = [CC.easy(), CC.hard(), CC(object_size_range=(0.03, 0.09), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))]
    K, max_steps = 90, 30
    envs = {}
    try:
        for impl in ("thread", "split"):
            _lib.set_rollout_impl(impl)
            env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense" if dense else "sparse",
                                            track_episodes=True, groups=cfgs, seed=31, env_gid0=11)
            env.reset(seed=31)
            env.enable_episode_log(n * K)                  # worst case: one episode per env per step
            env.enable_history(K)
            for chunk in (K // 3, K - K // 3):
                env.rollout(chunk, policy=policy, respawn=respawn, one_episode=one_ep)
            envs[impl] = env
    finally:
        _lib.set_rollout_impl("auto")
    a, b = envs["thread"], envs["split"]
    for name in ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
                 "_ep_stats", "_ep_return", "counters", "_hist"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0)
    la, lb = a.read_episode_log(), b.read_episode_log()
    order = lambda r: r[np.lexsort((r["episode"], r["env_gid"]))]
    assert a.episode_log_overflow == 0 and b.episode_log_overflow == 0
    assert len(la) == len(lb) and len(la) >= (n if not one_ep else 1)
    assert np.array_equal(order(la), order(lb))
    if not one_ep:
        assert int(a.counters[:, 0].sum()) > n


def _with_guard_bands(env, guard=4096):
    """Re-home every device array of the env in the middle of a larger buffer whose margins hold a byte
    pattern; returns a checker that fails if any kernel wrote outside its array (compute-sanitizer is not
    available on this pool, so this is the memcheck)."""
    names = ["_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
             "_ep_return", "_ep_stats", "_reward", "_terminated", "_truncated", "_num_contacts", "_finished", "_action_dev"]
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
    env._sync_groups()
    env._obs_view = env._obs[:, :n].t()
    env._info = None
    env._step_out = (env._obs_view, env._reward[:n], env._terminated[:n].view(torch.bool),
                     env._truncated[:n].view(torch.bool), env._make_info())
    env._io.counters, env._io.ret_sums = env.counters.data_ptr(), env.ret_sums.data_ptr()

    def check():
        torch.cuda.synchronize()
        for name, big, g, nb in bands:
            assert bool((big[:g] == 0xA5).all()) and bool((big[g + nb:] == 0xA5).all()), f"out-of-bounds write around {name}"
    return check


@pytest.mark.parametrize("n", [130, 5000, 70_001])
def test_no_out_of_bounds_writes(dx, n):
    from dexterous_rl_manipulation_b200 import _lib
    CC = dx.CurriculumConfig
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=15, reward_type="dense", auto_reset=True, respawn=True,
                                    loop_max_steps=15, track_episodes=True, groups=[CC.easy(), CC.hard()], seed=2)
    check = _with_guard_bands(env)
    env.reset(seed=2)
    check()
    gen = torch.Generator(device="cuda").manual_seed(1)
    try:
        for impl in ("tma", "register"):
            _lib.set_step_impl(impl)
            for t in range(20):
                env.step(torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1)
            check()
        _lib.set_step_impl("auto")
        for chunks in (1, 3, 8):
            for t in range(4):
                env.step_host(torch.rand(n, 15).mul_(2).sub_(1).pin_memory(), chunks=chunks)
            check()
        for impl in ("thread", "split"):
            _lib.set_rollout_impl(impl)
            env.rollout(40, policy="heuristic")
            check()
    finally:
        _lib.set_step_impl("auto"); _lib.set_rollout_impl("auto")
    env.reset()
    check()


@pytest.mark.parametrize("n", [130, 4097, 70_001])
def test_no_out_of_bounds_writes_counts_and_noise_paths(dx, n):
    """Guard bands around every array for the counts-only auto-reset mode (both step kernels, chunked host path) and
    for the in-kernel noise path (noisy_obs output included)."""
    from dexterous_rl_manipulation_b200 import _lib
    CC = dx.CurriculumConfig
    gen = torch.Generator(device="cuda").manual_seed(1)
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=10, reward_type="dense", auto_reset=True, respawn=True,
                                    loop_max_steps=10, track_episodes=False, groups=[CC.easy(), CC.hard()], seed=2)
    check = _with_guard_bands(env)
    env.reset(seed=2)
    try:
        for impl in ("tma", "tma_wide", "register"):
            _set_step_kernel(impl)
            for t in range(25):
                env.step(torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1)
            check()
        for tile_w in ("auto", "wide"):
            _set_step_kernel("auto")
            _lib.set_step_tile(tile_w)
            for chunks in (1, 5):
                env.step_host(torch.rand(n, 15).mul_(2).sub_(1).pin_memory(), chunks=chunks)
                check()
    finally:
        _set_step_kernel("auto")
    assert int(env.counters[:, 0].sum()) > n
    noisy = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=10, reward_type="sparse", auto_reset=True, respawn=True,
                                      loop_max_steps=10, track_episodes=True, curriculum_config=CC.medium(), seed=3,
                                      observation_noise_std=0.1, dynamics_noise_std=0.2)
    noisy.reset(seed=3)                       # allocates the noise buffers
    noisy.step(torch.zeros(n, 15, device="cuda"))
    check2 = _with_guard_bands(noisy)
    nbytes = noisy._noisy_obs.numel() * 4
    big = torch.full((nbytes + 8192,), 0xA5, dtype=torch.uint8, device="cuda")
    noisy._noisy_obs = big[4096:4096 + nbytes].view(torch.float32).view(45, noisy.ld)
    for t in range(25):
        obs = noisy.step(torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1)[0]
    check2()
    torch.cuda.synchronize()
    assert bool((big[:4096] == 0xA5).all()) and bool((big[4096 + nbytes:] == 0xA5).all()), "out-of-bounds write around noisy_obs"
    assert obs.data_ptr() == noisy._noisy_obs.data_ptr() and bool(torch.isfinite(obs).all())


def test_masked_reset_touches_only_masked_envs(dx):
    """options={"mask": ...}: the manual-reset pattern of RL loops that do not use in-kernel auto-reset."""
    CC = dx.CurriculumConfig
    n = 3000
    for rng_mode in ("philox", "numpy"):
        env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=20, reward_type="dense", curriculum_config=CC.easy(),
                                        rng=rng_mode, seed=4, respawn=True)
        env.reset(seed=4 if rng_mode == "philox" else list(range(n)))
        gen = torch.Generator(device="cuda").manual_seed(0)
        for t in range(12):
            obs, rew, te, tr, info = env.step(torch.rand(n, 15, device="cuda", generator=gen) - 0.8)
        done = te | tr
        assert 0 < int(done.sum()) < n
        before = {k: getattr(env, k).clone() for k in ("_obs", "_op64", "_step_count", "_cmask", "_episode", "_thr")}
        obs2, _ = env.reset(options={"mask": done})
        keep = ~done
        for k, v in before.items():
            cur = getattr(env, k)
            if cur.dim() == 2:
                assert torch.equal(cur[:, :n][:, keep], v[:, :n][:, keep]), k
            else:
                assert torch.equal(cur[:n][keep], v[:n][keep]), k
        assert int(env._step_count[:n][done].max()) == 0
        assert torch.equal(env._obs[15:30, :n][:, done], torch.zeros_like(env._obs[15:30, :n][:, done]))   # jv = 0
        assert float(env._obs[0:15, :n][:, done].abs().max()) <= 0.1                                        # fresh joints
        if rng_mode == "philox":
            assert torch.equal(env._episode[:n][done], before["_episode"][:n][done] + 1)


def test_more_unmodified_reference_callers(dx):
    """RobustnessTester (noise wrappers around the env), SeedVarianceAnalyzer and the component-ablation
    training loop of the reference, each run UNMODIFIED once with its own env and once with the drop-in."""
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("reference (source or byte-compiled) not present")
    import importlib
    R = ref_harness.load()
    make = lambda **kw: dx.BatchedManipulationEnv(1, "cuda", **kw)

    def both(module, fn, factories=None):
        out = []
        orig = module.DexterousManipulationEnv
        for factory in (factories or (orig, make)):
            module.DexterousManipulationEnv = factory
            try:
                out.append(fn())
            finally:
                module.DexterousManipulationEnv = orig
        return out

    # 1. RobustnessTester.evaluate_with_noise: CombinedNoiseWrapper(seeded default_rng) wraps the env
    cfg = R.CurriculumConfig(object_size=0.05, object_mass=0.1, friction_coefficient=0.4)

    def robust():
        np.random.seed(11)
        probe = R.DexterousManipulationEnv()
        tester = R.robustness_tests.RobustnessTester(R.policies.HeuristicPolicy(probe.action_space), cfg,
                                                     reward_type="dense", max_episode_steps=40)
        return tester.evaluate_with_noise(0.05, 0.1, num_episodes=4, seed=5)

    ref, got = both(R.robustness_tests, robust)
    assert ref["metrics"]["grasp_success_rate"] == got["metrics"]["grasp_success_rate"]
    assert ref["metrics"]["failure_type_frequency"] == got["metrics"]["failure_type_frequency"]
    for e0, e1 in zip(ref["episodes"], got["episodes"]):
        assert (e0["success"], e0["episode_steps"], e0["contact_history"]) == (e1["success"], e1["episode_steps"], e1["contact_history"])
        assert e1["episode_reward"] == pytest.approx(e0["episode_reward"], rel=1e-5)

    # 2. SeedVarianceAnalyzer.evaluate_multiple_seeds (Evaluator underneath)
    train = R.CurriculumConfig(object_size_range=(0.03, 0.07), object_mass_range=(0.05, 0.15), friction_range=(0.3, 0.7))
    held = R.heldout_objects.HeldOutObjectSet(train_config=train, eval_size_range=(0.03, 0.08), num_heldout_objects=3, seed=2)

    def seeds():
        np.random.seed(3)
        probe = R.DexterousManipulationEnv()
        an = R.seed_variance.SeedVarianceAnalyzer(R.policies.HeuristicPolicy(probe.action_space), held, "dense", 40)
        res = an.evaluate_multiple_seeds([1, 2, 3], num_episodes_per_object=2)
        return an.compute_variance_statistics(res)

    ref, got = both(R.evaluator, seeds)
    assert ref["variance_stats"]["grasp_success_rate"] == got["variance_stats"]["grasp_success_rate"]
    assert ref["variance_stats"]["mean_episode_length"] == got["variance_stats"]["mean_episode_length"]

    # 3. component ablation training loop: run_episode + SimpleLearner + CurriculumScheduler on a reused env
    ca = importlib.import_module("evaluation.component_ablation")

    def train():
        res = ca.train_with_config(ca.AblationConfig(use_curriculum=True, use_dense_reward=True, name="x"),
                                   num_episodes=12, max_episode_steps=40, seed=7)
        return res.episode_rewards, res.episode_steps

    # train_with_config never seeds env.reset(): gymnasium would seed the env's generator from OS entropy.
    # Give both env objects the same generator state so that the two runs are comparable.
    def ref_seeded(**kw):
        e = R.DexterousManipulationEnv(**kw)
        e._np_random = np.random.Generator(np.random.PCG64(np.random.SeedSequence(2024)))
        return e

    def drop_in_seeded(**kw):
        e = make(**kw)
        e._host_rngs(2024)
        return e

    (r0, l0), (r1, l1) = both(ca, train, (ref_seeded, drop_in_seeded))
    assert list(l0) == list(l1)
    np.testing.assert_allclose(r1, r0, rtol=1e-5)


def test_fuzz_extreme_inputs_match_oracle(dx):
    """Adversarial inputs: infinities, NaNs, denormals, huge magnitudes, objects outside the workspace, zero /
    negative / infinite sizes and frictions.  Observations (NaN patterns included), flags and contact counts must
    still equal the oracle bit for bit; rewards where finite."""
    from oracle import oracle
    rng = np.random.default_rng(2718)
    n = 4096
    specials = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1e30, -1e30, 3.4e38, 0.999999, -0.999999,
                         1.0000001, 1e-8], np.float32)
    jp0 = rng.uniform(-1.0, 1.0, (n, 15)).astype(np.float32)
    jp0[::7] = rng.choice(np.array([1.0, -1.0, 0.0, -0.0, 0.99999994, -0.99999994], np.float32), (len(jp0[::7]), 15))
    size = rng.choice([0.0, -0.05, 1e-300, 0.03, 0.05, 0.08, 0.2, 1e300, np.inf, np.nan], n)
    mass = rng.uniform(0.01, 1.0, n)
    fric = rng.choice([0.0, -3.0, 0.3, 0.8, 1e3, 1e6, 1e40, np.inf, np.nan], n)
    pos = rng.uniform(-0.5, 0.5, (n, 3)).astype(np.float32)
    pos[::11] = rng.choice(np.array([0.2, -0.2, 0.3, 0.0, -0.0, 1e30, -1e30, np.inf, np.nan, 0.20000001], np.float32), (len(pos[::11]), 3))
    for dense in (True, False):
        ob = oracle.OracleBatch(n, dense=dense, max_episode_steps=12)
        o0 = ob.reset_predrawn(jp0, size, mass, fric, pos)
        for impl_comps in (True, False):                      # register kernel (comps) and TMA pipeline (no comps)
            env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=12, reward_type="dense" if dense else "sparse",
                                            reward_components=impl_comps)
            g0, _ = env.reset_from_draws(jp0, size, mass, fric, pos)
            assert np.array_equal(g0.cpu().numpy(), o0, equal_nan=True)
            ob2 = oracle.OracleBatch(n, dense=dense, max_episode_steps=12)
            ob2.reset_predrawn(jp0, size, mass, fric, pos)
            arng = np.random.default_rng(5)
            for t in range(25):
                a = arng.uniform(-2.0, 2.0, (n, 15)).astype(np.float32)
                mask = arng.random((n, 15)) < 0.02
                a[mask] = arng.choice(specials, int(mask.sum()))
                oo, orr, _, ote, otr, onc = ob2.step(a)
                obs, rew, te, tr, info = env.step(torch.from_numpy(a).cuda())
                assert np.array_equal(obs.cpu().numpy(), oo, equal_nan=True), (dense, impl_comps, t)
                assert np.array_equal(te.cpu().numpy(), ote) and np.array_equal(tr.cpu().numpy(), otr)
                assert np.array_equal(info["num_contacts"].cpu().numpy(), onc)
                assert np.array_equal(info["object_position"].cpu().numpy(), ob2.env["op"], equal_nan=True)
                r = rew.cpu().numpy()
                fin = np.isfinite(orr)
                assert np.array_equal(np.isnan(r), np.isnan(orr))
                np.testing.assert_allclose(r[fin], orr[fin], rtol=REWARD_RTOL, atol=REWARD_ATOL)


def test_bench_b200_arm_prints_one_contract_line(tmp_path):
    """bench.py (a short run at a reduced env count): exactly one JSON line on stdout carrying every key of the
    bench contract, the roofline and the end-to-end object; --dump-outputs writes the last timed step's arrays."""
    import json
    import subprocess
    import sys
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    dump = tmp_path / "outputs"
    proc = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "20", "--warmup", "3", "--num-envs", "262144",
                           "--e2e-steps", "3", "--no-sweep", "--no-cpu-baseline", "--no-tracking-variant", "--dump-outputs", str(dump)],
                          capture_output=True, text=True, timeout=300)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert key in d, key
    assert d["metric"] == "env_steps_per_sec" and d["n_gpus"] == 1 and d["steps"] == 20 and d["warmup"] == 3
    assert d["gpu_launches"] == 20 and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    r = d["roofline"]
    # `achieved` counts ALGORITHMIC bytes: with consecutive steps walking the batch in opposite directions a fifth of them
    # is served by L2 (and a 262,144-env batch is almost L2-resident), so the fraction may exceed 1 -- but not by much
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and 0.0 < r["frac"] < 2.0
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["sustained_steps"] >= 400 and 0.0 < r["frac_sustained"] < 2.0 and "traffic_steady_state" in r
    assert abs(d["value"] - 262144 * 20 / (d["ms_per_step"] * 20e-3)) / d["value"] < 1e-6
    e = d["e2e"]
    # 32 observation rows + reward + 3 flag bytes + the contact mask cross PCIe every step; the 5 contact rows are expanded on
    # the host, object x, y and their velocities are mirrored by the step kernel when they change
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 262144 * 60 and e["d2h_bytes_per_step"] == 262144 * (32 * 4 + 8)
    assert e["all_rows_d2h_bytes_per_step"] == 262144 * (41 * 4 + 7) and e["copy_ceiling"]["value"] > e["value"] * 0.8
    assert e["value"] < d["value"]                       # host buffers cross PCIe: never faster than the device-resident loop
    # one seeded sample of 131,072 of the 262,144 envs, the same rows in every array, float32 / float64 only, <= 64 MB
    files = {p.stem: np.load(p) for p in dump.iterdir()}
    rows = files["env_index"].astype(np.int64)
    assert len(rows) == 131072 and np.all(np.diff(rows) > 0) and rows[-1] < 262144
    assert files["obs"].shape == (131072, 45) and files["info_object_position"].shape == (131072, 3)
    for name in ("reward", "terminated", "truncated", "info_num_contacts", "info_step_count", "info_finished"):
        assert files[name].shape == (131072,), name
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(p.stat().st_size for p in dump.iterdir()) <= 64 << 20
    assert files["info_step_count"].max() <= 200 and np.isfinite(files["obs"]).all()


def test_bench_dump_outputs_repeat_and_come_from_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs at 4,096 envs (every env written, no sampling): two runs with the same arguments write
    bit-identical arrays, and the step counters are those after the last timed step -- with no pre-roll, 2 warm-up and
    3 timed steps the envs that have not reset yet stand at step 5."""
    import subprocess
    import sys
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    runs = []
    for k in range(2):
        dump = tmp_path / f"run{k}"
        proc = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--num-envs", "4096", "--preroll-steps", "0",
                               "--warmup", "2", "--steps", "3", "--sustained-steps", "10", "--e2e-steps", "3", "--no-strong",
                               "--no-sweep", "--no-cpu-baseline", "--no-tracking-variant", "--dump-outputs", str(dump)],
                              capture_output=True, text=True, timeout=300)
        assert proc.returncode == 0, proc.stderr[-2000:]
        runs.append({p.stem: np.load(p) for p in dump.iterdir()})
    a, b = runs
    assert sorted(a) == sorted(b) and len(a) >= 10
    for name in a:
        assert a[name].dtype == b[name].dtype and np.array_equal(a[name], b[name], equal_nan=True), name
    assert np.array_equal(a["env_index"], np.arange(4096)) and a["obs"].shape == (4096, 45)
    steps = a["info_step_count"]
    assert steps.min() >= 0 and steps.max() == 2 + 3


def test_object_position_attribute_follows_the_reference(dx):
    """envs/manipulation_env.py:156-161: position None -> the next reset samples a spawn; a position -> the next reset
    keeps it; a reused env keeps wherever the last episode left the object."""
    env = dx.BatchedManipulationEnv(1, "cuda", reward_type="dense", max_episode_steps=50)
    assert env.object_position is None
    env.reset(seed=0)
    p0 = env.object_position.copy()
    assert np.allclose(p0, [-0.064868875, 0.072635785, 0.13121918])          # SURVEY.md 8c anchor of reset(seed=0)
    for _ in range(5):
        env.step(np.full(15, -0.5, np.float32))
    p5 = env.object_position.copy()
    assert p5[2] < p0[2]                                                      # the object falls
    _, info = env.reset(seed=1)
    assert np.array_equal(env.object_position, p5) and np.array_equal(info["object_position"], p5.astype(np.float64))
    env.object_position = None
    env.reset(seed=1)
    assert not np.array_equal(env.object_position, p5)                        # fresh spawn
    env.object_position = [0.01, -0.02, 0.07]
    env.reset(seed=2)
    assert np.array_equal(env.object_position, np.array([0.01, -0.02, 0.07], np.float32))
    obs, _ = env.reset(seed=0)
    obs, *_ = env.step(np.full(15, -0.5, np.float32))
    assert np.array_equal(env.joint_positions, obs[0:15]) and np.array_equal(env.joint_velocities, obs[15:30])
    assert np.array_equal(env.object_velocity, obs[37:40]) and np.array_equal(env.contacts, obs[40:45] > 0.5)
    assert env.step_count == 1 and env.joint_positions.dtype == np.float32 and env.contacts.dtype == bool
    batch = dx.BatchedManipulationEnv(64, "cuda")
    assert batch.object_position is None
    batch.reset(seed=3)
    assert tuple(batch.object_position.shape) == (64, 3) and batch.object_position.is_cuda
    assert tuple(batch.joint_positions.shape) == (64, 15) and tuple(batch.contacts.shape) == (64, 5)
    assert tuple(batch.step_count.shape) == (64,) and int(batch.step_count.sum()) == 0


def test_custom_python_reward_object_on_the_single_env_path(dx):
    """SURVEY.md 8f rank 4: a user's own reward class (the compute() duck type of envs/manipulation_env.py:318-325) is
    called on the host for num_envs == 1 with exactly the arguments the reference passes; batched envs refuse it."""
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("reference (source or byte-compiled) not present")
    R = ref_harness.load()

    class ShapedByHeight:
        def __init__(self):
            self.calls, self.resets = 0, 0

        def reset(self):
            self.resets += 1

        def compute(self, joint_positions, finger_tips, object_position, contacts, num_fingers, joints_per_finger):
            self.calls += 1
            d = np.linalg.norm(finger_tips - object_position, axis=1)
            total = float(np.exp(-3.0 * d.mean()) + 0.25 * contacts.sum() - 0.1 * abs(float(object_position[2]))
                          + 0.01 * float(np.abs(joint_positions).sum()))
            return {"total": total, "mean_distance": float(d.mean()), "n": int(num_fingers * joints_per_finger)}

    r_ref, r_new = ShapedByHeight(), ShapedByHeight()
    ref = R.DexterousManipulationEnv(reward_shaping=r_ref, max_episode_steps=40, curriculum_config=R.CurriculumConfig.easy())
    new = dx.BatchedManipulationEnv(1, "cuda", reward_shaping=r_new, max_episode_steps=40, curriculum_config=dx.CurriculumConfig.easy())
    rng = np.random.default_rng(5)
    for seed in (3, 4):
        o0, _ = ref.reset(seed=seed)
        o1, _ = new.reset(seed=seed)
        assert np.array_equal(o0, o1)
        for t in range(40):
            a = rng.uniform(-1.0, 0.3, 15).astype(np.float32)
            s0, s1 = ref.step(a), new.step(a)
            assert np.array_equal(s0[0], s1[0]) and s0[2] == s1[2] and s0[3] == s1[3]
            assert s1[1] == pytest.approx(s0[1], rel=1e-12, abs=1e-12)
            assert s1[4]["reward_components"]["mean_distance"] == pytest.approx(s0[4]["reward_components"]["mean_distance"], rel=1e-12)
            if s0[2] or s0[3]:
                break
    assert r_new.calls == r_ref.calls > 10 and r_new.resets == r_ref.resets == 2
    with pytest.raises(NotImplementedError):
        dx.BatchedManipulationEnv(8, "cuda", reward_shaping=ShapedByHeight())


def test_variance_ties_through_a_real_rollout(dx):
    """Exact variance ties (np.var(contact_counts) == 2.0 in exact arithmetic, where NumPy's pairwise float sum lands
    on either side) forced through a fused rollout with external actions: with the contact threshold raised to 5 and
    per-finger action biases the contact count wanders over 0..5 and a few in a thousand episodes hit the tie.  With the
    history recorded the device decides them with np.var's own arithmetic (var_tie == 2); every label must equal the
    oracle's (full-history np.var emulation, pinned to the reference) and -- when present -- the UNMODIFIED reference
    classifiers'; without the history the same episodes are only flagged (var_tie == 1, DEXSIM_CNT_VAR_TIES) and the
    evaluation front-end's host re-labelling gives the exact labels."""
    from oracle import oracle, ref_harness
    from dexterous_rl_manipulation_b200 import _lib
    from dexterous_rl_manipulation_b200.evaluation import _episode_dict, count_rows
    n, T, thr = 16384, 80, 5
    rng = np.random.default_rng(7)
    bias = rng.uniform(-1, 1, (1, n, 5, 1)).astype(np.float32)
    acts = np.clip(np.repeat(bias, 3, axis=3).reshape(1, n, 15) + rng.normal(0, 0.3, (T, n, 15)).astype(np.float32), -1.5, 1.5)
    acts = torch.from_numpy(acts.astype(np.float32))
    logs = {}
    for with_hist in (True, False):
        env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=T, reward_type="dense", track_episodes=True,
                                        curriculum_config=dx.CurriculumConfig.easy(), seed=7)
        env._params.success_threshold = thr
        env.reset(seed=7)
        env.enable_episode_log(n)
        if with_hist:
            env.enable_history(T)
        env.rollout(T, policy="external", actions=acts, success_is_terminated=False, one_episode=True, loop_max_steps=T,
                    zero_counters=True)
        log = env.read_episode_log()
        assert len(log) == n
        logs[with_hist] = (log, env._hist[:, :n].cpu().numpy() if with_hist else None, env.counters.cpu().numpy().copy())
    log, hist, cnt = logs[True]
    log0, _, cnt0 = logs[False]
    assert np.array_equal(log["env_gid"], log0["env_gid"]) and np.array_equal(log["steps"], log0["steps"])
    ties = np.nonzero(log["var_tie"] == 2)[0]
    assert len(ties) >= 5, len(ties)
    assert np.array_equal(log0["var_tie"] == 1, log["var_tie"] == 2) and not np.any(log["var_tie"] == 1)
    assert int(cnt[:, _lib.CNT_VAR_TIES].sum()) == 0 and int(cnt0[:, _lib.CNT_VAR_TIES].sum()) == len(ties)
    R = ref_harness.load() if ref_harness.available() else None
    changed = 0
    for q in range(n):
        r = log[q]
        i = int(r["env_gid"])
        counts = hist[:int(r["steps"]), i]
        ea, eb, _ = oracle.classify(False, int(r["steps"]), int(r["final_contacts"]), int(r["final_contacts"]), counts,
                                    max_steps=T, threshold=thr)
        ea, eb = (255 if ea < 0 else ea), (255 if eb < 0 else eb)
        assert (int(r["label_metrics"]), int(r["label_taxonomy"])) == (ea, eb), (q, counts.tolist())
        if r["var_tie"] == 2:
            # host re-labelling (evaluation front-ends) of the record the device could only flag
            d = _episode_dict(log0[q], counts, 0.08, 0.05, 0.8, max_steps=T, success_threshold=thr)
            assert d["failure_type"] == dx.LABELS_METRICS[ea] and d["failure_mode"] == dx.LABELS_TAXONOMY[eb]
            la, lb = _lib.classify_counts(False, int(r["steps"]), int(r["final_contacts"]), int(r["final_contacts"]), counts,
                                          max_steps=T, success_threshold=thr)
            assert (la, lb) == (ea, eb)
            changed += (int(log0[q]["label_metrics"]), int(log0[q]["label_taxonomy"])) != (ea, eb)
            if R is not None:
                ep = {"success": False, "episode_steps": int(r["steps"]), "num_contacts": int(r["final_contacts"]),
                      "final_contacts": int(r["final_contacts"]), "contact_history": count_rows(counts)}
                ra = R.metrics.EvaluationMetrics(thr).classify_failure(dict(ep), max_steps=T)
                rb, _conf = R.failure_taxonomy.FailureClassifier(thr).classify(dict(ep), max_steps=T)
                assert ra.value == dx.LABELS_METRICS[ea] and rb.value == dx.LABELS_TAXONOMY[eb]
    # the label counters follow the corrected labels
    for code in range(6):
        assert int(cnt[:, _lib.CNT_LABEL_METRICS + code].sum()) == int((log["label_metrics"] == code).sum())
        assert int(cnt[:, _lib.CNT_LABEL_TAXONOMY + code].sum()) == int((log["label_taxonomy"] == code).sum())


def test_misaligned_aos_action_pointer(dx, step_impl):
    """An [n,15] action slice that starts at an odd env (60-byte stride => base not 16-byte aligned) handed straight to
    the C ABI: the register-resident kernel reads it with scalar loads, results identical to an aligned copy."""
    import ctypes as C
    from dexterous_rl_manipulation_b200 import _lib
    n = 1000
    kw = dict(max_episode_steps=50, reward_type="dense", seed=2)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    a.reset(seed=2); b.reset(seed=2)
    big = torch.rand(n + 3, 15, device="cuda") * 2.4 - 1.2
    for off in (1, 2, 3):
        view = big[off:off + n]
        assert view.data_ptr() % 16 != 0
        io = a._io
        io.action, io.action_layout = view.data_ptr(), 1
        _lib.check(a._lib.dexsim_step(a._state_ref, a._params_ref, a._groups_ptr, a._goe_ptr, a._io_ref, a._stream()), "dexsim_step")
        step_impl("register")
        b.step(view.clone())
        step_impl("auto")
        assert torch.equal(a._obs, b._obs) and torch.equal(a._reward, b._reward) and torch.equal(a._op64, b._op64)


def test_state_dict_resumes_bit_for_bit(dx):
    """state_dict() / load_state_dict(): a resumed run continues exactly like the uninterrupted one -- device state,
    the host PCG64 generators of rng="numpy" resets, Philox seed, rollout step base and the per-env learners."""
    CC = dx.CurriculumConfig
    def make():
        env = dx.BatchedManipulationEnv(64, "cuda", max_episode_steps=15, reward_type="dense", track_episodes=True,
                                        rng="numpy", curriculum_config=CC(object_size_range=(0.03, 0.08)), seed=5)
        env.enable_learner()
        env.reset(seed=5)
        return env
    a = make()
    a.rollout(20, policy="learner", respawn=False)
    a.reset()                                              # draws from the host generators
    sd = a.state_dict()
    b = make()
    b.load_state_dict(sd)
    for env in (a, b):
        env.rollout(20, policy="learner", respawn=False)
        env.reset()                                        # the next host draws must agree as well
        env.rollout(7, policy="random")
    for name in ("_obs", "_op64", "_size", "_mass", "_friction", "_episode", "_step_count", "_learner_mean", "_learner_best",
                 "counters", "_ep_return", "_ep_stats"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert a._rollout_steps == b._rollout_steps and a.seed == b.seed


def test_run_episodes_batched_returns_the_reference_triple(dx):
    """run_episodes_batched == `run_episode` (training/episode_utils.py:13-55) for every env: (success, steps, total
    reward) against the oracle stepped with the same actions, float64 return summed in the reference's order."""
    from oracle import oracle
    n, T = 300, 40
    rng = np.random.default_rng(12)
    jp0, size, mass, fric, pos = _random_draws(rng, n, ragged=False)
    acts = rng.uniform(-1.0, 1.0, (T, n, 15)).astype(np.float32)
    acts[:, :, :] -= 0.4 * (np.arange(n) % 3 == 0)[None, :, None]        # a third of the envs close their fingers faster
    for info_success in (False, True):
        env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=30, reward_type="dense", track_episodes=True,
                                        info_success=info_success)
        env.reset_from_draws(jp0, size, mass, fric, pos)
        success, steps, total = dx.run_episodes_batched(env, policy="external", actions=acts, max_steps=T, reset=False)
        ob = oracle.OracleBatch(n, dense=True, max_episode_steps=30)
        ob.reset_predrawn(jp0, size, mass, fric, pos)
        e_steps, e_total, e_succ, live = np.zeros(n, np.int32), np.zeros(n), np.zeros(n, bool), np.ones(n, bool)
        for t in range(T):
            _, r, _, te, tr, _ = ob.step(acts[t])
            e_total[live] += r[live]
            e_steps[live] += 1
            ended = live & (te | tr)
            e_succ[ended] = te[ended] if info_success else False
            live &= ~ended
        assert np.array_equal(steps, e_steps) and np.array_equal(success, e_succ)
        np.testing.assert_allclose(total, e_total, rtol=1e-12, atol=0)
        assert success.any() == info_success and (steps < T).any()


def test_from_experiment_config(dx, tmp_path):
    """BatchedManipulationEnv.from_experiment_config: the reference's ExperimentConfig object, its dict and its JSON file."""
    import json
    cfg = {"experiment_name": "t", "training": {"max_episode_steps": 37, "reward_type": "sparse", "seed": 9, "num_fingers": 5,
                                                "joints_per_finger": 3}, "curriculum_scheduler": {"initial_config": "easy", "target_config": "hard"}}
    path = tmp_path / "cfg.json"
    path.write_text(json.dumps(cfg))
    for src in (cfg, str(path)):
        env = dx.BatchedManipulationEnv.from_experiment_config(src, num_envs=8, auto_reset=True)
        assert (env.max_episode_steps, env.reward_type, env.seed, env.num_envs, env.auto_reset) == (37, "sparse", 9, 8, True)
        assert env.curriculum_config.object_size == dx.CurriculumConfig.easy().object_size
    from oracle import ref_harness
    if ref_harness.available():
        R = ref_harness.load()
        import importlib
        ec = importlib.import_module("experiments.experiment_config").ExperimentConfig.quick_test()
        env = dx.BatchedManipulationEnv.from_experiment_config(ec, num_envs=4)
        assert env.max_episode_steps == ec.training.max_episode_steps and env.reward_type == ec.training.reward_type


def test_shared_learner_population_update(dx):
    """training.train_shared_learner_batched: after every episode all envs continue from the mean action of the env with
    the highest episode return (lowest global id on ties); sharding the population by global id -- what several GPUs do,
    with distributed.share_best_candidate picking the winner across ranks -- is covered on CPU with gloo; here the
    single-process history must be reproducible and the winner must really be the arg-max of the logged returns."""
    kw = dict(num_envs=512, num_episodes=4, curriculum_config=dx.CurriculumConfig.easy(), reward_type="dense",
              max_episode_steps=25, seed=3)
    a = dx.training.train_shared_learner_batched(**kw)
    b = dx.training.train_shared_learner_batched(**kw)
    assert np.array_equal(a["best_return"], b["best_return"]) and np.array_equal(a["winner_gid"], b["winner_gid"])
    assert np.array_equal(a["mean_action"], b["mean_action"])
    env = a["env"]
    m = env.learner_mean
    assert torch.equal(m, m[0:1].expand_as(m))                       # one shared mean
    log = env.read_episode_log(sort=False)                           # the last episode's records
    k = np.lexsort((log["env_gid"], -log["episode_reward"]))[0]
    assert a["winner_gid"][-1] == log["env_gid"][k] and a["best_return"][-1] == log["episode_reward"][k]
    assert np.all(np.abs(a["mean_action"]) <= 0.5 + 1e-7)


@pytest.mark.parametrize("n,track", [(70_001, "counts"), (150_000, True)])
def test_walk_direction_and_tile_schedule_do_not_change_results(dx, n, track, step_impl):
    """The pipelined step kernel hands tiles out dynamically (DexsimStepIO.sched) and walks the batch in alternating
    directions from step to step (DEXSIM_STEP_REVERSE_TILES, for L2 reuse): neither may change a bit -- against the same
    env stepped with static round-robin tiles in one direction, at sizes with several tiles per CTA."""
    step_impl("tma")
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=12, reward_type="dense", seed=21, groups=[CC.easy(), CC(object_size_range=(0.03, 0.09))],
              auto_reset=True, respawn=True, loop_max_steps=12, track_episodes=track is True)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    b._alternate_tiles = 0
    b._io.sched = None
    a.reset(seed=21); b.reset(seed=21)
    gen = torch.Generator(device="cuda").manual_seed(4)
    for t in range(40):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2.4 - 1.2
        ra, rb = a.step(act), b.step(act)
        for x, y in zip(ra[:4], rb[:4]):
            assert torch.equal(x, y), t
        assert torch.equal(ra[4]["finished"], rb[4]["finished"])
    assert a._io.flags in (0, 1) and b._io.flags == 0
    for name in ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert torch.equal(a.counters, b.counters) and int(a.counters[:, 0].sum()) > n
    assert int(a._sched.abs().sum()) == 0                       # the scheduler words are re-armed after every launch
