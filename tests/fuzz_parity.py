"""Randomised differential test (experiments / soak; the fixed-seed versions of these checks live in
tests/test_gpu_parity.py): CUDA fused rollout vs the oracle's rollout, dexsim_step (either step kernel, with and without
pre-drawn noise) vs the oracle's step on hostile actions, and API-mode auto-reset stepping with the exposed Philox
actions vs the oracle's rollout (the pipelined kernel's dynamic tile scheduler and reset path at multi-tile sizes), and the
host-buffer entry (copy and zero-copy transports) vs the device-tensor API.
Runs random configurations until the time budget is spent and stops at the first mismatch.

    python tests/fuzz_parity.py [seconds] [first_seed]
"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import dexterous_rl_manipulation_b200 as dx  # noqa: E402
from dexterous_rl_manipulation_b200 import _lib  # noqa: E402
from oracle import oracle  # noqa: E402

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 60.0
case = int(sys.argv[2]) if len(sys.argv) > 2 else 0
CC = dx.CurriculumConfig
t_end = time.time() + budget
done = episodes = 0
def fuzz_api_steps(case):
    """dexsim_step (TMA pipeline or register kernel, AoS actions) vs the oracle's step on hostile actions."""
    rng = np.random.default_rng(10_000_000 + case)
    n = int(rng.choice([2, 33, 128, 129, 1000, 4096, 9999, 70001, 131072]))
    dense = bool(rng.integers(2))
    comps = bool(rng.integers(2))
    noisy = bool(rng.integers(3) == 0)                  # pre-drawn dynamics + observation noise (EXTRA instantiations)
    impl = ["auto", "register", "tma"][int(rng.integers(3))] if n >= 128 else "auto"
    tile = ["auto", "narrow", "wide"][int(rng.integers(3))]      # tile width of the pipelined kernel (224-env tiles from 224 envs up)
    max_steps = int(rng.choice([1, 5, 60, 200]))
    T = int(rng.integers(1, 120 if n < 50000 else 10))
    w = tuple(float(x) for x in rng.uniform(0.0, 3.0, 4)) if dense and rng.integers(2) else None
    jp0 = rng.uniform(-1.0, 1.0, (n, 15)).astype(np.float32) if rng.integers(2) else rng.uniform(-0.1, 0.1, (n, 15)).astype(np.float32)
    size, mass, fric = rng.uniform(0.005, 0.4, n), rng.uniform(0.01, 3.0, n), rng.uniform(0.0, 2.0, n)
    pos = np.stack([rng.uniform(-0.3, 0.3, n), rng.uniform(-0.3, 0.3, n), rng.uniform(0.0, 0.4, n)], 1).astype(np.float32)
    kw = {}
    if w is not None:
        class _W:            # duck type of rewards/reward_shaping.py::RewardShaping(weights)
            distance_weight, contact_weight, closure_weight, stability_weight = w
        kw["reward_shaping"] = _W()
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense" if dense else "sparse",
                                    reward_components=comps, **kw)
    ob = oracle.OracleBatch(n, dense=dense, max_episode_steps=max_steps, **({"weights": w} if w is not None else {}))
    g0, _ = env.reset_from_draws(jp0, size, mass, fric, pos)
    desc = dict(case=case, mode="api", n=n, dense=dense, comps=comps, max_steps=max_steps, T=T, weights=w, noisy=noisy, impl=impl, tile=tile)
    assert np.array_equal(g0.cpu().numpy(), ob.reset_predrawn(jp0, size, mass, fric, pos)), ("reset", desc)
    _lib.set_step_impl(impl)
    _lib.set_step_tile(tile)
    for t in range(T):
        kind = int(rng.integers(5))
        a = (rng.uniform(-1.5, 1.5, (n, 15)) if kind < 2 else rng.normal(0, [0.3, 3.0, 1e3][kind - 2], (n, 15))).astype(np.float32)
        if rng.integers(4) == 0:
            idx = rng.integers(0, n, 3), rng.integers(0, 15, 3)
            a[idx] = [np.nan, np.inf, -np.inf]
        nz = {}
        if noisy:
            nz = dict(dyn_noise=rng.normal(0, 0.1, (n, 15)).astype(np.float32), obs_noise=rng.normal(0, 0.05, (n, 45)).astype(np.float32))
        oo, orr, oc, ote, otr, onc = ob.step(a, threads=8, **nz)
        obs, rew, te, tr, info = env.step(torch.from_numpy(a).cuda(), **nz)
        ok = (np.array_equal(obs.cpu().numpy(), oo, equal_nan=True) and np.array_equal(te.cpu().numpy(), ote)
              and np.array_equal(tr.cpu().numpy(), otr) and np.array_equal(info["num_contacts"].cpu().numpy(), onc)
              and np.allclose(rew.cpu().numpy(), orr, rtol=1e-6, atol=1e-7, equal_nan=True)
              and np.array_equal(info["object_position"].cpu().numpy(), ob.env["op"], equal_nan=True))
        if not ok:
            print("MISMATCH", desc, "step", t, flush=True)
            sys.exit(1)
    _lib.set_step_impl("auto")
    _lib.set_step_tile("auto")
    return T * n


def fuzz_api_autoreset(case):
    """API-mode stepping with in-kernel auto-reset and counters (either step kernel, counts-only or full tracking, multi-tile
    sizes that exercise the dynamic tile scheduler) fed with the exposed Philox policy actions, vs the oracle's rollout."""
    import ctypes as C
    rng = np.random.default_rng(20_000_000 + case)
    n = int(rng.choice([129, 1000, 4097, 60001, 131072]))
    dense, respawn = bool(rng.integers(2)), bool(rng.integers(2))
    policy_kind = int(rng.integers(1, 3))
    full = bool(rng.integers(2))
    impl = ["auto", "register", "tma"][int(rng.integers(3))]
    tile = ["auto", "narrow", "wide"][int(rng.integers(3))]
    max_steps = int(rng.choice([2, 7, 40]))
    loop_max = int(rng.choice([2 * max_steps, max_steps, max(1, max_steps // 2)]))
    K = int(rng.integers(3, 70 if n < 50000 else 14))
    seed = int(rng.integers(0, 2 ** 63))
    gid0 = int(rng.choice([0, 5, 2 ** 32 - 30_000]))
    cfgs = [CC.easy(), CC(object_size=0.06, object_size_range=(0.03, 0.09), friction_range=(0.1, 0.9))][:int(rng.integers(1, 3))]
    env = dx.BatchedManipulationEnv(n, "cuda", max_episode_steps=max_steps, reward_type="dense" if dense else "sparse",
                                    auto_reset=True, respawn=respawn, loop_max_steps=loop_max, track_episodes=full, groups=cfgs,
                                    seed=seed, env_gid0=gid0)
    env.reset(seed=seed)
    ob = oracle.OracleBatch(n, dense=dense, max_episode_steps=max_steps)
    groups = np.concatenate([oracle.make_group(c) for c in cfgs])
    G = len(cfgs)
    ob.reset_predrawn(env._obs[:15, :n].t().cpu().numpy(), env._size[:n].cpu().numpy(), env._mass[:n].cpu().numpy(),
                      env._friction[:n].cpu().numpy(), env._obs[30:33, :n].t().cpu().numpy())
    desc = dict(case=case, mode="api_autoreset", n=n, dense=dense, respawn=respawn, policy=policy_kind, full=full, impl=impl, tile=tile,
                max_steps=max_steps, loop_max=loop_max, K=K, gid0=gid0, groups=G)
    _lib.set_step_impl(impl)
    _lib.set_step_tile(tile)
    act = torch.zeros(15, env.ld, device="cuda")
    for _ in range(K):
        _lib.check(env._lib.dexsim_fill_policy_actions(C.byref(env._state), C.byref(env._params), policy_kind, act.data_ptr(),
                                                       env._stream()), "fill")
        env.step(act[:, :n].t().contiguous())
    _lib.set_step_impl("auto")
    _lib.set_step_tile("auto")
    cnt_o, _ = ob.rollout(groups, K, seed, policy_kind=policy_kind, respawn=respawn, env_gid0=gid0, loop_max_steps=loop_max, threads=8)
    cnt = env.counters.cpu().numpy()
    cols = list(range(16)) + [17] if full else [0, 1, 2, 3, 17]
    ok = (np.array_equal(cnt[:, cols], cnt_o[:, cols])
          and np.array_equal(env._obs[:, :n].t().cpu().numpy(), ob.observation(), equal_nan=True)
          and np.array_equal(env._op64[:, :n].t().cpu().numpy(), ob.env["op"])
          and np.array_equal(env._step_count[:n].cpu().numpy(), ob.env["step_count"])
          and np.array_equal(env._episode[:n].cpu().numpy().astype(np.uint32), ob.env["episode"]))
    if not ok:
        print("MISMATCH", desc, flush=True)
        sys.exit(1)
    return K * n, int(cnt[:, 0].sum())


def fuzz_host_transport(case):
    """env.step_host (copy transport and zero-copy transport, random chunk counts, contacts packed or expanded on the
    host, resets and device-side steps in between) against a twin env stepped through the device-tensor API: every
    returned host tensor every step, and the complete device state at the end."""
    rng = np.random.default_rng(30_000_000 + case)
    n = int(rng.choice([100, 128, 129, 1000, 4097, 33000, 70001, 150000]))
    dense, track = bool(rng.integers(2)), bool(rng.integers(2))
    max_steps = int(rng.choice([3, 9, 40]))
    zc = [True, False, "auto"][int(rng.integers(3))]
    K = int(rng.integers(5, 60 if n < 50000 else 16))
    seed = int(rng.integers(0, 2 ** 63))
    cfgs = [CC.easy(), CC(object_size=0.06, object_size_range=(0.03, 0.09), friction_range=(0.1, 0.9))][:int(rng.integers(1, 3))]
    kw = dict(max_episode_steps=max_steps, reward_type="dense" if dense else "sparse", groups=cfgs, seed=seed)
    if track:
        kw.update(auto_reset=True, respawn=bool(rng.integers(2)), loop_max_steps=max_steps, track_episodes=bool(rng.integers(2)))
    a_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    b_env = dx.BatchedManipulationEnv(n, "cuda", **kw)
    a_env.reset(seed=seed); b_env.reset(seed=seed)
    b_env.host_zero_copy = zc
    b_env.host_expand_contacts = bool(rng.integers(4))          # off: all rows downloaded (and no zero-copy)
    tile = ["auto", "narrow", "wide"][int(rng.integers(3))]
    _lib.set_step_tile(tile)
    desc = dict(case=case, mode="host", n=n, dense=dense, track=track, max_steps=max_steps, zc=zc, K=K,
                expand=b_env.host_expand_contacts, tile=tile)
    pins = [torch.empty(n, 15).pin_memory() for _ in range(2)]
    for t in range(K):
        act = torch.from_numpy(rng.uniform(-1.3, 1.3, (n, 15)).astype(np.float32))
        event = int(rng.integers(12))
        if event == 0:                                           # device-side step behind the host buffers
            a_env.step(act.cuda()); b_env.step(act.cuda())
        elif event == 1:
            s2 = int(rng.integers(0, 2 ** 31))
            a_env.reset(seed=s2); b_env.reset(seed=s2)
        chunks = [None, 1, 2, 3, 8][int(rng.integers(5))]
        packed = bool(rng.integers(3) == 0)
        pins[t % 2].copy_(act)
        o1, r1, te1, tr1, i1 = a_env.step(act.cuda())
        o2, r2, te2, tr2, i2 = b_env.step_host(pins[t % 2] if rng.integers(2) else act.numpy(), chunks=chunks, packed_contacts=packed)
        if packed:
            o2 = b_env.expand_contacts_host()
        ok = (torch.equal(o1.cpu(), o2) and torch.equal(r1.cpu(), r2) and torch.equal(te1.cpu(), te2) and torch.equal(tr1.cpu(), tr2)
              and torch.equal(i1["num_contacts"].cpu(), i2["num_contacts"]) and torch.equal(i2["contact_mask"], a_env._cmask[:n].cpu()))
        if not ok:
            print("MISMATCH", desc, "step", t, flush=True)
            sys.exit(1)
    ok = (torch.equal(a_env._obs, b_env._obs) and torch.equal(a_env._op64, b_env._op64) and torch.equal(a_env._episode, b_env._episode)
          and torch.equal(a_env._cmask, b_env._cmask) and torch.equal(a_env._step_count, b_env._step_count)
          and (not track or torch.equal(a_env.counters, b_env.counters)))
    if not ok:
        print("MISMATCH (final state)", desc, flush=True)
        sys.exit(1)
    _lib.set_step_tile("auto")
    return K * n


api_steps = 0
host_steps = 0
while time.time() < t_end:
    if case % 4 == 3:
        host_steps += fuzz_host_transport(case)
        done += 1
        case += 1
        continue
    if case % 3 == 1:
        api_steps += fuzz_api_steps(case)
        done += 1
        case += 1
        continue
    if case % 3 == 2:
        k, e = fuzz_api_autoreset(case)
        api_steps += k
        episodes += e
        done += 1
        case += 1
        continue
    rng = np.random.default_rng(case)
    n = int(rng.choice([1, 31, 32, 129, 777, 4096, 6000, 20011]))
    dense = bool(rng.integers(2))
    respawn = bool(rng.integers(2))
    policy = ["random", "heuristic"][int(rng.integers(2))]
    max_steps = int(rng.choice([1, 2, 7, 40, 200]))
    loop_max = int(rng.choice([2 * max_steps, max_steps, max(1, max_steps // 2)]))   # the oracle's loops always have a bound
    K = int(rng.integers(1, 260))
    gid0 = int(rng.choice([0, 5, 2 ** 31 - 50_000, 2 ** 32 - 30_000]))
    seed = int(rng.integers(0, 2 ** 63))
    n_groups = int(rng.choice([1, 2, 3, 4, 16, 17, 64, 65, 255, 256]))     # both sides of the 16 / 64 staging limits
    cfgs = []
    for _ in range(n_groups):
        kw = dict(object_size=float(rng.uniform(0.01, 0.3)), object_mass=float(rng.uniform(0.01, 2.0)),
                  friction_coefficient=float(rng.uniform(0.0, 1.5)))
        if rng.integers(2):
            lo = float(rng.uniform(0.01, 0.1)); kw["object_size_range"] = (lo, lo + float(rng.uniform(0, 0.2)))
        if rng.integers(2):
            lo = float(rng.uniform(0.01, 0.5)); kw["object_mass_range"] = (lo, lo + float(rng.uniform(0, 1.0)))
        if rng.integers(2):
            lo = float(rng.uniform(0.0, 0.5)); kw["friction_range"] = (lo, lo + float(rng.uniform(0, 1.0)))
        if rng.integers(2):
            kw["spawn_z_range"] = (0.0, float(rng.uniform(0.0, 0.3)))
        cfgs.append(CC(**kw))
    n_env = max(n, 2)
    goe = rng.integers(0, n_groups, n_env).astype(np.uint16) if rng.integers(2) else None   # explicit env -> group map
    env = dx.BatchedManipulationEnv(n_env, "cuda", max_episode_steps=max_steps, reward_type="dense" if dense else "sparse",
                                    track_episodes=True, groups=cfgs, seed=seed, env_gid0=gid0, group_of_env=goe)
    env.reset(seed=seed)
    ob = oracle.OracleBatch(n_env, dense=dense, max_episode_steps=max_steps)
    groups = np.concatenate([oracle.make_group(c) for c in cfgs])
    gidx = [((gid0 + i) & 0xFFFFFFFF) % n_groups if goe is None else int(goe[i]) for i in range(n_env)]
    draws = [oracle.reset_draws(seed, (gid0 + i) & 0xFFFFFFFF, 0, groups[gidx[i]:gidx[i] + 1]) for i in range(n_env)]
    ob.reset_predrawn(np.stack([d[0] for d in draws]), np.array([d[1] for d in draws]), np.array([d[2] for d in draws]),
                      np.array([d[3] for d in draws]), np.stack([d[4] for d in draws]))
    desc = dict(case=case, n=n_env, dense=dense, respawn=respawn, policy=policy, max_steps=max_steps, loop_max=loop_max, K=K,
                gid0=gid0, groups=n_groups, group_map=goe is not None)
    assert np.array_equal(env._obs[:, :n_env].t().cpu().numpy(), ob.observation()), ("reset", desc)
    env.rollout(K, policy=policy, respawn=respawn, loop_max_steps=loop_max)
    cnt_o, rs_o = ob.rollout(groups, K, seed, policy_kind=1 if policy == "random" else 2, respawn=respawn, env_gid0=gid0,
                             group_of_env=goe, loop_max_steps=loop_max)
    cnt = env.counters.cpu().numpy()
    ok = (np.array_equal(cnt[:, :16], cnt_o[:, :16]) and np.array_equal(cnt[:, 17], cnt_o[:, 17])
          and np.array_equal(env._obs[:, :n_env].t().cpu().numpy(), ob.observation(), equal_nan=True)
          and np.array_equal(env._op64[:, :n_env].t().cpu().numpy(), ob.env["op"])
          and np.array_equal(env._step_count[:n_env].cpu().numpy(), ob.env["step_count"])
          and np.array_equal(env._episode[:n_env].cpu().numpy().astype(np.uint32), ob.env["episode"])
          and np.allclose(env._ep_return[:n_env].cpu().numpy(), ob.env["ep_return"], rtol=1e-12, atol=1e-12)
          and np.allclose(env.ret_sums.cpu().numpy(), rs_o, rtol=1e-9))
    if not ok:
        print("MISMATCH", desc, flush=True)
        sys.exit(1)
    done += 1
    episodes += int(cnt[:, 0].sum())
    case += 1
    del env
print(f"fuzz ok: {done} random configurations, {episodes} finished episodes and {api_steps} API + {host_steps} host-transport env-steps compared, next seed {case}")
