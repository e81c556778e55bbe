"""ctypes face of the C restatement (oracle/dexsim_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Builds ``oracle/_build/libdexsim_oracle.so`` on first use when gcc is present (the GPU box
receives the prebuilt file with the snapshot).  See ``dexsim_oracle.h`` for the reference
file:line each function follows and for how parity is pinned.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libdexsim_oracle.so")

NJ, NF, OBS, HIST_MAX, NCOUNTERS = 15, 5, 45, 5248, 18     # HIST_MAX == DEXO_HIST_MAX (dexsim_oracle.h)
LABELS_METRICS = ["slippage", "unstable_contacts", "misaligned_grasp", "timeout", "object_dropped",
                  "insufficient_contacts"]           # evaluation/metrics.py:15-22
LABELS_TAXONOMY = ["slippage", "unstable_grasp", "misalignment", "timeout", "object_dropped",
                   "insufficient_contacts"]          # evaluation/failure_taxonomy.py:14-26

PARAMS_DTYPE = np.dtype([
    ("w_distance", "f8"), ("w_contact", "f8"), ("w_closure", "f8"), ("w_stability", "f8"),
    ("reward_type", "i4"), ("max_episode_steps", "i4"), ("success_threshold", "i4"), ("pad_", "i4"),
], align=True)

GROUP_DTYPE = np.dtype([
    ("size", "f8"), ("mass", "f8"), ("friction", "f8"),
    ("size_lo", "f8"), ("size_hi", "f8"), ("size_ranged", "i4"), ("pad0_", "i4"),
    ("mass_lo", "f8"), ("mass_hi", "f8"), ("mass_ranged", "i4"), ("pad1_", "i4"),
    ("fric_lo", "f8"), ("fric_hi", "f8"), ("fric_ranged", "i4"), ("pad2_", "i4"),
    ("spawn_lo", "f8", (3,)), ("spawn_hi", "f8", (3,)),
    ("sigma_obs", "f4"), ("sigma_dyn", "f4"),
], align=True)

ENV_DTYPE = np.dtype([
    ("jp", "f4", (NJ,)), ("jv", "f4", (NJ,)), ("op", "f8", (3,)), ("ov", "f4", (3,)),
    ("c", "f4", (NF,)), ("prev_c", "f4", (NF,)),
    ("has_prev", "i4"), ("step_count", "i4"), ("op_is_f32", "i4"), ("num_contacts", "i4"),
    ("size", "f8"), ("mass", "f8"), ("friction", "f8"),
    ("ep_return", "f8"), ("ep_steps", "i4"), ("episode", "u4"),
    ("hist", "u1", (HIST_MAX,)),
], align=True)

LEARNER_DTYPE = np.dtype([("mean", "u8"), ("best", "u8"), ("act_noise", "u8"), ("upd_noise", "u8"),
                          ("clip_range", "f4"), ("pad_", "i4")], align=True)

ROLLOUT_DTYPE = np.dtype([
    ("seed", "u8"), ("env_gid0", "i8"), ("k_steps", "i4"), ("policy_kind", "i4"), ("respawn", "i4"),
    ("success_is_terminated", "i4"), ("loop_max_steps", "i4"), ("num_groups", "i4"),
    ("threads", "i4"), ("pad_", "i4"),
], align=True)

_lib = None


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("dexsim_oracle.c", "dexsim_oracle.h")]   # the Makefile's prerequisites
    if force or not os.path.exists(_SO) or any(
            os.path.exists(f) and os.path.getmtime(f) > os.path.getmtime(_SO) for f in srcs):
        subprocess.run(["make", "-C", _HERE, "--no-print-directory"], check=True,
                       stdout=subprocess.DEVNULL)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.dexo_np_var_counts.restype = C.c_double
        _lib.dexo_classify_metrics.restype = C.c_int32
        _lib.dexo_classify_taxonomy.restype = C.c_int32
        _lib.dexo_sizeof_env.restype = C.c_int32
        _lib.dexo_sizeof_group.restype = C.c_int32
        _lib.dexo_rollout.restype = C.c_int32
        _lib.dexo_rollout_learner.restype = C.c_int32
        assert _lib.dexo_sizeof_env() == ENV_DTYPE.itemsize, (_lib.dexo_sizeof_env(), ENV_DTYPE.itemsize)
        assert _lib.dexo_sizeof_group() == GROUP_DTYPE.itemsize, (_lib.dexo_sizeof_group(), GROUP_DTYPE.itemsize)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _check_rollout(rc):
    if rc != 0:
        raise RuntimeError(f"oracle rollout: an episode ran past the {HIST_MAX}-step contact history (code {rc}); "
                           "its labels would need counts the oracle does not keep")


def make_params(dense=True, max_episode_steps=200, weights=(1.0, 0.5, 0.3, 0.2)):
    p = np.zeros(1, PARAMS_DTYPE)
    p["w_distance"], p["w_contact"], p["w_closure"], p["w_stability"] = weights
    p["reward_type"] = 1 if dense else 0
    p["max_episode_steps"] = max_episode_steps
    p["success_threshold"] = 3
    return p


def make_group(cfg=None, sigma_obs=0.0, sigma_dyn=0.0, **kw):
    """Build one group record from a CurriculumConfig-like object or keyword values
    (field meanings: experiments/config.py:17-42)."""
    g = np.zeros(1, GROUP_DTYPE)

    def get(name, default):
        if name in kw:
            return kw[name]
        return getattr(cfg, name, default) if cfg is not None else default

    g["size"] = get("object_size", 0.05)
    g["mass"] = get("object_mass", 0.1)
    g["friction"] = get("friction_coefficient", 0.5)
    for fld, name in (("size", "object_size_range"), ("mass", "object_mass_range"), ("fric", "friction_range")):
        r = get(name, None)
        if r is not None:
            g[fld + "_lo"], g[fld + "_hi"], g[fld + "_ranged"] = r[0], r[1], 1
    sx, sy, sz = get("spawn_x_range", (-0.1, 0.1)), get("spawn_y_range", (-0.1, 0.1)), get("spawn_z_range", (0.05, 0.2))
    g["spawn_lo"] = [sx[0], sy[0], sz[0]]
    g["spawn_hi"] = [sx[1], sy[1], sz[1]]
    g["sigma_obs"], g["sigma_dyn"] = sigma_obs, sigma_dyn
    return g


class OracleBatch:
    """A batch of independent oracle envs (array of ``dexo_env``)."""

    def __init__(self, n, dense=True, max_episode_steps=200, weights=(1.0, 0.5, 0.3, 0.2)):
        self.n = int(n)
        self.env = np.zeros(self.n, ENV_DTYPE)
        self.params = make_params(dense, max_episode_steps, weights)
        self.lib = lib()

    def reset_predrawn(self, jp0, size, mass, friction, pos=None):
        jp0 = np.ascontiguousarray(jp0, np.float32).reshape(self.n, NJ)
        size = np.ascontiguousarray(np.broadcast_to(np.asarray(size, np.float64), (self.n,)))
        mass = np.ascontiguousarray(np.broadcast_to(np.asarray(mass, np.float64), (self.n,)))
        friction = np.ascontiguousarray(np.broadcast_to(np.asarray(friction, np.float64), (self.n,)))
        if pos is not None:
            pos = np.ascontiguousarray(pos, np.float32).reshape(self.n, 3)
        self.lib.dexo_reset_predrawn_batch(_p(self.env), C.c_int64(self.n), _p(jp0), _p(size), _p(mass),
                                           _p(friction), _p(pos))
        return self.observation()

    def observation(self):
        obs = np.empty((self.n, OBS), np.float32)
        for i in range(self.n):
            self.lib.dexo_observation(C.c_void_p(self.env.ctypes.data + i * ENV_DTYPE.itemsize),
                                      C.c_void_p(obs.ctypes.data + i * OBS * 4))
        return obs

    def step(self, action, dyn_noise=None, obs_noise=None, threads=1):
        action = np.ascontiguousarray(action, np.float32).reshape(self.n, NJ)
        if dyn_noise is not None:
            dyn_noise = np.ascontiguousarray(dyn_noise, np.float32).reshape(self.n, NJ)
        if obs_noise is not None:
            obs_noise = np.ascontiguousarray(obs_noise, np.float32).reshape(self.n, OBS)
        obs = np.empty((self.n, OBS), np.float32)
        reward = np.empty(self.n, np.float64)
        comps = np.empty((self.n, 4), np.float64)
        term = np.empty(self.n, np.uint8)
        trunc = np.empty(self.n, np.uint8)
        nc = np.empty(self.n, np.uint8)
        self.lib.dexo_step_batch(_p(self.env), C.c_int64(self.n), _p(self.params), _p(action), _p(dyn_noise),
                                 _p(obs_noise), _p(obs), _p(reward), _p(comps), _p(term), _p(trunc), _p(nc),
                                 C.c_int32(threads))
        return obs, reward, comps, term.astype(bool), trunc.astype(bool), nc

    def rollout(self, groups, k_steps, seed, policy_kind=1, respawn=True, success_is_terminated=True,
                loop_max_steps=None, env_gid0=0, group_of_env=None, actions=None, dyn_noise=None,
                counters=None, ret_sums=None, threads=1):
        groups = np.ascontiguousarray(groups)
        G = groups.shape[0]
        cfg = np.zeros(1, ROLLOUT_DTYPE)
        cfg["seed"], cfg["env_gid0"], cfg["k_steps"], cfg["policy_kind"] = seed, env_gid0, k_steps, policy_kind
        cfg["respawn"], cfg["success_is_terminated"] = int(respawn), int(success_is_terminated)
        cfg["loop_max_steps"] = int(self.params["max_episode_steps"][0]) if loop_max_steps is None else loop_max_steps
        cfg["num_groups"], cfg["threads"] = G, threads
        if counters is None:
            counters = np.zeros((G, NCOUNTERS), np.int64)
        if ret_sums is None:
            ret_sums = np.zeros((G, 2), np.float64)
        if actions is not None:
            actions = np.ascontiguousarray(actions, np.float32).reshape(k_steps, self.n, NJ)
        if dyn_noise is not None:
            dyn_noise = np.ascontiguousarray(dyn_noise, np.float32).reshape(k_steps, self.n, NJ)
        if group_of_env is not None:
            group_of_env = np.ascontiguousarray(group_of_env, np.uint16)
        _check_rollout(self.lib.dexo_rollout(_p(self.env), C.c_int64(self.n), _p(self.params), _p(groups), _p(group_of_env),
                                             _p(cfg), _p(actions), _p(dyn_noise), _p(counters), _p(ret_sums)))
        return counters, ret_sums


def rollout_learner(batch, groups, k_steps, seed, mean, best, act_noise, upd_noise, clip_range=0.5, respawn=False,
                    success_is_terminated=False, loop_max_steps=None, env_gid0=0, counters=None, ret_sums=None):
    """SimpleLearner rollout (policies/simple_learner.py) on an OracleBatch; mean [n,15] float32 and best [n]
    float64 are updated in place; act_noise [k, n, 15] float32 and upd_noise [k, n, 15] float64 are pre-drawn."""
    groups = np.ascontiguousarray(groups)
    G = groups.shape[0]
    cfg = np.zeros(1, ROLLOUT_DTYPE)
    cfg["seed"], cfg["env_gid0"], cfg["k_steps"], cfg["policy_kind"] = seed, env_gid0, k_steps, 3
    cfg["respawn"], cfg["success_is_terminated"] = int(respawn), int(success_is_terminated)
    cfg["loop_max_steps"] = int(batch.params["max_episode_steps"][0]) if loop_max_steps is None else loop_max_steps
    cfg["num_groups"], cfg["threads"] = G, 1
    counters = np.zeros((G, NCOUNTERS), np.int64) if counters is None else counters
    ret_sums = np.zeros((G, 2), np.float64) if ret_sums is None else ret_sums
    assert mean.dtype == np.float32 and mean.flags.c_contiguous and best.dtype == np.float64
    act_noise = np.ascontiguousarray(act_noise, np.float32).reshape(k_steps, batch.n, NJ)
    upd_noise = np.ascontiguousarray(upd_noise, np.float64).reshape(k_steps, batch.n, NJ)
    L = np.zeros(1, LEARNER_DTYPE)
    L["mean"], L["best"] = mean.ctypes.data, best.ctypes.data
    L["act_noise"], L["upd_noise"], L["clip_range"] = act_noise.ctypes.data, upd_noise.ctypes.data, clip_range
    _check_rollout(batch.lib.dexo_rollout_learner(_p(batch.env), C.c_int64(batch.n), _p(batch.params), _p(groups), None,
                                                  _p(cfg), _p(L), _p(counters), _p(ret_sums)))
    return counters, ret_sums


def reset_draws(seed, env_gid, episode, group):
    jp0 = np.empty(NJ, np.float32)
    pos = np.empty(3, np.float32)
    s, m, f = C.c_double(), C.c_double(), C.c_double()
    lib().dexo_reset_draws(C.c_uint64(seed), C.c_uint32(env_gid), C.c_uint32(episode), _p(group), _p(jp0),
                           C.byref(s), C.byref(m), C.byref(f), _p(pos))
    return jp0, s.value, m.value, f.value, pos


def policy_action(seed, env_gid, episode, step, policy_kind):
    a = np.empty(NJ, np.float32)
    lib().dexo_policy_action(C.c_uint64(seed), C.c_uint32(env_gid), C.c_uint32(episode), C.c_uint32(step),
                             C.c_int32(policy_kind), _p(a))
    return a


def philox(ctr, key):
    ctr = np.ascontiguousarray(ctr, np.uint32)
    key = np.ascontiguousarray(key, np.uint32)
    out = np.empty(4, np.uint32)
    lib().dexo_philox4x32_10(_p(ctr), _p(key), _p(out))
    return out


def normal_pair_ref(wa, wb):
    """Float64 Box-Muller (z0, z1) of Philox words wa, wb (arrays of uint32) -- DESIGN.md "RNG"."""
    wa, wb = np.broadcast_arrays(np.asarray(wa, np.uint32), np.asarray(wb, np.uint32))
    shape = wa.shape
    wa, wb = np.ascontiguousarray(wa).ravel(), np.ascontiguousarray(wb).ravel()
    z0, z1 = np.empty(wa.size), np.empty(wa.size)
    lib().dexo_normal_pair_ref(_p(wa), _p(wb), C.c_int64(wa.size), _p(z0), _p(z1))
    return z0.reshape(shape), z1.reshape(shape)


def normal_rows_ref(seed, env_gid, episode, step, stream, rows, sigma):
    """Float64 sigma * N(0,1) [n, rows] that dexsim_fill_normal draws for envs with these (gid, episode, step) words
    (arrays, broadcast; each taken modulo 2^32 like the device's counter words)."""
    gid, ep, st = (np.ascontiguousarray(np.asarray(a, np.int64) & 0xFFFFFFFF, np.uint32)
                   for a in np.broadcast_arrays(env_gid, episode, step))
    out = np.empty((gid.size, rows))
    lib().dexo_normal_rows_ref(C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), _p(gid), _p(ep), _p(st), C.c_int64(gid.size),
                               C.c_uint32(stream), C.c_int32(rows), C.c_double(sigma), _p(out))
    return out


def np_var_counts(counts):
    counts = np.ascontiguousarray(counts, np.uint8)
    return lib().dexo_np_var_counts(_p(counts), C.c_int64(counts.size))


def classify(success, episode_steps, num_contacts, final_contacts, counts, max_steps=200, threshold=3):
    """Returns (metrics.py label code, taxonomy label code, taxonomy confidence); -1 = None."""
    counts = np.ascontiguousarray(counts, np.uint8)
    a = lib().dexo_classify_metrics(int(bool(success)), int(episode_steps), int(num_contacts),
                                    int(final_contacts), _p(counts), C.c_int64(counts.size),
                                    int(max_steps), int(threshold))
    conf = C.c_double()
    b = lib().dexo_classify_taxonomy(int(bool(success)), int(episode_steps), int(num_contacts),
                                     int(final_contacts), _p(counts), C.c_int64(counts.size),
                                     int(max_steps), int(threshold), C.byref(conf))
    return a, b, conf.value
