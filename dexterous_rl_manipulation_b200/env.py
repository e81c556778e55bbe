"""BatchedManipulationEnv -- drop-in for the reference's DexterousManipulationEnv
(envs/manipulation_env.py:14-356) that steps ``num_envs`` independent envs on one B200.

Same constructor keywords, ``reset(seed=None, options=None) -> (obs, info)``,
``step(action) -> (obs, reward, terminated, truncated, info)``, ``action_space``,
``observation_space``, ``max_episode_steps``, mutable ``curriculum_config``, ``metadata``,
``close()``.  With ``num_envs == 1`` it returns NumPy arrays / Python scalars / the reference's
``info`` keys, so ``run_episode`` (training/episode_utils.py:13-55), ``Evaluator``
(evaluation/evaluator.py:71-189), ``RobustnessTester`` (evaluation/robustness_tests.py:240-328)
run against it unmodified.  With ``num_envs > 1`` everything is a CUDA tensor (batch first).

Env state lives in torch tensors (structure-of-arrays, ``[field, ld]``); all arithmetic is in
libdexsim_b200.so (csrc/dexsim_kernels.cu).  There is no CPU path.
"""
import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .config import CurriculumConfig, group_table
from .policy import MlpPolicy

_L = _lib


class Box:
    """The slice of ``gymnasium.spaces.Box`` the reference's policies use
    (policies/heuristic_policy.py:62, policies/random_policy.py:40, policies/simple_learner.py:46,69)."""

    def __init__(self, low, high, shape, dtype=np.float32, seed=None):
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)
        self.low = np.full(self.shape, low, dtype=self.dtype)
        self.high = np.full(self.shape, high, dtype=self.dtype)
        self._rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed)))

    def seed(self, seed=None):
        self._rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed)))
        return [seed]

    def sample(self):
        if not (np.all(np.isfinite(self.low)) and np.all(np.isfinite(self.high))):
            return self._rng.normal(size=self.shape).astype(self.dtype)
        return self._rng.uniform(self.low, self.high, self.shape).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return bool(x.shape == self.shape and np.all(x >= self.low) and np.all(x <= self.high))


def _public_raw_stream(device_index):
    return torch.cuda.current_stream(device_index).cuda_stream


# cudaStream_t of torch's current stream on a device: the private fast getter (a fraction of a microsecond, what
# torch's own extension loaders use) when this torch build has it, else the public API
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None) or _public_raw_stream


def _round_up(x, m):
    return (x + m - 1) // m * m


def _reward_spec(reward_type, reward_shaping):
    """(reward_type code, weights) from the reference's constructor arguments
    (envs/manipulation_env.py:65-74; rewards/reward_shaping.py:20-25)."""
    default = (1.0, 0.5, 0.3, 0.2)
    if reward_shaping is None:
        if reward_type not in ("dense", "sparse"):
            # the reference treats anything that is not "dense" as sparse (:68-74)
            return 0, default
        return (1 if reward_type == "dense" else 0), default
    names = ("distance_weight", "contact_weight", "closure_weight", "stability_weight")
    cls = type(reward_shaping).__name__
    if all(hasattr(reward_shaping, k) for k in names) and (cls == "RewardShaping" or not callable(getattr(reward_shaping, "compute", None))):
        return 1, tuple(float(getattr(reward_shaping, k)) for k in names)
    if cls == "SparseReward":
        return 0, default
    if callable(getattr(reward_shaping, "compute", None)):
        # a user's own reward class (the duck type of envs/manipulation_env.py:318-325): arbitrary Python cannot be fused
        # into the kernel; BatchedManipulationEnv calls it on the host for num_envs == 1 (SURVEY.md 8f rank 4)
        return _CUSTOM_REWARD, default
    raise NotImplementedError(
        "reward_shaping must be RewardShaping(weights), SparseReward or an object with a compute(...) method")


_CUSTOM_REWARD = -1


class BatchedManipulationEnv:
    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 30}   # envs/manipulation_env.py:22

    def __init__(
        self,
        num_envs: int = 1,
        device="cuda",
        num_fingers: int = 5,
        joints_per_finger: int = 3,
        object_position=None,
        max_episode_steps: int = 200,
        render_mode: Optional[str] = None,
        reward_type: str = "sparse",
        reward_shaping=None,
        curriculum_config=None,
        *,
        auto_reset: bool = False,
        respawn: Optional[bool] = None,
        loop_max_steps: int = 0,
        success_is_terminated: bool = True,
        info_success: bool = False,
        track_episodes: Optional[bool] = None,
        reward_components: Optional[bool] = None,
        rng: Optional[str] = None,
        seed: int = 0,
        env_gid0: int = 0,
        groups: Optional[Sequence] = None,
        group_sigma_obs=0.0,
        group_sigma_dyn=0.0,
        group_of_env=None,
        observation_noise_std: float = 0.0,
        dynamics_noise_std: float = 0.0,
        final_observation: bool = False,
        autoreset_mode: str = "same_step",
    ):
        if num_fingers != 5 or joints_per_finger != 3:
            raise _lib.DexsimError(-1006, "BatchedManipulationEnv")
        if num_envs < 1:
            raise ValueError("num_envs must be >= 1")
        self.final_observation = bool(final_observation)
        if self.final_observation and not auto_reset:
            raise ValueError("final_observation=True needs auto_reset=True: without it step() does not reset, and the "
                             "returned observation is already the final one")
        if self.final_observation and int(num_envs) == 1:
            raise NotImplementedError("final_observation is for batched envs; num_envs == 1 mirrors the reference, "
                                      "which has no auto-reset")
        # "same_step": a step that ends an episode resets the env in the same launch and returns the new episode's first
        # observation.  "next_step" (Gymnasium's AutoresetMode.NEXT_STEP, dexsim_step_next_reset): that step returns the
        # terminal observation and info["finished"]; the env's next step ignores its action and resets it instead,
        # returning the first observation, reward 0 and both flags False.
        if autoreset_mode not in ("same_step", "next_step"):
            raise ValueError("autoreset_mode must be 'same_step' or 'next_step'")
        self.autoreset_mode = autoreset_mode
        self._next_step = autoreset_mode == "next_step"
        if self._next_step and not auto_reset:
            raise ValueError("autoreset_mode='next_step' needs auto_reset=True")
        if self._next_step and self.final_observation:
            raise ValueError("autoreset_mode='next_step' already returns the terminal observation from step(); "
                             "final_observation=True is for the same-step reset")
        if self._next_step and int(num_envs) == 1:
            raise NotImplementedError("autoreset_mode='next_step' is for batched envs; num_envs == 1 mirrors the "
                                      "reference, which has no auto-reset")
        self._lib = _lib.lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BatchedManipulationEnv needs a CUDA device; there is no CPU path")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_envs = int(num_envs)
        self.num_fingers, self.joints_per_finger, self.num_joints = 5, 3, 15
        self.max_episode_steps = int(max_episode_steps)
        self.render_mode = render_mode
        self.reward_type = reward_type
        self.reward_shaping = reward_shaping
        self._reward_code, self._weights = _reward_spec(reward_type, reward_shaping)
        self._custom_reward = None
        if self._reward_code == _CUSTOM_REWARD:
            if int(num_envs) != 1:
                raise NotImplementedError(
                    "a custom Python reward_shaping object is called on the host and therefore only supported with "
                    "num_envs == 1; batched envs fuse RewardShaping(weights) / SparseReward into the step kernel")
            self._custom_reward, self._reward_code = reward_shaping, 1
        self.auto_reset = bool(auto_reset)
        self.respawn = respawn
        self.loop_max_steps = int(loop_max_steps)
        self.success_is_terminated = bool(success_is_terminated)
        self.info_success = bool(info_success)
        self.single = self.num_envs == 1
        self.track_episodes = self.auto_reset if track_episodes is None else bool(track_episodes)
        self.reward_components = self.single if reward_components is None else bool(reward_components)
        self.rng_mode = rng or ("numpy" if self.single else "philox")
        if self.rng_mode not in ("numpy", "philox"):
            raise ValueError("rng must be 'numpy' or 'philox'")
        self.seed = int(seed)
        self.env_gid0 = int(env_gid0)
        self.observation_noise_std = float(observation_noise_std)
        self.dynamics_noise_std = float(dynamics_noise_std)

        self.action_space = Box(-1.0, 1.0, (15,), np.float32)                 # :85-90
        self.observation_space = Box(-np.inf, np.inf, (45,), np.float32)      # :96-106
        self._curriculum_config = curriculum_config if curriculum_config is not None else CurriculumConfig()
        self._group_cfgs = list(groups) if groups is not None else None
        self._group_sigma = (group_sigma_obs, group_sigma_dyn)
        self._groups_dirty = True
        self._object_position_arg = None if object_position is None else np.asarray(object_position, np.float32)
        self._spawned = False          # reference: self.object_position is None until the first reset (:156)
        self._np_rngs = None

        n, ld = self.num_envs, _round_up(self.num_envs, 32)
        self.ld = ld
        dev = self.device
        z = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=dev)
        self._obs = z(45, ld, dtype=torch.float32)
        self._obs[_L.ROW_QUAT].fill_(1.0)
        self._op64 = z(3, ld, dtype=torch.float64)
        self._thr = z(ld, dtype=torch.float64)
        self._damp = z(ld, dtype=torch.float32)
        self._step_count = z(ld, dtype=torch.int32)
        self._cmask = z(ld, dtype=torch.uint8)
        self._size = z(ld, dtype=torch.float64)
        self._mass = z(ld, dtype=torch.float64)
        self._friction = z(ld, dtype=torch.float64)
        self._episode = z(ld, dtype=torch.int32)
        self._ep_return = z(ld, dtype=torch.float64) if self.track_episodes else None
        self._ep_stats = z(2, ld, dtype=torch.int32) if self.track_episodes else None
        self._reward = z(ld, dtype=torch.float32)
        self._reward64 = z(ld, dtype=torch.float64) if self.single else None   # exact Python-float reward for drop-in use
        self._comps = z(4, ld, dtype=torch.float32) if self.reward_components else None
        self._terminated = z(ld, dtype=torch.uint8)
        self._truncated = z(ld, dtype=torch.uint8)
        self._num_contacts = z(ld, dtype=torch.uint8)
        self._finished = z(ld, dtype=torch.uint8) if self.auto_reset else None
        # terminal observation of every episode a step ends (dexsim_step_final), read where info["finished"]
        self._final_obs = z(45, ld, dtype=torch.float32) if self.final_observation else None
        self._action_dev = z(n, 15, dtype=torch.float32)
        self._sched = z(_L.SCHED_WORDS, dtype=torch.int32)      # dynamic tile scheduler words of the pipelined step kernel
        self._noisy_obs = None
        self._obs_noise = None
        self._dyn_noise = None
        self._goe = self._goe_ptr = None
        if group_of_env is not None:
            self._set_group_of_env(group_of_env)
        self._groups_dev = None
        self.counters = None
        self.ret_sums = None
        self._state = _lib.DexsimState()
        self._params = _lib.DexsimParams()
        self._io = _lib.DexsimStepIO()
        self._refresh_structs()
        self._sync_groups()
        # persistent output views (batch first) and ctypes references for the allocation-free hot path
        self._obs_view = self._obs[:, :n].t()
        self._info = None
        self._did_reset = False
        self._rollout_steps = 0
        self._n15 = n * 15
        # Philox noise of noisy envs is drawn inside the step kernel; False = separate dexsim_fill_normal launches
        # (same numbers, kept for cross-checking)
        self.fused_noise = True
        self._io_has_noise = False
        self._alternate_tiles = _L.STEP_REVERSE_TILES    # 0 switches the alternation off (experiments)
        self.host_expand_contacts = True                 # step_host(): contact columns travel packed, expanded on the host
        self.host_static_rows = True                     # step_host(): reset-only rows mirrored by the kernel, not downloaded
        # step_host(): the step kernel writes its results straight into the pinned host buffers (no download copies).
        # "auto": batches up to 160K envs, where it beats the chunked copy pipeline (no pipeline fill; B200, PCIe 5:
        # 32K envs 0.174 vs 0.213 ms/step, 128K 0.515 vs 0.530, 256K 1.02 vs 0.96, 1M 3.67 vs 3.20); True / False force it
        self.host_zero_copy = "auto"
        self._h_primed_slot = None                       # result slot whose pinned observation is current (see step_host)
        self._state_ref, self._params_ref, self._io_ref = C.byref(self._state), C.byref(self._params), C.byref(self._io)
        # the step entry of this env, chosen once; dexsim_step_final takes the final-observation buffer before the stream
        self._step_entry_name = ("dexsim_step_final" if self.final_observation else
                                 "dexsim_step_next_reset" if self._next_step else "dexsim_step")
        self._step_entry = getattr(self._lib, self._step_entry_name)
        self._step_final_obs = self._ptr(self._final_obs)
        # filled on first use: pinned host buffers (a batched env pins none it does not use), the rollout's optional outputs
        self._action_pin = self._pack_host = self._ep_log = self._ep_log_count = self._hist = self._learner_mean = None
        self._traj, self._traj_rows, self._traj_has_action = None, 0, False
        self._h_slots, self._host_keepalive = {}, {}
        self._step_out = None
        if not self.single:
            self._step_out = (self._obs_view, self._reward[:n], self._terminated[:n].view(torch.bool),
                              self._truncated[:n].view(torch.bool), self._make_info())

    @classmethod
    def from_experiment_config(cls, cfg, num_envs: int = 1, device="cuda", curriculum_config=None, **kw):
        """Build the env from the reference's ``ExperimentConfig`` (experiments/experiment_config.py:236-300) or from the
        dict / JSON it serialises to (``config_default.json`` ...): ``training.max_episode_steps``, ``training.reward_type``,
        ``training.num_fingers`` / ``joints_per_finger`` and ``training.seed`` are taken from it exactly as the reference's
        drivers pass them to ``DexterousManipulationEnv`` (evaluation/component_ablation.py:132-140); the curriculum starts
        at ``curriculum_config`` or, when the config carries a ``curriculum_scheduler`` section, at that scheduler's
        initial preset.  Other keywords go to the constructor (``auto_reset=...``, ``track_episodes=...``)."""
        if isinstance(cfg, str):
            import json
            with open(cfg) as fh:
                cfg = json.load(fh)
        get = (lambda o, k, d=None: o.get(k, d)) if isinstance(cfg, dict) else (lambda o, k, d=None: getattr(o, k, d))
        tr = get(cfg, "training", {}) or {}
        tget = (lambda k, d: tr.get(k, d)) if isinstance(tr, dict) else (lambda k, d: getattr(tr, k, d))
        if curriculum_config is None:
            sch = get(cfg, "curriculum_scheduler", None)
            name = None if sch is None else (sch.get("initial_config") if isinstance(sch, dict) else getattr(sch, "initial_config", None))
            if isinstance(name, str) and hasattr(CurriculumConfig, name):
                curriculum_config = getattr(CurriculumConfig, name)()
        kw.setdefault("seed", int(tget("seed", 0)))
        return cls(num_envs, device, num_fingers=int(tget("num_fingers", 5)), joints_per_finger=int(tget("joints_per_finger", 3)),
                   max_episode_steps=int(tget("max_episode_steps", 200)), reward_type=tget("reward_type", "dense"),
                   curriculum_config=curriculum_config, **kw)

    # ------------------------------------------------------------------ plumbing
    @staticmethod
    def _ptr(t):
        return None if t is None else t.data_ptr()

    def _refresh_structs(self):
        s, p, io = self._state, self._params, self._io
        s.n, s.ld = self.num_envs, self.ld
        s.obs, s.op64, s.thr, s.damp = self._ptr(self._obs), self._ptr(self._op64), self._ptr(self._thr), self._ptr(self._damp)
        s.step_count, s.cmask = self._ptr(self._step_count), self._ptr(self._cmask)
        s.size, s.mass, s.friction = self._ptr(self._size), self._ptr(self._mass), self._ptr(self._friction)
        s.episode, s.ep_return, s.ep_stats = self._ptr(self._episode), self._ptr(self._ep_return), self._ptr(self._ep_stats)
        p.w_distance, p.w_contact, p.w_closure, p.w_stability = self._weights
        p.reward_type = self._reward_code
        p.max_episode_steps = self.max_episode_steps
        p.success_threshold = 3
        p.auto_reset = int(self.auto_reset)
        p.respawn = int(True if self.respawn is None else self.respawn)
        p.success_is_terminated = int(self.success_is_terminated)
        p.loop_max_steps = self.loop_max_steps
        p.seed = self.seed & 0xFFFFFFFFFFFFFFFF
        p.env_gid0 = self.env_gid0
        io.reward, io.reward_comps = self._ptr(self._reward), self._ptr(self._comps)
        io.terminated, io.truncated = self._ptr(self._terminated), self._ptr(self._truncated)
        io.num_contacts, io.finished = self._ptr(self._num_contacts), self._ptr(self._finished)
        io.counters, io.ret_sums = self._ptr(self.counters), self._ptr(self.ret_sums)
        io.reward64 = self._ptr(self._reward64)
        io.sched = self._ptr(self._sched)
        self._io_single = None

    @property
    def curriculum_config(self):
        return self._curriculum_config

    @curriculum_config.setter
    def curriculum_config(self, cfg):
        # callers assign this between episodes (evaluation/component_ablation.py:163-166);
        # effective at the next reset, including in-kernel auto-resets of later launches
        self._curriculum_config = cfg
        if self._group_cfgs is None:
            self._groups_dirty = True

    def set_groups(self, configs, sigma_obs=0.0, sigma_dyn=0.0, group_of_env=None):
        """Several curriculum / object / noise cells in one batch; env -> group is
        ``group_of_env`` or ``global env id % len(configs)``."""
        self._group_cfgs = list(configs)
        self._group_sigma = (sigma_obs, sigma_dyn)
        if group_of_env is not None:
            self._set_group_of_env(group_of_env)
        self._groups_dirty = True

    def _set_group_of_env(self, group_of_env):
        self._goe = torch.zeros(self.ld, dtype=torch.int16, device=self.device)
        self._goe[:self.num_envs] = torch.as_tensor(group_of_env).to(torch.int16).to(self.device)
        self._goe_ptr = self._goe.data_ptr()

    @property
    def num_groups(self):
        return len(self._group_cfgs) if self._group_cfgs is not None else 1

    def _sync_groups(self):
        if not self._groups_dirty:
            return
        cfgs = self._group_cfgs if self._group_cfgs is not None else [self._curriculum_config]
        so, sd = self._group_sigma
        if self._group_cfgs is None:
            so, sd = self.observation_noise_std, self.dynamics_noise_std
        table = group_table(cfgs, so, sd)
        # noise cells of a multi-group batch (group_sigma_*): step() draws them in-kernel with each env's group value
        self._group_noise = (self._group_cfgs is not None and bool(np.any(np.asarray(so, np.float64) > 0.0)),
                             self._group_cfgs is not None and bool(np.any(np.asarray(sd, np.float64) > 0.0)))
        self._noisy_env = (self.observation_noise_std > 0.0 or self.dynamics_noise_std > 0.0 or any(self._group_noise))
        raw = torch.frombuffer(bytearray(bytes(table)), dtype=torch.uint8)
        if self._groups_dev is None or self._groups_dev.numel() != raw.numel():
            self._groups_dev = torch.empty(raw.numel(), dtype=torch.uint8, device=self.device)
        self._groups_dev.copy_(raw, non_blocking=False)
        G = len(cfgs)
        if self.counters is None or self.counters.shape[0] != G:
            self.counters = torch.zeros(G, _L.NCOUNTERS, dtype=torch.int64, device=self.device)
            self.ret_sums = torch.zeros(G, 2, dtype=torch.float64, device=self.device)
        self._params.num_groups = G
        self._io.counters, self._io.ret_sums = self._ptr(self.counters), self._ptr(self.ret_sums)
        self._io_single = None                      # persistent copy used by the single-env fast path: rebuild lazily
        self._groups_ptr = self._groups_dev.data_ptr()
        self._groups_dirty = False

    def _stream(self):
        return C.c_void_p(_raw_stream(self.device.index))

    # ------------------------------------------------------------------ reset
    def _host_rngs(self, seed):
        n = self.num_envs
        if self._np_rngs is None:
            self._np_rngs = [None] * n
        if seed is not None:
            seeds = [int(seed) + i for i in range(n)] if np.isscalar(seed) else [int(s) for s in seed]
            if len(seeds) != n:
                raise ValueError("need one seed per env")
            for i, s in enumerate(seeds):
                self._np_rngs[i] = np.random.Generator(np.random.PCG64(np.random.SeedSequence(s)))
        for i in range(n):
            if self._np_rngs[i] is None:          # gymnasium seeds lazily from entropy
                self._np_rngs[i] = np.random.Generator(np.random.PCG64(np.random.SeedSequence(None)))
        return self._np_rngs

    def _config_of_env(self, i):
        if self._group_cfgs is None:
            return self._curriculum_config
        if self._goe is not None:
            return self._group_cfgs[int(self._goe[i])]
        return self._group_cfgs[(self.env_gid0 + i) % len(self._group_cfgs)]

    @property
    def object_position(self):
        """The reference's attribute (envs/manipulation_env.py:57,156-161): None until the first reset, then the
        current position -- float32[3] for one env, a float64 CUDA view [num_envs, 3] for a batch.  Assigning None
        makes the next reset sample a fresh spawn; assigning a position makes the next reset start from it."""
        if not self._spawned:
            return None if self._object_position_arg is None else self._object_position_arg
        p = self._op64[:, :self.num_envs].t()
        return p[0].cpu().numpy().astype(np.float32) if self.single else p

    @object_position.setter
    def object_position(self, value):
        self._object_position_arg = None if value is None else np.asarray(value, np.float32)
        self._spawned = False

    # read-only views of the reference env's state attributes (envs/manipulation_env.py:54-62): NumPy copies for
    # one env, CUDA views [num_envs, ...] of the SoA state for a batch
    def _rows(self, lo, hi, dtype=np.float32):
        v = self._obs[lo:hi, :self.num_envs].t()
        return v[0].cpu().numpy().astype(dtype) if self.single else v

    @property
    def joint_positions(self):
        return self._rows(_L.ROW_JP, _L.ROW_JP + 15)

    @property
    def joint_velocities(self):
        return self._rows(_L.ROW_JV, _L.ROW_JV + 15)

    @property
    def object_velocity(self):
        return self._rows(_L.ROW_OV, _L.ROW_OV + 3)

    @property
    def contacts(self):
        c = self._rows(_L.ROW_CONTACT, _L.ROW_CONTACT + 5)
        return c.astype(bool) if self.single else c.to(torch.bool)

    @property
    def step_count(self):
        return int(self._step_count[0]) if self.single else self._step_count[:self.num_envs]

    def _respawn_now(self):
        if self.respawn is not None:
            return bool(self.respawn)
        return not self._spawned and self._object_position_arg is None

    def reset(self, seed=None, options=None):
        """envs/manipulation_env.py:124-182.  ``options={"mask": BoolTensor[num_envs]}`` resets a subset."""
        self._h_primed_slot = None
        with torch.cuda.device(self.device):
            self._sync_groups()
            mask = None
            if options and options.get("mask") is not None:
                m = torch.as_tensor(options["mask"]).to(self.device).to(torch.uint8)
                mask = torch.zeros(self.ld, dtype=torch.uint8, device=self.device)
                mask[:self.num_envs] = m
            n = self.num_envs
            respawn = self._respawn_now()
            if self.rng_mode == "numpy":
                rngs = self._host_rngs(seed)
                jp0 = np.zeros((n, 15), np.float32)
                size = np.zeros(n); mass = np.zeros(n); fric = np.zeros(n)
                pos = np.zeros((n, 3), np.float32) if (respawn or (not self._spawned and self._object_position_arg is not None)) else None
                mask_host = None if mask is None else mask.cpu().numpy()
                for i in range(n):
                    if mask_host is not None and not mask_host[i]:
                        continue
                    r, cfg = rngs[i], self._config_of_env(i)
                    jp0[i] = r.uniform(low=-0.1, high=0.1, size=(15,)).astype(np.float32)          # :143-145
                    size[i] = cfg.get_object_size(r); mass[i] = cfg.get_object_mass(r)            # :151-153
                    fric[i] = cfg.get_friction_coefficient(r)
                    if respawn:
                        pos[i] = np.array(cfg.get_spawn_position(r), dtype=np.float32)            # :156-159
                    elif pos is not None:
                        a = self._object_position_arg
                        pos[i] = a if a.ndim == 1 else a[i]                                        # :160-161
                self._reset_predrawn(jp0, size, mass, fric, pos, mask)
            else:
                if seed is not None:
                    self.seed = int(seed)
                    self._params.seed = self.seed & 0xFFFFFFFFFFFFFFFF
                    if mask is None:
                        self._episode.zero_()
                elif self._did_reset:
                    if mask is None:
                        self._episode.add_(1)
                    else:
                        self._episode.add_(mask.to(torch.int32))
                if not respawn and not self._spawned and self._object_position_arg is not None:
                    a = torch.as_tensor(self._object_position_arg, device=self.device)
                    self._op64[:, :n] = (a.reshape(3, 1) if a.ndim == 1 else a.t()).to(torch.float64)
                _lib.check(self._lib.dexsim_reset_philox(
                    C.byref(self._state), C.byref(self._params), self._ptr(self._groups_dev), self._ptr(self._goe),
                    self._ptr(mask), int(respawn), self._stream()), "dexsim_reset_philox")
            self._spawned = True
            self._did_reset = True
            if self._custom_reward is not None and callable(getattr(self._custom_reward, "reset", None)):
                self._custom_reward.reset()                  # envs/manipulation_env.py:177
            if mask is None:
                self._rollout_steps = 0
                if self._ep_log_count is not None:
                    self._ep_log_count.zero_()
                if self.rng_mode == "numpy":
                    self._episode.zero_()
            return self._reset_outputs()

    def reset_from_draws(self, jp0, size, mass, friction, pos=None, mask=None):
        """Reset with caller-supplied draws (batch first): jp0 [n,15] float32, size/mass/friction [n]
        float64, pos [n,3] float32 or None = keep each env's current position cast to float32
        (envs/manipulation_env.py:160-161).  This is the parity entry: identical initial states."""
        n, ld, dev = self.num_envs, self.ld, self.device
        self._h_primed_slot = None
        with torch.cuda.device(dev):
            self._sync_groups()
            mask_d = None
            if mask is not None:
                mask_d = torch.zeros(ld, dtype=torch.uint8, device=dev)
                mask_d[:n] = torch.as_tensor(np.asarray(mask)).to(torch.uint8).to(dev)
            self._reset_predrawn(jp0, size, mass, friction, pos, mask_d)
            self._spawned = True
            self._did_reset = True
            return self._reset_outputs()

    def _reset_predrawn(self, jp0, size, mass, friction, pos, mask):
        """dexsim_reset_predrawn of the envs in ``mask`` (device uint8 [ld], None = all) from host draws, batch first as
        reset_from_draws() takes them; returns once the kernel has read them."""
        per_env = lambda x: self._soa(np.broadcast_to(np.asarray(x, np.float64), (self.num_envs,)).copy(), 1,
                                       torch.float64)
        jp0_d, size_d, mass_d, fric_d = self._soa(jp0, 15), per_env(size), per_env(mass), per_env(friction)
        pos_d = None if pos is None else self._soa(pos, 3)
        _lib.check(self._lib.dexsim_reset_predrawn(
            self._state_ref, self._params_ref, self._ptr(mask), self._ptr(jp0_d), self._ptr(size_d),
            self._ptr(mass_d), self._ptr(fric_d), self._ptr(pos_d), self._stream()), "dexsim_reset_predrawn")
        torch.cuda.current_stream(self.device).synchronize()

    # ------------------------------------------------------------------ step
    def _ingest_action(self, action):
        n = self.num_envs
        if isinstance(action, torch.Tensor) and action.is_cuda:
            a = action
            if a.dtype != torch.float32:
                a = a.to(torch.float32)
            a = a.reshape(n, 15)
            if not a.is_contiguous():
                a = a.contiguous()
            if a.data_ptr() % 16:
                self._action_dev.copy_(a)
                a = self._action_dev
            return a
        a = np.asarray(action.detach().cpu() if isinstance(action, torch.Tensor) else action)
        if a.dtype != np.float32:
            # the reference silently promotes float64 actions and corrupts its own dtypes
            # (SURVEY.md 8a-1); the batched env takes float32 only
            a = a.astype(np.float32)
        if self.single:
            # 60 bytes: the kernel reads them from mapped page-locked host memory, no copy call.  Safe to
            # overwrite: every single-env step ends by waiting for its result, so no kernel is still reading.
            self._pin_action()[:15] = a.reshape(15)
            return self._action_pin
        self._action_dev.copy_(torch.from_numpy(np.ascontiguousarray(a.reshape(n, 15))), non_blocking=False)
        return self._action_dev

    def _pin_action(self):
        """NumPy view of the single env's page-locked action buffer, allocated on first use."""
        if self._action_pin is None:
            self._action_pin = torch.zeros(16, dtype=torch.float32).pin_memory()
            self._action_pin_np = self._action_pin.numpy()
        return self._action_pin_np

    def _noise_buffers(self):
        if self._noisy_obs is None:
            self._noisy_obs = torch.zeros(45, self.ld, dtype=torch.float32, device=self.device)
            self._obs_noise = torch.zeros(45, self.ld, dtype=torch.float32, device=self.device)
            self._dyn_noise = torch.zeros(15, self.ld, dtype=torch.float32, device=self.device)

    def _soa(self, x, rows, dtype=torch.float32, steps=None):
        """Batch-first [n, rows] (or [rows] for a single env; [steps, n, rows] with ``steps``) -> SoA [rows, ld]
        ([steps, rows, ld]) device tensor, zero past n."""
        lead = () if steps is None else (steps,)
        t = torch.as_tensor(x, dtype=dtype, device=self.device).reshape(*lead, self.num_envs, rows)
        out = torch.zeros(*lead, rows, self.ld, dtype=dtype, device=self.device)
        out[..., :self.num_envs] = t.transpose(-1, -2)
        return out

    @staticmethod
    def _clear_noise(io):
        io.dyn_noise = io.obs_noise = io.noisy_obs = None
        io.sigma_dyn = io.sigma_obs = 0.0

    def step(self, action, dyn_noise=None, obs_noise=None):
        """envs/manipulation_env.py:184-252 for every env.  ``dyn_noise`` [n,15] / ``obs_noise`` [n,45]
        are optional PRE-DRAWN float32 noise tensors (evaluation/robustness_tests.py:177-207); without
        them, ``dynamics_noise_std`` / ``observation_noise_std`` > 0 draw Philox normals on the device."""
        if not self._did_reset:
            raise RuntimeError("call reset() before step()")
        if self._groups_dirty:
            self._sync_groups()
        self._h_primed_slot = None
        plain = (dyn_noise is None and obs_noise is None and not self._noisy_env and not self.single
                 and isinstance(action, torch.Tensor) and action.is_cuda and action.dtype is torch.float32
                 and action.is_contiguous() and action.numel() == self._n15 and not (action.data_ptr() & 15))
        if plain and torch.cuda.current_device() == self.device.index:
            # hot path: one ctypes call, persistent output views, no allocation
            io = self._io
            io.action, io.action_layout = action.data_ptr(), 1
            io.flags ^= self._alternate_tiles          # walk the batch back and forth: a step starts on what is still in L2
            if self._io_has_noise:
                self._clear_noise(io)
                self._io_has_noise = False
            # two spelled-out calls: a starred one costs ~0.1 us, which shows at the host-bound batch sizes
            fo = self._step_final_obs
            if fo is None:
                rc = self._step_entry(self._state_ref, self._params_ref, self._groups_ptr, self._goe_ptr, self._io_ref,
                                      _raw_stream(self.device.index))
            else:
                rc = self._step_entry(self._state_ref, self._params_ref, self._groups_ptr, self._goe_ptr, self._io_ref,
                                      fo, _raw_stream(self.device.index))
            if rc:
                raise _lib.DexsimError(rc, self._step_entry_name)
            return self._step_out
        if (self.single and dyn_noise is None and obs_noise is None and not self._noisy_env
                and not (isinstance(action, torch.Tensor) and action.is_cuda)
                and torch.cuda.current_device() == self.device.index):
            return self._step_single_fast(action)
        with torch.cuda.device(self.device):
            return self._step_general(action, dyn_noise, obs_noise)

    def _step_single_fast(self, action):
        """num_envs == 1, host action, no noise: the drop-in path under the reference's callers.  One ctypes call
        (dexsim_step_single), persistent argument structs, result decoded from mapped host memory."""
        io = self._io_single
        if io is None:
            self._pin_action()
            if self._pack_host is None:
                self._next_pack_tag()                   # allocates the mapped result record
            io = self._io_single = _lib.DexsimStepIO.from_buffer_copy(self._io)
            io.action, io.action_layout = self._action_pin.data_ptr(), 1
            self._clear_noise(io)
            self._io_single_ref = C.byref(io)
            self._pack_ptr = self._pack_host.data_ptr()
        # float64 / list actions are cast exactly like the general path's astype(np.float32)
        self._action_pin_np[:15] = np.asarray(action).reshape(15)
        self._pack_tag = tag = self._pack_tag + 1.0
        rc = self._lib.dexsim_step_single(self._state_ref, self._params_ref, self._groups_ptr, self._goe_ptr,
                                          self._io_single_ref, self._pack_ptr, tag, _raw_stream(self.device.index))
        if rc:
            raise _lib.DexsimError(rc, "dexsim_step_single")
        return self._single_wait_decode(tag, False)

    def _step_general(self, action, dyn_noise, obs_noise):
        io = self._io
        a = self._ingest_action(action)
        io.action, io.action_layout = a.data_ptr(), 1
        io.flags ^= self._alternate_tiles
        keep = [a]
        group_obs, group_dyn = self._group_noise
        want_dyn = dyn_noise is not None or self.dynamics_noise_std > 0.0 or group_dyn
        want_obs = obs_noise is not None or self.observation_noise_std > 0.0 or group_obs
        self._clear_noise(io)
        self._io_has_noise = want_dyn or want_obs
        if want_dyn or want_obs:
            self._noise_buffers()
        fused = self.fused_noise
        if want_dyn:
            if dyn_noise is not None:
                dn = self._soa(dyn_noise, 15)
                io.dyn_noise = dn.data_ptr(); keep.append(dn)
            elif group_dyn and not self.dynamics_noise_std > 0.0:
                io.sigma_dyn = -1.0                         # each env's group value, drawn inside the step kernel
            elif fused:
                io.sigma_dyn = self.dynamics_noise_std      # Philox normals drawn inside the step kernel
            else:
                dn = self._dyn_noise
                _lib.check(self._lib.dexsim_fill_normal(
                    self._state_ref, self._params_ref, _L.RNG_STREAM_DYN, 15,
                    C.c_float(self.dynamics_noise_std), dn.data_ptr(), self._stream()), "dexsim_fill_normal")
                io.dyn_noise = dn.data_ptr(); keep.append(dn)
        if obs_noise is not None:
            on = self._soa(obs_noise, 45)
            io.obs_noise, io.noisy_obs = on.data_ptr(), self._noisy_obs.data_ptr()
            keep.append(on)
        elif want_obs and (fused or not self.observation_noise_std > 0.0):
            io.sigma_obs = self.observation_noise_std if self.observation_noise_std > 0.0 else -1.0
            io.noisy_obs = self._noisy_obs.data_ptr()
        post_step_noise = want_obs and obs_noise is None and not fused and self.observation_noise_std > 0.0
        if post_step_noise and self._final_obs is not None:
            raise NotImplementedError("final_observation needs the observation noise drawn inside the step kernel "
                                      "(fused_noise=True)")
        if self.single and not post_step_noise:
            # one launch: the step and the packed read-back of what step() returns (dexsim_step_single)
            tag = self._next_pack_tag()
            _lib.check(self._lib.dexsim_step_single(self._state_ref, self._params_ref, self._groups_ptr, self._goe_ptr,
                                                    self._io_ref, self._pack_host.data_ptr(), tag, self._stream()),
                       "dexsim_step_single")
            return self._single_wait_decode(tag, after_reset=False)
        self._launch_step()
        if post_step_noise:
            # Philox observation noise is keyed by (episode, step count AFTER the step), so it is
            # drawn once the step has run (evaluation/robustness_tests.py:204-205)
            _lib.check(self._lib.dexsim_fill_normal(
                self._state_ref, self._params_ref, _L.RNG_STREAM_OBS, 45,
                C.c_float(self.observation_noise_std), self._obs_noise.data_ptr(), self._stream()), "dexsim_fill_normal")
            torch.add(self._obs, self._obs_noise, out=self._noisy_obs)
        if self.single:
            return self._single_readback(after_reset=False, noisy=want_obs)
        obs = self._emit_obs(noisy=want_obs)
        n = self.num_envs
        return (obs, self._reward[:n], self._terminated[:n].view(torch.bool), self._truncated[:n].view(torch.bool),
                self._make_info())

    def capture_step(self, action_buffer, steps=1):
        """CUDA-graph the hot path for small batches, where one step is bound by the ~8 us host launch path
        rather than by the GPU: returns ``replay()`` which re-runs ``steps`` env-steps reading the actions
        from ``action_buffer`` (CUDA float32 [num_envs, 15], or [steps, num_envs, 15], or a sequence of ``steps``
        [num_envs, 15] tensors, which may repeat; refill them in place between replays) and returns the same persistent
        output tensors as ``step()``.
        Kernel parameters (seed, reward weights, group count ...) are frozen at capture time; curriculum
        updates still apply because the group table is read from device memory at replay."""
        if self.single or self._noisy_env:
            raise RuntimeError("capture_step() is for batched, noise-free stepping")
        if isinstance(action_buffer, (list, tuple)):
            if len(action_buffer) != steps:
                raise ValueError("capture_step(): one action tensor per captured step")
            a = [t.reshape(self.num_envs, 15) for t in action_buffer]
        else:
            a = action_buffer.reshape(steps, self.num_envs, 15)
        if self._groups_dirty:
            self._sync_groups()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):                  # warm-up outside capture (lazy module load, attribute calls)
            state = self.state_dict()
            self.step(a[0])
            self.load_state_dict(state)
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for k in range(steps):
                self.step(a[k])
        out = self._step_out

        def replay():
            if self._groups_dirty:
                self._sync_groups()
            self._h_primed_slot = None
            graph.replay()
            return out

        replay.graph = graph
        return replay

    def _step_soa(self, action_soa):
        """Step with actions already in the device layout [15, ld] (tests / internal callers)."""
        io = self._io
        self._h_primed_slot = None
        io.action, io.action_layout = action_soa.data_ptr(), 0
        self._clear_noise(io)
        self._launch_step()
        return self._step_out

    def _launch_step(self):
        extra = () if self._step_final_obs is None else (self._step_final_obs,)
        _lib.check(self._step_entry(self._state_ref, self._params_ref, self._groups_ptr, self._goe_ptr, self._io_ref,
                                    *extra, self._stream()), self._step_entry_name)

    def _reset_outputs(self):
        obs = self._emit_obs(reset=True)          # also draws the reset observation's noise when enabled
        if self.single:
            o, _, _, _, info = self._single_readback(after_reset=True, noisy=self.observation_noise_std > 0.0)
            return o, info
        return obs, self._make_info(after_reset=True)

    def _single_readback(self, after_reset, noisy):
        """num_envs == 1: one pack kernel + one 512-byte D2H copy -> the reference's return values
        (obs float32[45], reward float, terminated, truncated, info dict of envs/manipulation_env.py:266-283)."""
        io = _lib.DexsimStepIO.from_buffer_copy(self._io)
        if noisy:
            io.noisy_obs, io.obs_noise = self._noisy_obs.data_ptr(), self._noisy_obs.data_ptr()
        else:
            io.noisy_obs = io.obs_noise = None
        tag = self._next_pack_tag()
        _lib.check(self._lib.dexsim_pack_env_tagged(self._state_ref, C.byref(io), 0, int(after_reset),
                                                    self._pack_host.data_ptr(), tag, self._stream()), "dexsim_pack_env_tagged")
        return self._single_wait_decode(tag, after_reset)

    def _next_pack_tag(self):
        if self._pack_host is None:
            # page-locked and (unified addressing) mapped into the device: the pack code writes straight into it
            self._pack_host = torch.zeros(64, dtype=torch.float64).pin_memory()
            self._pack_np = self._pack_host.numpy()
            self._pack_tag = 0.0
        self._pack_tag += 1.0
        return self._pack_tag

    def _single_wait_decode(self, tag, after_reset):
        h = self._pack_np
        # the tag lands after the 63 data slots: poll it instead of paying a stream synchronize, but never
        # spin forever -- a failed launch surfaces through the synchronize below
        for _ in range(20000):
            if h[63] == tag:
                break
        else:
            torch.cuda.current_stream(self.device).synchronize()
            if h[63] != tag:
                raise RuntimeError("dexsim_pack_env_tagged: result did not arrive")
        obs = h[:45].astype(np.float32)
        info = {
            "step_count": int(h[49]),
            "object_position": h[50:53].copy(),
            "num_contacts": int(h[48]),
            "curriculum": {"object_size": float(h[53]), "object_mass": float(h[54]), "friction_coefficient": float(h[55])},
        }
        reward = float(h[45])
        if not after_reset and self._custom_reward is not None:
            # envs/manipulation_env.py:297-325: finger tips as the reference builds them (float32 sum of a finger's
            # joints, "* 0.1" in float32, broadcast into a float64 triple), then the user's compute()
            jp = obs[0:15]
            tips = np.stack([np.zeros(3) + np.sum(jp[3 * f:3 * f + 3]) * 0.1 for f in range(5)])
            comps = self._custom_reward.compute(joint_positions=jp, finger_tips=tips, object_position=h[50:53].copy(),
                                                contacts=obs[40:45].copy(), num_fingers=5, joints_per_finger=3)
            reward = comps["total"]
            info["reward_components"] = comps
        elif not after_reset and self._comps is not None:
            info["reward_components"] = {"total": float(h[45]), "distance": float(h[56]), "contact": float(h[57]),
                                         "closure": float(h[58]), "stability": float(h[59])}
        if self.info_success and not after_reset:
            info["success"] = bool(h[46])
        return obs, reward, bool(h[46]), bool(h[47]), info

    def _emit_obs(self, reset=False, noisy=False):
        n = self.num_envs
        if reset and self.observation_noise_std > 0.0:
            # evaluation/robustness_tests.py:171-175: noise is added to the reset observation too
            self._noise_buffers()
            _lib.check(self._lib.dexsim_fill_normal(
                C.byref(self._state), C.byref(self._params), _L.RNG_STREAM_OBS, 45,
                C.c_float(self.observation_noise_std), self._obs_noise.data_ptr(), self._stream()), "dexsim_fill_normal")
            torch.add(self._obs, self._obs_noise, out=self._noisy_obs)
            noisy = True
        src = self._noisy_obs if noisy else self._obs
        if self.single:
            return None                           # read back by _single_readback
        return src[:, :n].t()

    def _make_info(self, after_reset=False):
        n = self.num_envs
        if self._info is None:
            self._info = {
                "step_count": self._step_count[:n],
                "object_position": self._op64[:, :n].t(),
                "num_contacts": self._num_contacts[:n],
                "curriculum": {"object_size": self._size[:n], "object_mass": self._mass[:n],
                               "friction_coefficient": self._friction[:n]},
            }
            if self._comps is not None:
                self._info["reward_components"] = {
                    "total": self._reward[:n], "distance": self._comps[0, :n], "contact": self._comps[1, :n],
                    "closure": self._comps[2, :n], "stability": self._comps[3, :n]}
            if self._finished is not None:
                self._info["finished"] = self._finished[:n].view(torch.bool)
            if self._final_obs is not None:
                # batch first like obs; row i is the observation that ended env i's episode, valid where info["finished"]
                self._info["final_observation"] = self._final_obs[:, :n].t()
            if self.info_success:
                self._info["success"] = self._terminated[:n].view(torch.bool)
        if after_reset:
            info = dict(self._info)
            info["num_contacts"] = sum(((self._cmask[:n] >> f) & 1) for f in range(5)).to(torch.uint8)
            info.pop("reward_components", None)
            info.pop("final_observation", None)
            return info
        return self._info

    # ------------------------------------------------------------------ host-buffer step (end to end)
    def _host_buffers(self, slot):
        bufs = self._h_slots
        if slot not in bufs:
            n, ld = self.num_envs, self.ld
            pin = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype).pin_memory()
            b = {"obs": pin(45, ld, dtype=torch.float32), "reward": pin(ld, dtype=torch.float32),
                 "term": pin(ld, dtype=torch.uint8), "trunc": pin(ld, dtype=torch.uint8), "nc": pin(ld, dtype=torch.uint8),
                 "cmask": pin(ld, dtype=torch.uint8)}
            b["obs"][_L.ROW_QUAT].fill_(1.0)          # constant quaternion rows are never re-copied
            b["info"] = {"num_contacts": b["nc"][:n], "contact_mask": b["cmask"][:n]}
            if self.final_observation:
                # written by the finish-and-reset pass through the mapped buffer: ~180 bytes per FINISHED env cross PCIe
                b["fin"], b["final"] = pin(ld, dtype=torch.uint8), pin(n, 45, dtype=torch.float32)
                b["info"].update(finished=b["fin"][:n].view(torch.bool), final_observation=b["final"])
            b["out"] = (b["obs"][:, :n].t(), b["reward"][:n], b["term"][:n].view(torch.bool), b["trunc"][:n].view(torch.bool),
                        b["info"])
            bufs[slot] = b
        return bufs[slot]

    def step_host(self, action_host, chunks=None, sync=True, packed_contacts=False, slot=0):
        """One step with HOST buffers: ``action_host`` is a float32 [num_envs, 15] NumPy array or CPU
        tensor (pinned memory makes the copies true DMA); returns CPU tensors
        ``(obs [num_envs,45], reward, terminated, truncated, info)`` living in pinned buffers that
        the next call with the same ``slot`` overwrites.  One C-ABI call (dexsim_step_host): H2D copy of the actions,
        the step kernel, D2H copies of observation / reward / flags, stream synchronize.  Large batches are
        split into ``chunks`` ranges (default: one per 8,192 envs, at most 8) so that the upload of one
        range overlaps the kernel and the download of the others.  Batches up to 160K envs (``host_zero_copy``) skip the
        download copies once the buffers are current: the step kernel stores its results into the pinned buffers itself.

        ``sync=False``: return as soon as everything is enqueued; call ``host_sync()`` (or synchronize the current
        stream) before reading the returned tensors.  With two result ``slot`` s a caller can overlap the upload of the
        next step (or of another env group) with this step's download.
        ``packed_contacts=True``: the five 0/1 contact columns of the observation (obs[:, 40:45]) are NOT downloaded;
        ``info["contact_mask"]`` (uint8, bit f = finger f) carries the same information in one byte per env
        (-11 % download bytes).  ``expand_contacts_host(slot)`` fills the columns in on the host when needed.

        ``final_observation=True`` envs (dexsim_step_host_final): ``info["finished"]`` (bool [num_envs]) marks the envs
        whose episode ended in this step and was reset, and ``info["final_observation"]`` (float32 [num_envs, 45]) holds,
        where ``info["finished"]``, the observation that ended it -- all 45 entries, also with ``packed_contacts``.  Its
        other rows keep stale values.  Both are pinned buffers of the ``slot`` like the other outputs; the GPU writes the
        rows of finished envs only, straight into the buffer.

        Not available in ``autoreset_mode="next_step"`` (its per-env outputs carry no ``finished`` vector)."""
        if self._next_step:
            raise NotImplementedError("step_host() does not support autoreset_mode='next_step'; use step()")
        if not self._did_reset:
            raise RuntimeError("call reset() before step_host()")
        n = self.num_envs
        b = self._host_buffers(slot)
        a = action_host if isinstance(action_host, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(action_host, np.float32))
        if a.dtype != torch.float32 or not a.is_contiguous() or a.numel() != n * 15:
            a = a.to(torch.float32).reshape(n, 15).contiguous()
        flags = _L.HOST_SKIP_QUAT | (0 if sync else _L.HOST_ASYNC) | (_L.HOST_PACKED_CONTACTS if packed_contacts else 0)
        if sync and not packed_contacts and self.host_expand_contacts:
            # default transport of a synchronous call: the contact columns travel as their 1-byte mask and the calling
            # thread expands them into the pinned observation while the other rows are still being downloaded --
            # the returned observation is complete, 20 of 171 bytes per env never cross PCIe
            flags |= _L.HOST_PACKED_CONTACTS | _L.HOST_EXPAND_CONTACTS
        if sync and self.host_static_rows and self._h_primed_slot == slot:
            # object x, y and their velocities only change when an episode is reset; the step kernel mirrors every such
            # change straight into this slot's pinned observation, which has been current since the previous call:
            # those four rows are not downloaded (another 16 bytes per env)
            flags |= _L.HOST_STATIC_ROWS
            zc = self.host_zero_copy
            if (n <= 163840 if zc == "auto" else bool(zc)) and (flags & _L.HOST_PACKED_CONTACTS):
                # ... and nothing else is downloaded either: the step kernel's own bulk stores write the joint rows, z, its
                # velocity, the contact masks, reward and flags into the pinned buffers tile by tile (DEXSIM_HOST_ZERO_COPY)
                flags |= _L.HOST_ZERO_COPY
                if chunks is None:
                    chunks = max(1, min(8, n // 16384))
        with torch.cuda.device(self.device):
            self._sync_groups()
            io = self._io
            io.action, io.action_layout = self._action_dev.data_ptr(), 1
            self._clear_noise(io)
            args = (C.byref(self._state), C.byref(self._params), self._ptr(self._groups_dev), self._ptr(self._goe),
                    C.byref(io), a.data_ptr(), b["obs"].data_ptr(), b["reward"].data_ptr(), b["term"].data_ptr(),
                    b["trunc"].data_ptr(), b["nc"].data_ptr(), b["cmask"].data_ptr())
            tail = (int(chunks) if chunks is not None else max(1, min(8, n // 8192)), flags, self._stream())
            if self.final_observation:
                _lib.check(self._lib.dexsim_step_host_final(*args, b["fin"].data_ptr(), b["final"].data_ptr(), *tail),
                           "dexsim_step_host_final")
            else:
                _lib.check(self._lib.dexsim_step_host(*args, *tail), "dexsim_step_host")
        # this slot's observation is current now; any other entry point that touches the state resets the marker
        self._h_primed_slot = slot if sync else None
        if not sync:
            # the upload may still be reading the action buffer: keep it alive until this slot is used again
            self._host_keepalive[slot] = a
        return b["out"]

    def host_sync(self):
        """Wait for every ``step_host(sync=False)`` issued on the current stream: their host tensors are valid afterwards."""
        torch.cuda.current_stream(self.device).synchronize()

    def expand_contacts_host(self, slot=0):
        """Fill obs[:, 40:45] of a ``packed_contacts`` result in from its contact mask (host-side, vectorised)."""
        b = self._host_buffers(slot)
        _lib.check(self._lib.dexsim_expand_contact_rows(b["obs"].data_ptr(), b["cmask"].data_ptr(), self.num_envs, self.ld),
                   "dexsim_expand_contact_rows")
        return b["out"][0]

    # ------------------------------------------------------------------ fused rollout
    def enable_episode_log(self, capacity):
        """Allocate a device log of finished episodes (one 32-byte record each, the per-episode dict of
        evaluation/evaluator.py:163-173); ``read_episode_log()`` returns it.  Records beyond the capacity
        are counted but dropped."""
        self._ep_log = torch.zeros(int(capacity) * 32, dtype=torch.uint8, device=self.device)
        self._ep_log_count = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._ep_log_capacity = int(capacity)

    def enable_history(self, steps):
        """Allocate a device buffer [steps, ld] of per-step contact COUNTS (the contact_history of
        evaluation/evaluator.py:148-150 is count-encoded) written by rollout()."""
        self._hist = torch.zeros(int(steps), self.ld, dtype=torch.uint8, device=self.device)
        self._hist_steps = int(steps)

    def enable_trajectory(self, steps, final_observation=False):
        """Allocate device buffers for ``steps`` rows of per-step trajectory that every later ``rollout()`` of at most
        that many steps fills as it steps (``dexsim_rollout_record``); ``trajectory`` returns them.  Row t of a call
        holds what the (t+1)-th step would return from ``step()`` on a same-step auto-reset env: the observation after
        the step and a possible reset, the float32 reward, ``terminated`` / ``truncated``, ``finished`` (the loop bound
        included) and the policy's action before dynamics noise.  The buffers take ``steps x num_envs x 247`` bytes:
        about 13 GB for 1 Mi envs x 50 steps.  A recording rollout always runs the one-thread-per-env kernel.
        ``final_observation=True`` also records, on every row where ``finished`` is set, the observation that ended the
        episode, before its reset (``dexsim_rollout_record_final``): what ``info["final_observation"]`` of a
        ``final_observation=True`` env's ``step()`` holds, and the ``next_obs`` of that transition.  Its buffer adds
        ``steps x num_envs x 180`` bytes: 9.4 GB more for 1 Mi envs x 50 steps."""
        k, ld, dev = int(steps), self.ld, self.device
        if k < 1:
            raise ValueError("steps must be >= 1")
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)
        self._traj = {"obs": z(k, 45, ld), "action": z(k, 15, ld), "reward": z(k, ld), "terminated": z(k, ld, dtype=torch.uint8),
                      "truncated": z(k, ld, dtype=torch.uint8), "finished": z(k, ld, dtype=torch.uint8)}
        if final_observation:
            self._traj["final_observation"] = z(k, 45, ld)
        self._traj_rows, self._traj_has_action = 0, False

    @property
    def trajectory(self):
        """The rows the last ``rollout()`` recorded, as batch-first views of the device buffers: ``obs`` [k, n, 45],
        ``action`` [k, n, 15] (absent after ``policy="external"``: the caller holds the actions), ``reward`` [k, n]
        float32 and ``terminated`` / ``truncated`` / ``finished`` [k, n] bool.  After
        ``enable_trajectory(steps, final_observation=True)`` also ``final_observation`` [k, n, 45]: the observation that
        ended the episode, valid where ``finished`` is True (other entries are not written).  With ``one_episode=True``
        an env's rows after the step that ended its episode are not written.  The next ``rollout()`` overwrites them."""
        if self._traj is None:
            raise RuntimeError("enable_trajectory() first")
        k, n, tr = self._traj_rows, self.num_envs, self._traj
        out = {"obs": tr["obs"][:k, :, :n].transpose(1, 2), "reward": tr["reward"][:k, :n]}
        if "final_observation" in tr:
            out["final_observation"] = tr["final_observation"][:k, :, :n].transpose(1, 2)
        if self._traj_has_action:
            out["action"] = tr["action"][:k, :, :n].transpose(1, 2)
        for name in ("terminated", "truncated", "finished"):
            out[name] = tr[name][:k, :n].view(torch.bool)
        return out

    def enable_learner(self, learning_rate=0.01, exploration_noise=0.3, action_clip_range=0.5):
        """One independent SimpleLearner per env (policies/simple_learner.py:27-47): ``learner_mean``
        [num_envs, 15] starts at zero, ``learner_best`` at -inf; ``rollout(policy="learner")`` trains them."""
        self._learner_mean = torch.zeros(15, self.ld, dtype=torch.float32, device=self.device)
        self._learner_best = torch.full((self.ld,), float("-inf"), dtype=torch.float64, device=self.device)
        self._learner_hp = (float(exploration_noise), float(learning_rate), float(action_clip_range))

    @property
    def learner_mean(self):
        return self._learner_mean[:, :self.num_envs].t()

    @property
    def learner_best(self):
        return self._learner_best[:self.num_envs]

    def read_episode_log(self, sort=True):
        """Finished episodes as a NumPy structured array (fields of DexsimEpisodeRecord), ordered by
        (t_end, env_gid) -- the order a sequential caller would have seen them in."""
        if self._ep_log is None:
            raise RuntimeError("enable_episode_log() first")
        produced = int(self._ep_log_count.item())
        kept = min(produced, self._ep_log_capacity)
        raw = self._ep_log[:kept * 32].cpu().numpy()
        rec = raw.view(_L.EPISODE_RECORD_DTYPE).copy()
        if sort and kept:
            rec = rec[np.lexsort((rec["env_gid"], rec["t_end"]))]
        self.episode_log_overflow = produced - kept
        return rec

    def rollout(self, k_steps, policy="random", actions=None, dyn_noise=None, loop_max_steps=None,
                success_is_terminated=None, respawn=True, zero_counters=False, one_episode=False,
                learner_act_noise=None, learner_upd_noise=None):
        """k env-steps per env in ONE kernel launch with the policy generated in-kernel
        (caller loops of training/episode_utils.py:42-53 / evaluation/evaluator.py:135-158).
        Returns (counters [G, 18] int64, ret_sums [G, 2] float64) device tensors (accumulated).
        ``one_episode=True``: every env stops at the end of its first episode and is left un-reset
        (run_episode / evaluate_episode semantics); otherwise finished episodes auto-reset.
        Not available in ``autoreset_mode="next_step"``: the fused rollout resets in the same step, and an episode a
        step() left pending would be counted twice.
        After ``enable_trajectory(steps)`` the call also records every step (``trajectory``), with
        ``final_observation=True`` the terminal observation of every episode it ends too; ``k_steps`` must not exceed
        ``steps``.
        ``policy`` may also be an ``MlpPolicy``: every env acts on the observation ``step()`` would return for its
        current state (with the env's observation noise where its ``sigma_obs`` > 0), through the network, in the same
        launch (``dexsim_rollout_mlp``); recorded actions are the policy's, before dynamics noise."""
        if self._next_step:
            raise NotImplementedError("rollout() resets finished episodes in the same step; it does not support "
                                      "autoreset_mode='next_step'")
        if not self._did_reset:
            raise RuntimeError("call reset() before rollout()")
        self._h_primed_slot = None
        if self._ep_return is None:
            raise RuntimeError("rollout() needs track_episodes=True (per-env history summaries)")
        mlp = policy if isinstance(policy, MlpPolicy) else None
        if mlp is not None:
            if actions is not None or learner_act_noise is not None or learner_upd_noise is not None:
                raise ValueError("an MlpPolicy rollout takes no actions and no learner noise")
            if mlp.device != self.device:
                raise ValueError(f"the policy lives on {mlp.device}, the env on {self.device}")
            kind = None
        else:
            kind = {"external": _L.POLICY_EXTERNAL, "random": _L.POLICY_RANDOM, "heuristic": _L.POLICY_HEURISTIC,
                    "learner": _L.POLICY_LEARNER}[policy]
        if kind == _L.POLICY_LEARNER and self._learner_mean is None:
            self.enable_learner()
        with torch.cuda.device(self.device):
            self._sync_groups()
            if zero_counters:
                self.counters.zero_(); self.ret_sums.zero_()
            p = _lib.DexsimParams.from_buffer_copy(self._params)
            p.loop_max_steps = self.max_episode_steps if loop_max_steps is None else int(loop_max_steps)
            p.success_is_terminated = int(self.success_is_terminated if success_is_terminated is None else success_is_terminated)
            p.respawn = int(respawn)
            keep = []
            rio = _lib.DexsimRolloutIO()
            if kind == _L.POLICY_EXTERNAL:
                buf = self._soa(actions, 15, steps=k_steps)
                rio.actions = buf.data_ptr(); keep.append(buf)
            if dyn_noise is not None:
                nbuf = self._soa(dyn_noise, 15, steps=k_steps)
                rio.dyn_noise = nbuf.data_ptr(); keep.append(nbuf)
            rio.counters, rio.ret_sums = self._ptr(self.counters), self._ptr(self.ret_sums)
            if kind == _L.POLICY_LEARNER:
                rio.learner_mean, rio.learner_best = self._learner_mean.data_ptr(), self._learner_best.data_ptr()
                rio.learner_exploration, rio.learner_lr, rio.learner_clip = self._learner_hp
                for name, src, dt in (("learner_act_noise", learner_act_noise, torch.float32),
                                      ("learner_upd_noise", learner_upd_noise, torch.float64)):
                    if src is not None:         # pre-drawn [k, n, 15] (parity runs)
                        b = self._soa(src, 15, dt, steps=k_steps)
                        setattr(rio, name, b.data_ptr()); keep.append(b)
            if self._ep_log is not None:
                rio.ep_log, rio.ep_log_count = self._ep_log.data_ptr(), self._ep_log_count.data_ptr()
                rio.ep_log_capacity = self._ep_log_capacity
            if self._hist is not None:
                rio.hist, rio.hist_steps = self._hist.data_ptr(), self._hist_steps
            rio.step_base = self._rollout_steps
            rio.one_episode = int(bool(one_episode))
            so, sd = self._group_sigma if self._group_cfgs is not None else (0.0, self.dynamics_noise_std)
            no_noise = not np.any(np.asarray(sd, dtype=np.float64) > 0.0)
            rio.flags = _L.ROLLOUT_NO_DYN_NOISE if no_noise else 0
            args = (C.byref(self._state), C.byref(p), self._ptr(self._groups_dev), self._ptr(self._goe), int(k_steps), kind,
                    C.byref(rio))
            if mlp is not None:
                traj, fo = None, None
                if self._traj is not None:
                    tr = self._traj
                    traj = _lib.DexsimTrajectory(tr["obs"].data_ptr(), tr["action"].data_ptr(), tr["reward"].data_ptr(),
                                                 tr["terminated"].data_ptr(), tr["truncated"].data_ptr(),
                                                 tr["finished"].data_ptr(), tr["obs"].shape[0])
                    fo = tr["final_observation"].data_ptr() if "final_observation" in tr else None
                _lib.check(self._lib.dexsim_rollout_mlp(
                    C.byref(self._state), C.byref(p), self._ptr(self._groups_dev), self._ptr(self._goe), int(k_steps),
                    C.byref(rio), C.byref(mlp._struct), None if traj is None else C.byref(traj), fo, self._stream()),
                    "dexsim_rollout_mlp")
                if traj is not None:
                    self._traj_rows, self._traj_has_action = int(k_steps), True
            elif self._traj is None:
                _lib.check(self._lib.dexsim_rollout(*args, self._stream()), "dexsim_rollout")
            else:
                tr = self._traj
                traj = _lib.DexsimTrajectory(tr["obs"].data_ptr(), None if kind == _L.POLICY_EXTERNAL else tr["action"].data_ptr(),
                                             tr["reward"].data_ptr(), tr["terminated"].data_ptr(), tr["truncated"].data_ptr(),
                                             tr["finished"].data_ptr(), tr["obs"].shape[0])
                if "final_observation" in tr:
                    _lib.check(self._lib.dexsim_rollout_record_final(*args, C.byref(traj), tr["final_observation"].data_ptr(),
                                                                     self._stream()), "dexsim_rollout_record_final")
                else:
                    _lib.check(self._lib.dexsim_rollout_record(*args, C.byref(traj), self._stream()), "dexsim_rollout_record")
                self._traj_rows, self._traj_has_action = int(k_steps), kind != _L.POLICY_EXTERNAL
            self._rollout_steps += int(k_steps)
            self._spawned = True
        return self.counters, self.ret_sums

    # ------------------------------------------------------------------ misc API of the reference env
    def render(self):
        if self.render_mode == "rgb_array":
            return np.zeros((480, 640, 3), dtype=np.uint8)     # envs/manipulation_env.py:338-346 placeholder
        return None

    def close(self):
        pass

    @property
    def unwrapped(self):
        return self

    def state_dict(self):
        """Everything a resumed run needs to continue bit for bit: all device state, the host-side PCG64 generators that
        drive later resets in rng="numpy" mode, the Philox seed, the rollout step base (history rows / t_end), the
        first-reset flag and the per-env SimpleLearner state when enabled.  ``torch.save``-able."""
        keys = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction",
                "_episode", "_ep_return", "_ep_stats", "counters", "ret_sums", "_learner_mean", "_learner_best")
        sd = {k: getattr(self, k).clone() for k in keys if getattr(self, k, None) is not None}
        sd["_host"] = {
            "seed": self.seed, "rollout_steps": self._rollout_steps, "spawned": self._spawned, "did_reset": self._did_reset,
            "np_rngs": None if self._np_rngs is None else [None if r is None else r.bit_generator.state for r in self._np_rngs],
            "learner_hp": getattr(self, "_learner_hp", None),
        }
        return sd

    def load_state_dict(self, sd):
        self._h_primed_slot = None
        host = sd.get("_host")
        for k, v in sd.items():
            if k == "_host":
                continue
            if getattr(self, k, None) is None and k in ("_learner_mean", "_learner_best"):
                explo, lr, clip = (host or {}).get("learner_hp") or (0.3, 0.01, 0.5)
                self.enable_learner(learning_rate=lr, exploration_noise=explo, action_clip_range=clip)
            getattr(self, k).copy_(v)
        self._did_reset = True
        self._spawned = True
        if host is not None:
            self.seed = int(host["seed"])
            self._params.seed = self.seed & 0xFFFFFFFFFFFFFFFF
            self._rollout_steps = int(host["rollout_steps"])
            self._spawned, self._did_reset = bool(host["spawned"]), bool(host["did_reset"])
            if host["np_rngs"] is not None:
                self._np_rngs = []
                for state in host["np_rngs"]:
                    if state is None:
                        self._np_rngs.append(None)
                    else:
                        r = np.random.Generator(np.random.PCG64())
                        r.bit_generator.state = state
                        self._np_rngs.append(r)
