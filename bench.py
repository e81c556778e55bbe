#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched manipulation simulator (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--num-envs E] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one env.step() of EVERY env of the job (E envs per GPU, weak scaling).
Workload (BASELINE.json configs[1] scaled to the metric's 1M-env end so the state is larger than
L2): experiments/config_default.json -- dense reward, max_episode_steps 200,
CurriculumScheduler(easy -> hard, threshold 0.3, window 15, min episodes 20, 5 steps) fed from
the device counters, random policy actions U(-1,1) resident in HBM, auto-reset (respawn) with per-group
episode counters (what the scheduler consumes).  Untimed before the W warm-up steps: a 100-step curriculum
pre-roll (--preroll-steps) in which the scheduler climbs to its final level.

Printed JSON (one line, rank 0):
  value      whole-job env-steps/s, inputs resident in HBM (API mode: dexsim_step per step)
  e2e        same metric through env.step_host(): pinned HOST actions in, obs/reward/flags out,
             H2D + D2H copies inside the timed region
  roofline   step kernel: algorithmic 410 B/env-step (SURVEY.md 8d) / CUDA-event kernel time; `frac` over the K timed
             steps, `frac_sustained` over an extra window of >= 400 steps (two full 200-step episode cycles) whatever K is
  cpu_baseline   the reference's own Python loop on this box's host cores (bounded sample)
  tracking_full       the same loop with full per-env episode tracking (returns, failure labels), >= 250 steps
  noisy_api           CombinedNoiseWrapper semantics in API mode: sigma_obs 0.05, sigma_dyn 0.1 drawn inside the step kernel
  strong_1m           BASELINE configs[3] at every GPU count: 1,048,576 envs IN TOTAL (config_variable ranges) sharded
                      over the N ranks -- API mode eager / CUDA-graph replay / fused rollout, per-GPU roofline fraction,
                      and a sha256 of the all-reduced counter table that must not depend on N
  single_env_dropin   configs[0]: ONE env behind the reference's reset/step API with a host policy
  fused_rollout, sweep   extra measurements (in-kernel policy; other env counts, eager and CUDA-graph replay)
`--impl reference` times the UNMODIFIED reference (byte-compiled in oracle/_ref) with one
process per host core; it never touches CUDA.
`--dump-outputs DIR` writes what the last timed step returned (rank 0's envs) as DIR/<name>.npy; the inputs depend
on the arguments only, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALGO_BYTES_PER_ENV_STEP = 410          # SURVEY.md 8d / BASELINE.md section 4 (API mode)
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
# experiments/config_default.json:16-23 and :3-12
SCHED = dict(success_rate_threshold=0.3, window_size=15, min_episodes_before_progression=20, progression_steps=5)
MAX_EPISODE_STEPS = 200
SEED = 42
DUMP_ROWS = 1 << 17                    # --dump-outputs: ~34 MB of arrays at this many envs, under the 64 MB budget


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--num-envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--poll-every", type=int, default=100, help="curriculum driver poll period (steps)")
    ap.add_argument("--preroll-steps", type=int, default=100,
                    help="untimed steps before the warm-up in which the curriculum climbs to its final level")
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--sustained-steps", type=int, default=400,
                    help="extra timed window for roofline.frac_sustained (two full 200-step episode cycles)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong_1m section")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-tracking-variant", action="store_true", help="skip the extra run with full per-env episode tracking")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--ref-steps-per-proc", type=int, default=0,
                    help="reference arm: env-steps per process per bench step (0 = size from --ref-budget-seconds)")
    ap.add_argument("--ref-budget-seconds", type=float, default=120.0, help="reference arm: target wall time of the whole run")
    ap.add_argument("--ref-procs", type=int, default=0, help="reference arm: processes (0 = all host cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the observation, reward, flags and info arrays of the last timed step as DIR/<name>.npy "
                         f"(rank 0's envs; a fixed, seeded sample of {DUMP_ROWS} envs above that count)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------ reference arm
def _ref_worker(conn, steps_per_call, seed):
    """One process = one reference env driven exactly like config 2 on the CPU: dense reward,
    RandomPolicy, CurriculumScheduler(easy -> hard) updated per episode, fresh spawn per episode."""
    try:
        from oracle import ref_harness
        R = ref_harness.load()
        import numpy as np
        np.random.seed(seed)
        sched = R.CurriculumScheduler(R.CurriculumConfig.easy(), R.CurriculumConfig.hard(), **SCHED)
        env = R.DexterousManipulationEnv(curriculum_config=sched.get_current_config(), reward_type="dense",
                                         max_episode_steps=MAX_EPISODE_STEPS)
        policy = R.policies.RandomPolicy(env.action_space)
        obs, _ = env.reset(seed=seed)
        ep_steps = 0
        conn.send(("ready", ref_harness.kind()))
        while True:
            msg = conn.recv()
            if msg == "stop":
                break
            steps_per_call = int(msg[1])
            t0 = time.perf_counter()
            for _ in range(steps_per_call):
                obs, r, term, trunc, info = env.step(policy.select_action(obs))
                ep_steps += 1
                if term or trunc or ep_steps >= MAX_EPISODE_STEPS:
                    if sched.update(bool(term), ep_steps):
                        env.curriculum_config = sched.get_current_config()
                    env.object_position = None          # fresh-env semantics: respawn the object
                    obs, _ = env.reset()
                    ep_steps = 0
            conn.send(("done", time.perf_counter() - t0))
    except Exception as exc:       # pragma: no cover - reported to the parent
        conn.send(("error", repr(exc)))


def _oracle_port_worker(conn, steps_per_call, seed):
    """Fallback when the byte-compiled reference is absent: the C restatement (oracle port)."""
    try:
        import numpy as np
        from oracle import oracle
        n = 256
        ob = oracle.OracleBatch(n, dense=True, max_episode_steps=MAX_EPISODE_STEPS)
        grp = oracle.make_group(object_size=0.03, object_mass=0.2, friction_coefficient=0.3)
        rng = np.random.default_rng(seed)
        ob.reset_predrawn(rng.uniform(-0.1, 0.1, (n, 15)).astype(np.float32), 0.03, 0.2, 0.3,
                          np.stack([rng.uniform(-0.1, 0.1, n), rng.uniform(-0.1, 0.1, n), rng.uniform(0.05, 0.2, n)], 1).astype(np.float32))
        conn.send(("ready", "port"))
        while True:
            msg = conn.recv()
            if msg == "stop":
                break
            steps_per_call = int(msg[1])
            t0 = time.perf_counter()
            ob.rollout(grp, max(steps_per_call // n, 1), seed, policy_kind=1, respawn=True, loop_max_steps=MAX_EPISODE_STEPS)
            conn.send(("done", time.perf_counter() - t0))
    except Exception as exc:       # pragma: no cover
        conn.send(("error", repr(exc)))


def run_reference(args, n_gpus):
    """--impl reference: all host cores, each bench step = every process advances its env by
    `ref_steps_per_proc` env-steps.  Never imports torch.cuda."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import ref_harness
    kind = "reference" if ref_harness.available() else "port"
    ctx = mp.get_context("fork")
    procs = args.ref_procs or (os.cpu_count() or 1)
    target = _ref_worker if kind == "reference" else _oracle_port_worker
    workers = []
    for k in range(procs):
        a, b = ctx.Pipe()
        p = ctx.Process(target=target, args=(b, 0, SEED + k), daemon=True)
        p.start()
        workers.append((p, a))
    form = None
    for _, c in workers:
        tag, val = c.recv()
        if tag != "ready":
            print(json.dumps({"impl": "reference", "unavailable": f"worker failed: {val}"}))
            return 0
        form = val

    busy = [0.0] * procs            # per-process compute time: the reference is not charged for this harness's barriers

    def one_step(k):
        for _, c in workers:
            c.send(("go", k))
        for w, (_, c) in enumerate(workers):
            tag, val = c.recv()
            if tag != "done":
                raise RuntimeError(val)
            busy[w] += float(val)

    # size the per-step sample so that the whole --steps/--warmup run ends within a few minutes
    if args.ref_steps_per_proc > 0:
        spc = args.ref_steps_per_proc
    else:
        probe = 256
        t0 = time.perf_counter()
        one_step(probe)
        tau = (time.perf_counter() - t0) / probe                  # seconds per env-step per process
        budget = args.ref_budget_seconds / max(args.steps + args.warmup, 1)
        spc = int(max(256 if kind == "port" else 16, min(20000, budget / max(tau, 1e-9))))
    for _ in range(args.warmup):
        one_step(spc)
    busy = [0.0] * procs
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_step(spc)
    dt = time.perf_counter() - t0
    for p, c in workers:
        c.send("stop")
    for p, _ in workers:
        p.join(timeout=5)
    steps_per_bench_step = procs * (spc if kind == "reference" else max(spc // 256, 1) * 256)
    # whole-host throughput = sum over processes of (env-steps / that process's own compute time): the per-step
    # barrier of this harness (stragglers, pipe round trips) is not held against the reference
    per_proc_steps = steps_per_bench_step / procs * args.steps
    value = sum(per_proc_steps / b for b in busy if b > 0) if all(b > 0 for b in busy) else steps_per_bench_step * args.steps / dt
    sample = (f"{procs} processes x 1 env x {spc} env-steps per bench step, {args.steps} steps; config_default dense + "
              f"CurriculumScheduler + RandomPolicy; reference form: {form}; value = sum over processes of env-steps / own "
              f"compute time (wall clock incl. harness barriers would give {steps_per_bench_step * args.steps / dt:.0f})")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": {"workload": "config_default.json dense + curriculum_scheduler, random_policy; reference Python loop, "
                               "one env per host process", "envs": procs},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            parts = [x.strip() for x in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx = float(parts[1])
            except ValueError:
                continue
            for name, flag in zip(names, parts[3:7]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------ output dump
def dump_outputs(out_dir, step_out, n):
    """Write what env.step() returned -- observation, reward, flags and every info array -- as <out_dir>/<name>.npy for
    the same fixed, seeded sample of env rows (all n when n <= DUMP_ROWS; env_index.npy lists them).  float64 arrays
    stay float64, the others are written as float32 (flags and counts are small integers, exact in float32)."""
    import numpy as np
    import torch
    obs, reward, terminated, truncated, info = step_out
    arrays = {"obs": obs, "reward": reward, "terminated": terminated, "truncated": truncated}

    def add(prefix, d):
        for k, v in d.items():
            if isinstance(v, dict):
                add(f"{prefix}{k}_", v)
            else:
                arrays[prefix + k] = v
    add("info_", info)
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(SEED).choice(n, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(obs.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))
    for name, t in arrays.items():
        a = t.index_select(0, idx).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))
    print(f"bench.py: wrote {len(arrays) + 1} arrays ({len(rows)} envs) to {out_dir}", file=sys.stderr)


# ------------------------------------------------------------------------------------ b200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    import dexterous_rl_manipulation_b200 as dx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = world                      # one rank per GPU; --gpus N without torchrun cannot use more than one
    if args.gpus != world and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run for multi-GPU "
              f"(measuring {world} GPU)", file=sys.stderr)

    cpu_base = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        cpu_base = measure_cpu_baseline(args)      # before CUDA is initialised (workers fork)

    # The contract is ONE JSON line on stdout.  NCCL (and anything else writing to the C-level stdout)
    # is sent to stderr for the whole run; the JSON line goes to the saved descriptor at the end.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    numa_bound = dx.distributed.bind_to_gpu_numa(local) if world > 1 else False   # before any pinned allocation
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    E = args.num_envs
    CC = dx.CurriculumConfig

    def make_env(n, seed=SEED, gid0=0, track=False):
        # track=False: auto-reset + per-group episode counters (episodes, successes, lengths) -- everything the
        # CurriculumScheduler consumes; track=True adds the per-env return / contact-history arrays that the
        # evaluation outputs (failure labels, return statistics) need
        env = dx.BatchedManipulationEnv(n, dev, max_episode_steps=MAX_EPISODE_STEPS, reward_type="dense",
                                        curriculum_config=CC.easy(), auto_reset=True, respawn=True,
                                        loop_max_steps=MAX_EPISODE_STEPS, track_episodes=track, seed=seed, env_gid0=gid0)
        sched = dx.CurriculumScheduler(CC.easy(), CC.hard(), **SCHED)
        drv = dx.BatchedCurriculumDriver(env, sched)
        env.reset(seed=seed)
        return env, sched, drv

    def action_pool(n, k=4):
        g = torch.Generator(device=dev).manual_seed(SEED + rank)
        return [torch.rand(n, 15, device=dev, generator=g) * 2 - 1 for _ in range(k)]

    def timed_api(env, drv, pool, steps, warmup, poll_every, preroll=True):
        # the scheduler reacts per episode in the reference; while it can still progress the counters are
        # polled every 10 steps (one tiny D2H), afterwards every `poll_every` steps
        def maybe_poll(t):
            if not poll_every or drv is None:
                return
            period = 10 if drv.scheduler.current_difficulty_level < 1.0 else poll_every
            if (t + 1) % period == 0:
                drv.poll()

        # curriculum pre-roll (untimed, before the W warm-up steps): the scheduler climbs easy -> hard within the first
        # few dozen steps of a million-env batch; short runs (--steps 2 --warmup 3) must not time that transient, with
        # its per-episode scheduler replay on the host, as if it were the steady state
        for t in range(args.preroll_steps if (poll_every and preroll) else 0):
            env.step(pool[t % len(pool)])
            maybe_poll(t)
        for t in range(warmup):
            env.step(pool[t % len(pool)])
            maybe_poll(t)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for t in range(steps):
            out = env.step(pool[t % len(pool)])
            maybe_poll(t)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tms = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        return ms, out

    # ---- main timed region: API mode, device-resident actions -------------------------------------
    env, sched, drv = make_env(E, gid0=rank * E)
    pool = action_pool(E)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, last_out = timed_api(env, drv, pool, args.steps, args.warmup, args.poll_every)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_out, E)      # before any later step overwrites the output buffers
    value = E * n_gpus * args.steps / (ms * 1e-3)
    launches = args.steps

    # ---- roofline of the dominant kernel: algorithmic bytes per launch / average launch duration over
    #      the timed region (CUDA events on the launching stream; one launch per step, GPU-bound at this
    #      size, so region time / steps is the kernel's average duration including reset waves) ----------
    k_ms = ms / args.steps
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = ALGO_BYTES_PER_ENV_STEP * E / (k_ms * 1e-3) / 1e9
    # sustained figure: the same loop continued for >= 400 steps (two full 200-step episode cycles with their reset
    # waves and curriculum polls), so that a short --steps window can neither flatter nor hide it
    sus_steps = max(int(args.sustained_steps), 1)
    ms_sus, _ = timed_api(env, drv, pool, sus_steps, 0, args.poll_every, preroll=False)
    k_ms_sus = ms_sus / sus_steps
    # measured DRAM traffic of this kernel (ncu, per launch) -- only quoted while the library is still built from the
    # sources it was measured on
    traffic, traffic_note, traffic_steady = None, None, None
    try:
        from dexterous_rl_manipulation_b200.build import build_info
        with open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")) as fh:
            tr = json.load(fh)
        bi = build_info()
        cur = bi.get("step_kernel_sha256") if bi.get("fresh") else None      # device code of the step kernel the library was built from
        if int(tr.get("envs", 0)) == E and tr.get("step_kernel_sha256") and tr.get("step_kernel_sha256") == cur:
            traffic = tr["dram_bytes_per_launch"]
            traffic_steady = tr.get("steady_state")
            traffic_note = (f"ncu dram__bytes_read+write.sum of one isolated launch (caches flushed), {tr.get('report', 'profiles/')}, "
                            f"kernel sources sha256 {cur[:16]}; traffic_steady_state = the same counters inside a stepping loop "
                            f"(application replay, caches not flushed): a step walks the batch in the opposite direction of the "
                            f"previous one and finds its last tiles in L2, which is how `achieved` (algorithmic bytes / time) can "
                            f"exceed the DRAM copy peak")
        else:
            traffic_note = (f"not quoted: profiles/step_kernel_traffic.json was measured on kernel sources "
                            f"{str(tr.get('step_kernel_sha256'))[:16]}, this library is built from {str(cur)[:16]}")
    except (OSError, ValueError, KeyError, ImportError):
        traffic_note = "profiles/step_kernel_traffic.json not readable"
    roofline = {"bound": "hbm", "kernel": "dexsim::step_tma_kernel<dense, AoS action, auto-reset + counters, 2 stages, dynamic tiles, alternating walk>",
                "achieved": achieved,
                "peak": peak, "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_steady_state": traffic_steady, "traffic_note": traffic_note,
                "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_ENV_STEP, "envs_per_launch": E,
                "kernel_ms": k_ms, "how": "timed-region average per launch (includes auto-reset waves and 1 curriculum poll per 100 steps)",
                "frac_sustained": ALGO_BYTES_PER_ENV_STEP * E / (k_ms_sus * 1e-3) / 1e9 / peak, "kernel_ms_sustained": k_ms_sus,
                "sustained_steps": sus_steps}

    dx.distributed.allreduce_counters(env.counters, env.ret_sums)       # after the last poll of the curriculum driver

    # ---- the same loop with full per-env episode tracking (returns + history summaries -> failure labels) ----
    tracking_full = None
    if not args.no_tracking_variant:
        env_t, _, drv_t = make_env(E, gid0=rank * E, track=True)
        t_steps = max(250, args.steps // 4)
        ms_t, _ = timed_api(env_t, drv_t, pool, t_steps, max(args.warmup, 3), args.poll_every)
        tracking_full = {"value": E * n_gpus * t_steps / (ms_t * 1e-3), "ms_per_step": ms_t / t_steps, "steps": t_steps,
                         "roofline_frac": ALGO_BYTES_PER_ENV_STEP * E / (ms_t / t_steps * 1e-3) / 1e9 / peak,
                         "note": "track_episodes=True: +32 B/env-step of per-env return / history traffic that the "
                                 "410 B algorithmic figure does not count"}
        del env_t, drv_t

    # ---- configs[0] through the drop-in: ONE env behind the reference's Gymnasium API (NumPy action in, NumPy
    #      observation / Python scalars / info dict out), heuristic-style host policy, dense reward, 200-step episodes ----
    single_env = None
    if rank == 0:
        import numpy as np
        env1 = dx.BatchedManipulationEnv(1, dev, reward_type="dense", max_episode_steps=MAX_EPISODE_STEPS, respawn=True)
        rng1 = np.random.default_rng(SEED)
        obs1, _ = env1.reset(seed=SEED)
        def host_policy(_obs):                        # policies/heuristic_policy.py:55-62 in spirit: close + jitter
            return np.clip(-0.5 + rng1.uniform(-1.0, 1.0, 15) * 0.1, -1.0, 1.0).astype(np.float32)
        def run_steps(k):
            nonlocal obs1
            for _ in range(k):
                obs1, r1, te1, tr1, _info = env1.step(host_policy(obs1))
                if te1 or tr1:
                    obs1, _ = env1.reset()            # fresh spawn (respawn=True), like a new env object per episode
        run_steps(300)
        n1 = 3000
        t0 = time.perf_counter()
        run_steps(n1)
        dt1 = time.perf_counter() - t0
        single_env = {"value": n1 / dt1, "unit": UNIT, "us_per_step": 1e6 * dt1 / n1, "env_steps": n1,
                      "note": "num_envs=1 drop-in under the reference's reset/step API incl. the host policy and resets "
                              "(dexsim_step_single: one launch per step, mapped host buffers)"}
        del env1

    # ---- CombinedNoiseWrapper.step (evaluation/robustness_tests.py:177-207) in API mode: both noises drawn inside the
    #      step kernel (60 Philox / Box-Muller normals per env-step) -- bound by instruction issue, not by HBM ----------
    noisy_api = None
    if not args.no_tracking_variant:
        env_n = dx.BatchedManipulationEnv(E, dev, max_episode_steps=MAX_EPISODE_STEPS, reward_type="dense", seed=SEED,
                                          curriculum_config=CC.hard(), observation_noise_std=0.05, dynamics_noise_std=0.1,
                                          env_gid0=rank * E)
        env_n.reset(seed=SEED)
        for t in range(10):
            env_n.step(pool[t % len(pool)])
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_steps = 100
        e0.record()
        for t in range(n_steps):
            env_n.step(pool[t % len(pool)])
        e1.record()
        barrier()
        ms_n = e0.elapsed_time(e1)
        if world > 1:
            tms = torch.tensor([ms_n], device=dev, dtype=torch.float64)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms_n = float(tms.item())
        noisy_api = {"value": E * n_gpus * n_steps / (ms_n * 1e-3), "unit": UNIT, "us_per_step": 1e3 * ms_n / n_steps, "steps": n_steps,
                     "sigma_obs": 0.05, "sigma_dyn": 0.1, "kernel": "dexsim::step_tma_kernel<..., EXTRA>",
                     "bound": "instruction issue (60 normals per env-step: 15 Philox blocks, 30 log/sqrt, 60 sin/cos); "
                              "+180 B/env-step of noisy-observation rows written beside the state",
                     "hbm_frac_of_measured_peak": (ALGO_BYTES_PER_ENV_STEP + 180) * E / (ms_n / n_steps * 1e-3) / 1e9 / peak}
        del env_n

    # ---- end to end: pinned host actions in, obs / reward / flags out ------------------------------
    h_pool = [torch.rand(E, 15).mul_(2).sub_(1).pin_memory() for _ in range(2)]

    def timed_e2e(call, steps):
        for t in range(3):
            call(t)
        env.host_sync()
        barrier()
        t0 = time.perf_counter()
        for t in range(steps):
            call(t)
        env.host_sync()
        barrier()
        sec = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([sec], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            sec = float(tt.item())
        return sec

    # (1) what a caller with a host-side policy does: every call returns with the complete results in host memory.
    #     Transport of the default call: the five 0/1 contact columns travel as their 1-byte mask and are expanded into the
    #     pinned observation by the calling thread while the other rows are still being downloaded.
    e2e_s = timed_e2e(lambda t: env.step_host(h_pool[t % 2]), args.e2e_steps)
    # (2) two result slots, no synchronisation between steps (observation-independent policy, or two env groups taking
    #     turns): the upload of step t+1 overlaps the download of step t; all 41 rows travel
    e2e_async_s = timed_e2e(lambda t: env.step_host(h_pool[t % 2], sync=False, slot=t % 2), args.e2e_steps)
    # (3) as (1) without the host-side expansion (the caller reads info["contact_mask"] or expands on demand)
    e2e_packed_s = timed_e2e(lambda t: env.step_host(h_pool[t % 2], packed_contacts=True), args.e2e_steps)
    # (4) as (1) with all 41 observation rows crossing PCIe (round 1's transport)
    env.host_expand_contacts = env.host_static_rows = False
    e2e_full_s = timed_e2e(lambda t: env.step_host(h_pool[t % 2]), args.e2e_steps)
    env.host_expand_contacts = env.host_static_rows = True
    # the ceiling: the same bytes per step in both directions at once, no kernels (tools/pcie_ceiling.py)
    ceiling = None
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import pcie_ceiling
        cm = pcie_ceiling.measure(E, steps=max(10, args.e2e_steps // 2), device=dev, barrier=barrier, rows=32, extra_bytes_per_env=8)
        csec = cm["seconds_per_step"]
        if world > 1:
            tt = torch.tensor([csec], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            csec = float(tt.item())
        ceiling = {"value": E * n_gpus / csec, "seconds_per_step": csec, "h2d_gbs_per_gpu": cm["h2d_gbs"], "d2h_gbs_per_gpu": cm["d2h_gbs"],
                   "how": "tools/pcie_ceiling.py: this step's H2D and D2H bytes (32 observation rows, reward, flags, contact mask) copied "
                          "concurrently from / to pinned memory on two streams by every rank at once, no kernels; max over ranks"}
    except Exception as exc:       # the ceiling is context for e2e, never a reason to lose the line
        ceiling = {"value": None, "how": f"failed: {exc!r}"}
    e2e_value = E * n_gpus * args.e2e_steps / e2e_s
    d2h_bytes = (env.ld * 32 * 4 + E * (4 + 3 + 1)) * n_gpus
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": E * 15 * 4 * n_gpus,
           "d2h_bytes_per_step": d2h_bytes, "steps": args.e2e_steps,
           "note": "synchronous step_host(), complete [n,45] observation in pinned host memory on return: 32 observation rows + reward + "
                   "flags + the 1-byte contact mask cross PCIe every step (the constant quaternion rows are never re-copied; the five 0/1 "
                   "contact rows are written by the calling thread from the masks while the download is still running; object x, y and "
                   "their velocities only change at a reset and are mirrored into the pinned buffer by the step kernel); 8 chunks, "
                   "H2D / kernel / D2H overlapped",
           "api": "BatchedManipulationEnv.step_host -> dexsim_step_host", "gpu_launches": args.e2e_steps * max(1, min(8, E // 8192)),
           "numa_bound": bool(numa_bound),
           "copy_ceiling": ceiling,
           "frac_of_copy_ceiling": (e2e_value / ceiling["value"]) if ceiling and ceiling.get("value") else None,
           "all_rows_value": E * n_gpus * args.e2e_steps / e2e_full_s,
           "all_rows_d2h_bytes_per_step": (env.ld * 41 * 4 + E * (4 + 3)) * n_gpus,
           "async_value": E * n_gpus * args.e2e_steps / e2e_async_s,
           "async_note": "step_host(sync=False, slot=t%2): two pinned result slots, one host_sync() at the end; every step still "
                         "uploads its actions and downloads all 41 rows",
           "packed_contacts_value": E * n_gpus * args.e2e_steps / e2e_packed_s,
           "packed_contacts_note": "as `value` without the host-side expansion of the contact rows (info['contact_mask'] instead)"}

    # ---- fused rollout (policy in-kernel, K steps per launch) ---------------------------------------
    fused = None
    if rank == 0 or world > 1:
        env2 = dx.BatchedManipulationEnv(E, dev, max_episode_steps=MAX_EPISODE_STEPS, reward_type="dense",
                                         curriculum_config=CC.hard(), track_episodes=True, seed=SEED, env_gid0=rank * E)
        env2.reset(seed=SEED)
        chunk = 50
        env2.rollout(chunk, policy="random")
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nl = 4
        for _ in range(nl):
            env2.rollout(chunk, policy="random")
        e1.record()
        barrier()
        f_ms = e0.elapsed_time(e1)
        fused = {"value": E * n_gpus * chunk * nl / (f_ms * 1e-3), "unit": UNIT, "steps_per_launch": chunk,
                 "launches": nl, "policy": "random (Philox, in-kernel)", "note": "state in registers across the launch"}
        del env2

    # ---- BASELINE configs[3], the north star's own size: 1,048,576 envs IN TOTAL with config_variable's ranged size /
    #      mass / friction, sharded over the N ranks by global env id (strong scaling; 131,072 envs per GPU at N = 8) ----
    strong = None
    if not args.no_strong:
        strong = run_strong_1m(dx, torch, dist, dev, rank, world, barrier, peak)

    # ---- sweep over env counts: API mode (one launch per step) and the fused rollout (50 steps per
    #      launch); these sizes are L2-resident and launch/latency-bound, see DESIGN.md section 7 ----------
    sweep = []
    if not args.no_sweep and world == 1:
        for n in (4096, 65536, 131072):
            if n == E:
                continue
            env_s, _, drv_s = make_env(n)
            pool_s = action_pool(n)
            s_ms, _ = timed_api(env_s, drv_s, pool_s, 300, 120, 100)
            v = n * 300 / (s_ms * 1e-3)
            # the same API step replayed from a CUDA graph (8 steps per replay over the same four action tensors as the
            # eager loop, so that both see the same working set in L2): removes the host launch path
            buf = pool_s + pool_s
            replay = env_s.capture_step(buf, steps=8)
            for _ in range(10):
                replay()
            torch.cuda.synchronize(dev)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(40):
                replay()
            g1.record()
            torch.cuda.synchronize(dev)
            gv = n * 320 / (g0.elapsed_time(g1) * 1e-3)
            del replay, buf
            env_f = dx.BatchedManipulationEnv(n, dev, max_episode_steps=MAX_EPISODE_STEPS, reward_type="dense",
                                              curriculum_config=CC.hard(), track_episodes=True, seed=SEED)
            env_f.reset(seed=SEED)
            env_f.rollout(50, policy="random")
            torch.cuda.synchronize(dev)
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(8):
                env_f.rollout(50, policy="random")
            f1.record()
            torch.cuda.synchronize(dev)
            fv = n * 400 / (f0.elapsed_time(f1) * 1e-3)
            sweep.append({"envs": n, "value": v, "ms_per_step": s_ms / 300,
                          "roofline_frac": v * ALGO_BYTES_PER_ENV_STEP / 1e9 / peak, "graph_replay_value": gv,
                          "fused_rollout_value": fv,
                          "note": "state is L2-resident at this size: one step is a launch plus one load-compute-store round trip (latency-bound, ~5 us of host issue per step)"})
            del env_s, pool_s, env_f

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32+f64", "data": "synthetic",
            "config": {
                "workload": f"config_default.json dense + curriculum_scheduler(easy->hard), random_policy actions resident in HBM, "
                            f"{E} envs per GPU, auto-reset respawn with per-group episode counters feeding the scheduler, "
                            f"max_episode_steps 200",
                "envs_per_gpu": E, "envs_total": E * n_gpus, "l2": "state + actions per step exceed the 126 MB L2 (no flush needed)"
                if E * ALGO_BYTES_PER_ENV_STEP > 130e6 else "state fits in L2 at this size",
                "curriculum": {"difficulty": sched.current_difficulty_level, "progressions": drv.progressions,
                               "poll_every": args.poll_every, "preroll_steps": args.preroll_steps},
                "parallelism": f"env-sharded dp{n_gpus}, no data-path collective",
            },
            "e2e": e2e, "gpu_launches": launches, "gpu_launches_note": "step_tma_kernel launches inside the main timed region (one per step)",
            "roofline": roofline, "cpu_baseline": cpu_base,
            "tracking_full": tracking_full, "noisy_api": noisy_api, "strong_1m": strong, "single_env_dropin": single_env, "fused_rollout": fused, "sweep": sweep, "clocks": clocks,
            "episodes": int(env.counters[:, 0].sum().item()),
        }
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    os.close(json_fd)
    return 0


def run_strong_1m(dx, torch, dist, dev, rank, world, barrier, peak, n_total=1 << 20):
    """experiments/config_variable.json (BASELINE configs[3]) at a FIXED total of 1,048,576 envs on every GPU count."""
    import hashlib
    CC = dx.CurriculumConfig
    lo, hi = dx.distributed.shard_range(n_total, rank, world)
    m = hi - lo
    cfg = CC(object_size=0.05, object_size_range=(0.03, 0.07), object_mass=0.1, object_mass_range=(0.05, 0.15),
             friction_coefficient=0.5, friction_range=(0.3, 0.7), spawn_distance=0.15, spawn_distance_range=(0.10, 0.20))

    def make(track, auto=True):
        e = dx.BatchedManipulationEnv(m, dev, reward_type="dense", max_episode_steps=MAX_EPISODE_STEPS, curriculum_config=cfg,
                                      auto_reset=auto, respawn=True, loop_max_steps=MAX_EPISODE_STEPS, track_episodes=track,
                                      seed=SEED, env_gid0=lo)
        e.reset(seed=SEED)
        return e

    def max_ms(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def sha(c):
        c = c.clone()
        dx.distributed.allreduce_counters(c)
        return hashlib.sha256(c.cpu().numpy().tobytes()).hexdigest(), c

    # (1) GPU-count independence: counters of a 200-step fused rollout from reset (random policy, Philox keyed by global
    #     env id), all-reduced over the ranks -- the same bytes on 1, 2, 4 and 8 GPUs
    env = make(True, auto=False)
    env.rollout(200, policy="random", zero_counters=True)
    sha_fused, c_all = sha(env.counters)
    # (2) the API path reaches the same table: 40 steps of dexsim_step with the Philox actions the fused kernel draws
    #     (dexsim_fill_policy_actions) against a 40-step fused rollout
    import ctypes as C
    from dexterous_rl_manipulation_b200 import _lib
    env_a, env_f = make(True), make(True, auto=False)
    act = torch.zeros(15, env_a.ld, device=dev)
    for _ in range(40):
        _lib.check(env_a._lib.dexsim_fill_policy_actions(C.byref(env_a._state), C.byref(env_a._params), _lib.POLICY_RANDOM,
                                                         act.data_ptr(), env_a._stream()), "dexsim_fill_policy_actions")
        env_a.step(act[:, :m].t().contiguous())
    env_f.rollout(40, policy="random", zero_counters=True)
    sha_api40, _ = sha(env_a.counters)
    sha_fused40, _ = sha(env_f.counters)
    del env_a, env_f

    # (3) throughput at this size: API mode eager, API mode replayed from a CUDA graph (8 steps per replay), fused rollout
    g = torch.Generator(device=dev).manual_seed(SEED + rank)
    pool = [torch.rand(m, 15, device=dev, generator=g) * 2 - 1 for _ in range(4)]
    env_t = make(False)
    for t in range(50):
        env_t.step(pool[t % 4])
    barrier()
    steps = 400
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(steps):
        env_t.step(pool[t % 4])
    e1.record()
    barrier()
    ms_eager = max_ms(e0.elapsed_time(e1)) / steps
    buf = pool + pool            # the eager loop's four action tensors, twice: same working set in L2
    replay = env_t.capture_step(buf, steps=8)
    for _ in range(10):
        replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        replay()
    e1.record()
    barrier()
    ms_graph = max_ms(e0.elapsed_time(e1)) / 400
    del replay, buf, env_t
    env.rollout(50, policy="random")
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(4):
        env.rollout(50, policy="random")
    e1.record()
    barrier()
    ms_fused = max_ms(e0.elapsed_time(e1)) / 200
    frac = lambda ms: ALGO_BYTES_PER_ENV_STEP * m / (ms * 1e-3) / 1e9 / peak
    eps = int(c_all[:, 0].sum().item())
    return {
        "workload": "experiments/config_variable.json (size 0.03-0.07, mass 0.05-0.15, friction 0.3-0.7 redrawn at every reset), "
                    "dense reward, auto-reset respawn, 200-step episodes", "envs_total": n_total, "envs_per_gpu": m,
        "scaling": "strong", "unit": UNIT,
        "api_eager": {"value": n_total / (ms_eager * 1e-3), "us_per_step": 1e3 * ms_eager, "per_gpu_roofline_frac": frac(ms_eager), "steps": steps},
        "api_graph_replay": {"value": n_total / (ms_graph * 1e-3), "us_per_step": 1e3 * ms_graph, "per_gpu_roofline_frac": frac(ms_graph),
                             "steps_per_replay": 8},
        "fused_rollout": {"value": n_total / (ms_fused * 1e-3), "us_per_step": 1e3 * ms_fused, "steps_per_launch": 50},
        "counters_sha256": sha_fused, "counters_steps": 200, "counters_episodes": eps,
        "counters_note": "sha256 of the all-reduced [G,18] int64 counter table after a 200-step fused rollout from reset; "
                         "Philox is keyed by global env id, so the hash must be identical at N = 1, 2, 4, 8",
        "api_counters_sha256_40": sha_api40, "fused_counters_sha256_40": sha_fused40, "api_equals_fused": sha_api40 == sha_fused40,
        "l2": "state + actions per GPU are L2-resident below ~262,144 envs per GPU: a step is launch / latency-bound there "
              "and the HBM roofline fraction is only a yardstick",
    }


def measure_cpu_baseline(args):
    """cpu_baseline leg: the reference arm on a bounded sample, in a subprocess (never shares the
    CUDA context).  Sized from a 1-step probe to take about --cpu-seconds."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-steps-per-proc", "500"]   # 500 env-steps x P procs per step
    try:
        probe = subprocess.run(cmd + ["--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=180)
        line = json.loads(probe.stdout.strip().splitlines()[-1])
        if "unavailable" in line:
            return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": line["unavailable"]}
        per_step = line["ms_per_step"] * 1e-3
        steps = max(2, min(200, int(args.cpu_seconds / max(per_step, 1e-3))))
        full = subprocess.run(cmd + ["--steps", str(steps), "--warmup", "1"], capture_output=True, text=True, timeout=600)
        line = json.loads(full.stdout.strip().splitlines()[-1])
        base = line["cpu_baseline"]
        # BASELINE.md section 3: also the single-core figure (one process, same loop), a few seconds
        one = subprocess.run(cmd + ["--steps", "8", "--warmup", "1", "--ref-procs", "1"], capture_output=True, text=True, timeout=300)
        try:
            base["one_core_value"] = json.loads(one.stdout.strip().splitlines()[-1])["value"]
        except (ValueError, IndexError, KeyError):
            base["one_core_value"] = None
        return base
    except Exception as exc:       # report, never fake a number
        return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {exc!r}"}


def main():
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, max(args.gpus, world))
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
