#!/usr/bin/env python
"""bench.py -- control env-steps/s of the batched Go1+PEA step path on B200.

    python bench.py --gpus N --steps K --warmup W [--config {2,3,4,5}] [--dump-outputs DIR]     (ours; N>1 under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W [--config ...]

One "step" = one control step (action_repeat = 10 physics ticks + task/obs epilogue, finished envs
re-settled in place) of every env of the job.  `--config` picks one of BASELINE.json's GPU configurations
(numbered as in SURVEY.md 8d; the default, 3, is the one the metric is quoted on):

  2  configs[1]  Go1 without springs, JUMPING_IN_PLACE, joint PD, 4096 envs, random actions
  3  configs[2]  Go1 + PEA, JUMPING_FORWARD, CARTESIAN_PD (IK -> joint PD), 65536 envs per GPU, random actions
  4  configs[3]  Go1 + PEA driven by the Hopf CPG (hopf_network.py __main__: TORQUE mode, action_repeat = 1),
                 65536 envs per GPU; a bench step = 10 CPG + physics ticks (one 10 ms control period)
  5  configs[4]  Go1 + PEA, BACKFLIP with the backflip landing controller, SB3-shaped MlpPolicy (2 x 64 tanh) +
                 VecNormalize evaluated on the device every step, 32768 envs per GPU (262144 over 8)

Envs are independent, so N GPUs run N shards with no data-path collective ("weak" scaling); NCCL is used for the
timing barrier / max-over-ranks and for the all-gather of rollout statistics.

Steady state: the metric includes the resets (BASELINE.md section 3), and reset()'s 2500-tick settle of the next
episodes is spread over the steps by the settle conveyor.  Right after reset() every env is in phase and its ring
of settled episodes is full, so the first steps do almost no settle work.  Whatever --warmup says, the timed
region therefore only starts after an untimed PRE-ROLL has brought the episode ends and the conveyor to their
stationary rates (`steady_state` in the JSON line says how that was judged).

The reference arm times the CPU restatement of the reference path (the oracle, kind "port": the reference itself
needs pybullet, which is neither vendored nor installable here or on the GPU box, profiles/r02_pybullet_probe.log)
on all host cores, one process per core.
"""
import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree, which may be read-only

CONFIGS = {
    2: dict(name="go1_nosprings_jumping_in_place_pd_4096env", kind="random", envs_per_gpu=4096,
            env=dict(enable_springs=False, task_env="JUMPING_IN_PLACE", motor_control_mode="PD",
                     action_space_mode="SYMMETRIC", observation_space_mode="ARS_BASIC")),
    3: dict(name="go1_pea_jumping_forward_cartesian_pd_65536env_per_gpu", kind="random", envs_per_gpu=65536,
            env=dict(enable_springs=True, task_env="JUMPING_FORWARD", motor_control_mode="CARTESIAN_PD",
                     action_space_mode="SYMMETRIC", observation_space_mode="ARS_BASIC")),
    4: dict(name="go1_pea_hopf_cpg_torque_65536env_per_gpu", kind="cpg", envs_per_gpu=65536,
            env=dict(enable_springs=True, isRLGymInterface=False, action_repeat=1, motor_control_mode="TORQUE"),
            cpg=dict(gait="TROT", omega_swing=16 * 3.141592653589793, omega_stance=4 * 3.141592653589793)),
    5: dict(name="go1_pea_backflip_ppo_policy_32768env_per_gpu", kind="policy", envs_per_gpu=32768,
            env=dict(enable_springs=True, task_env="BACKFLIP_PPO", motor_control_mode="PD", action_space_mode="SYMMETRIC",
                     observation_space_mode="PPO_BACKFLIP", landing_wrapper="LandingWrapperBackflip")),
}
METRIC = "control_env_steps_per_sec"
UNIT = "env-steps/s"
SM_COUNT, FP32_LANES = 148, 128


# ----------------------------------------------------------------------------- CPU arm (oracle port)
def _cpu_worker(args):
    seed, budget_s, max_steps, cfg_id = args
    import numpy as np
    from oracle import oracle as O
    cfg = CONFIGS[cfg_id]
    rng = np.random.default_rng(seed)
    if cfg["kind"] == "cpg":
        return _cpu_worker_cpg(cfg, rng, budget_s, max_steps)
    kw = {k: v for k, v in cfg["env"].items() if k != "landing_wrapper"}
    if "landing_wrapper" in cfg["env"]:
        kw["landing_mode"] = {"LandingWrapper": 1, "LandingWrapper2": 2, "LandingWrapperContinuous": 3,
                              "LandingWrapperBackflip": 4, "LandingWrapperBackflip2": 5}[cfg["env"]["landing_wrapper"]]
    env = O.Env(enable_limits=1, body_contact_response=1, **kw)
    policy = None
    if cfg["kind"] == "policy":   # the same MlpPolicy arithmetic in numpy (2 x 64 tanh, DiagGaussian sample, clip)
        pr = np.random.default_rng(7)
        od, ad = env.obs_dim, env.action_dim
        W = [pr.standard_normal((od, 64)) / np.sqrt(od), pr.standard_normal((64, 64)) / 8.0, pr.standard_normal((64, ad)) / 8.0]
        policy = lambda o: np.clip(np.tanh(np.tanh(o @ W[0]) @ W[1]) @ W[2] + rng.standard_normal(ad), -1, 1)
    t_reset = time.perf_counter()
    o = env.reset(mu=0.5 + 0.5 * rng.random())
    t_reset = time.perf_counter() - t_reset
    steps = resets = 0
    t0 = time.perf_counter()
    while steps < max_steps and time.perf_counter() - t0 < budget_s:
        a = policy(np.clip(o, -10, 10)) if policy else rng.uniform(-1, 1, env.action_dim)
        o, r, d, tr = env.step(a)
        steps += 1
        if d:
            o = env.reset(mu=0.5 + 0.5 * rng.random())
            resets += 1
    return steps, time.perf_counter() - t0, resets, t_reset


def _cpu_worker_cpg(cfg, rng, budget_s, max_steps):
    """hopf_network.py:241-289 on the oracle: per 1 ms tick cpg_step -> cpg_torque -> env.step (TORQUE mode,
    action_repeat = 1); ten ticks count as one control-step equivalent"""
    import numpy as np
    from oracle import oracle as O
    env = O.Env(enable_limits=1, body_contact_response=1, **cfg["env"])
    t_reset = time.perf_counter()
    env.reset(mu=0.5 + 0.5 * rng.random())
    t_reset = time.perf_counter() - t_reset
    pi = np.pi
    PHI = np.array({"BOUND": [[0, 0, -pi, -pi], [0, 0, -pi, -pi], [pi, pi, 0, 0], [pi, pi, 0, 0]],
                    "TROT": [[0, -pi, -pi, 0], [pi, 0, 0, pi], [pi, 0, 0, pi], [0, -pi, -pi, 0]]}[cfg["cpg"]["gait"]], dtype=np.float64)
    X = np.zeros((2, 4))
    X[0] = rng.random(4) * 0.1
    X[1] = PHI[0]
    ticks = resets = 0
    t0 = time.perf_counter()
    while ticks < 10 * max_steps and time.perf_counter() - t0 < budget_s:
        X, xs, zs = O.cpg_step(X, PHI, 2.0, cfg["cpg"]["omega_swing"], cfg["cpg"]["omega_stance"], 1.0, 0.001, 0.04, 0.25, 0.05, 0.01)
        st = env.world.get_state()
        q, qd = st[13:25], st[25:37]
        tau = O.cpg_torque(xs, zs, q, qd, 0.0838, (150, 70, 70), (2, 0.5, 0.5), 2500.0, 40.0, True)
        o, r, d, tr = env.step(tau)
        ticks += 1
        if d:
            env.reset(mu=0.5 + 0.5 * rng.random())
            resets += 1
    return ticks // 10, time.perf_counter() - t0, resets, t_reset


def cpu_sample(budget_s, cfg_id, max_steps=10**9, procs=None, seed0=0):
    """P processes (one per host core) each stepping the oracle env; returns aggregate env-steps/s"""
    from oracle import oracle as O
    O.build()
    procs = procs or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs) as pool:
        res = pool.map(_cpu_worker, [(seed0 + i, budget_s, max_steps, cfg_id) for i in range(procs)])
    steps = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    return dict(value=steps / wall, steps=steps, wall_s=wall, cores=procs, resets=sum(r[2] for r in res),
                reset_s=statistics.mean(r[3] for r in res))


def cpu_baseline_dict(s, seconds):
    return {"value": s["value"], "unit": UNIT, "cores": s["cores"], "kind": "port",
            "per_core_value": s["value"] / s["cores"], "reset_s": s["reset_s"], "resets": s["resets"], "env_steps": s["steps"],
            "sample": f"{s['cores']} processes x {seconds:.1f} s of the oracle env (C port of the reference path, fp64, "
                      f"general solver on) on the same workload, one env per process, re-reset (settle included) on done"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    per_step_budget = min(8.0, 150.0 / max(args.steps + args.warmup, 1))
    for _ in range(args.warmup):
        cpu_sample(min(per_step_budget, 2.0), args.config)
    agg = dict(steps=0, wall_s=0.0, cores=0, resets=0, reset_s=0.0)
    for i in range(args.steps):
        s = cpu_sample(per_step_budget, args.config, seed0=1000 * (i + 1))
        agg["steps"] += s["steps"]; agg["wall_s"] += s["wall_s"]; agg["cores"] = s["cores"]; agg["resets"] += s["resets"]
        agg["reset_s"] += s["reset_s"] / max(args.steps, 1)
    agg["value"] = agg["steps"] / max(agg["wall_s"], 1e-9)
    value = agg["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * agg["wall_s"] / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["name"], **cfg["env"], "envs": agg["cores"], "host": "cpu"},
        "cpu_baseline": cpu_baseline_dict(agg, per_step_budget),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """SM clock, power and throttle reasons sampled DURING the timed region.  In-process NVML (the library nvidia-smi
    itself reads): forking an nvidia-smi every 200 ms stalled the kernels of the next 3 steps by ~1 ms each, which is
    9 % of a 20-step window (round-2 measurement, DESIGN.md section 5); `nvidia-smi` is only the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt, self.period = index, [], threading.Event(), period
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.nvml = pynvml
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self._sample_nvml()      # first call paths warmed up outside the timed region
            self.samples.clear()
        except Exception:
            self.nvml = None
            self.period = 0.2

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].isdigit():
                return int(ids[index])
        return index

    def _sample_nvml(self):
        nv, h = self.nvml, self.handle
        sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        try:
            reasons = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            reasons = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        try:
            power = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            power = float("nan")
        bits = [nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap]
        self.samples.append([sm, self.sm_max, power] + [bool(reasons & b) for b in bits])

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in out.strip().split(",")]
        if len(f) >= 7:
            self.samples.append([float(f[0]), float(f[1]), float(f[2])] + [x.lower().startswith("active") for x in f[3:7]])

    def run(self):
        while not self._halt.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"]}
        reasons = [n for i, n in enumerate(self.NAMES) if any(s[3 + i] for s in self.samples)]
        pw = [s[2] for s in self.samples if s[2] == s[2]]
        return {"sm_mhz": statistics.median(s[0] for s in self.samples), "sm_max_mhz": self.samples[0][1],
                "power_w_max": max(pw) if pw else None, "samples": len(self.samples), "reasons": reasons,
                "source": "NVML in-process, every 20 ms" if self.nvml else "nvidia-smi every 200 ms"}


# ----------------------------------------------------------------------------- ours
class Job:
    """One shard of a BASELINE configuration: the env plus whatever drives it (random actions, the CPG, a policy)."""

    def __init__(self, cfg, n, dev, rank, seed):
        import torch
        import quadruped_springs_b200 as qs
        self.cfg, self.n, self.dev, self.kind = cfg, n, dev, cfg["kind"]
        self.torch = torch
        self.env = qs.BatchedQuadrupedGymEnv(num_envs=n, device=dev, seed=seed, env_id_offset=rank * n, auto_reset=True,
                                             enable_noise=True, **cfg["env"])
        self.A, self.O = self.env.action_dim, self.env.obs_dim
        self.gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        self.episodes_seen = 0
        self.obs = self.env.reset()
        if self.kind == "cpg":
            self.cpg = qs.HopfNetwork(num_envs=n, device=dev, time_step=0.001, seed=rank, **cfg["cpg"])
        if self.kind == "policy":
            torch.manual_seed(7)
            self.policy = qs.MlpPolicyTorch(self.O, self.A).to(dev)
            venv = qs.BatchedVecEnv(env=self.env)
            self.vn = qs.VecNormalizeTorch(venv, training=False, norm_reward=False)   # load_model.py:114-116

    def next_input(self):
        """what is resident in HBM before the timed region of a step starts"""
        if self.kind == "random":   # fixed-seed uniform(-1, 1) actions, a new draw for every env and step
            return (self.torch.rand(self.n, self.A, device=self.dev, generator=self.gen) * 2 - 1).contiguous()
        return None

    def step(self, inp):
        """one bench step; returns what the env hands its caller: (obs, reward, done, infos), views of the env's buffers"""
        env = self.env
        if self.kind == "random":
            return env.step(inp)
        if self.kind == "cpg":      # hopf_network.py:241-289, ten 1 ms ticks: qs_cpg_steps
            return self.cpg.drive(env, 10)
        # load_model.py:127-134 with the policy on the device (stochastic, as in PPO rollouts)
        a = self.policy.predict(self.vn.normalize_obs(self.obs), deterministic=False, generator=self.gen)
        out = env.step(a)
        self.obs = out[0]
        return out

    def take_done_count(self):
        """episodes finished since the last call (the env's own rollout statistics, kernel K5)"""
        total = int(round(float(self.env.rollout_stats()[1].item())))
        v = total - self.episodes_seen
        self.episodes_seen = total
        return v


def preroll(job, L, lib, max_steps, world, dist, dev, min_steps=150):
    """Untimed steps until the episode ends and the settle conveyor are stationary: at least 150 steps, then chunks of 25
    until (a) the reset rate of a chunk is within tol of the previous chunk's and (b) the settle ticks the conveyor ran
    in the chunk are within 10 % of resets x settle length (every finished episode is paid for by one settle).
    tol = max(2 %, 3 / sqrt(resets in the chunk)): the 2 % the rates must agree to, widened by the counting noise
    of small jobs.  All ranks stop together (the slowest decides)."""
    import torch
    env = job.env
    nsettle = 2500 if job.cfg["env"].get("isRLGymInterface", True) else 1500
    sw = (C.c_uint64 * 3)()
    lib.check(L.qs_settle_work_counters(env._h, sw, None))
    prev_ticks, prev_rate, steps, ok = int(sw[0]), None, 0, False
    info = {}
    chunk = 25
    job.take_done_count()
    while steps < max_steps:
        for _ in range(chunk):
            job.step(job.next_input())
        steps += chunk
        resets = job.take_done_count()
        lib.check(L.qs_settle_work_counters(env._h, sw, None))
        ticks = int(sw[0]) - prev_ticks
        prev_ticks = int(sw[0])
        rate = resets / chunk
        tol = max(0.02, 3.0 / max(resets, 1) ** 0.5)
        paid = ticks / max(resets * nsettle, 1)
        stationary = prev_rate is not None and abs(rate - prev_rate) <= tol * max(rate, prev_rate, 1e-9) and abs(paid - 1.0) <= 0.10
        if resets < 30 and steps >= min_steps:
            stationary = True    # (almost) no episode ends: nothing to wait for; counting noise would never let two chunks agree
        prev_rate = rate
        info = {"preroll_steps": steps, "resets_per_step": rate, "settle_ticks_per_step": ticks / chunk,
                "settle_ticks_per_reset": ticks / max(resets, 1), "rate_tolerance": tol}
        flag = torch.tensor([1.0 if (stationary and steps >= min_steps) else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() > 0:
            ok = True
            break
    info["converged"] = ok
    return info


DUMP_BYTES = 64 * 10**6    # all .npy files of --dump-outputs together
DUMP_NAMES = {"TimeLimit.truncated": "truncated"}


def dump_outputs(out_dir, outputs, seed=0):
    """Writes what one step returned to its caller (obs, reward, done and the infos tensors) as out_dir/<name>.npy in float32,
    one row per env.  If all rows exceed DUMP_BYTES, a fixed seeded sample of env rows is written instead, the same rows in
    every array, and their indices go to env_index.npy (float64)."""
    import numpy as np
    import torch
    o, r, d, infos = outputs
    arrays = {"obs": o, "reward": r, "done": d, **{DUMP_NAMES.get(k, k): v for k, v in infos.items()}}
    n = o.shape[0]
    row_bytes = sum(4 * a[0].numel() for a in arrays.values())
    budget = DUMP_BYTES - 128 * (len(arrays) + 1)      # .npy headers
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(seed).choice(n, budget // (row_bytes + 8), replace=False))
        idx = torch.as_tensor(rows, device=o.device)
        arrays = {k: v.index_select(0, idx) for k, v in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        a = v if isinstance(v, np.ndarray) else v.detach().to(torch.float32).cpu().numpy()
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from quadruped_springs_b200 import _lib, stats

    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.envs_per_gpu or cfg["envs_per_gpu"]
    L = _lib.lib()
    job = Job(cfg, n, dev, rank, args.seed)
    env, A, O = job.env, job.A, job.O
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- untimed: pre-roll to the stationary regime, then the caller's warm-up
    steady = preroll(job, L, _lib, args.max_preroll, world, dist, dev, args.min_preroll)
    for i in range(args.warmup):
        job.step(job.next_input())
    barrier()
    job.take_done_count()

    # ---------------- device-resident timing ("value")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    work0, swork0 = (C.c_uint64 * 3)(), (C.c_uint64 * 3)()
    _lib.check(L.qs_work_counters(env._h, work0, None))
    _lib.check(L.qs_settle_work_counters(env._h, swork0, None))
    dbg = (C.c_int32 * 4)()
    launches0 = L.qs_launch_count()
    nsteps0 = L.qs_step_count(env._h)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    urgent = 0
    # the pre-roll's length follows the computed reset counts: reseeding here keeps the timed steps' random draws the same
    # for builds whose rounding differs, so that their --dump-outputs can be compared
    job.gen.manual_seed(4321 + rank)
    barrier()
    t_wall = time.perf_counter()
    host_s = 0.0
    for i in range(args.steps):
        flush.fill_(float(i))          # L2 flush between timed iterations (outside the event pair)
        a = job.next_input()           # inputs resident in HBM before the timed region of the step starts
        ev[i][0].record()
        th = time.perf_counter()
        last = job.step(a)
        host_s += time.perf_counter() - th
        ev[i][1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    launches = L.qs_launch_count() - launches0
    env_calls = int(L.qs_step_count(env._h) - nsteps0)      # qs_step calls in the timed region (10 per bench step for the CPG)
    resets_timed = job.take_done_count()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    kms = C.c_float()
    kk = min(env_calls, int(L.qs_timing_window(env._h)))
    _lib.check(L.qs_step_kernel_time(env._h, kk, C.byref(kms)))
    k_step_ms = kms.value / kk * (env_calls / args.steps)
    _lib.check(L.qs_settle_kernel_time(env._h, kk, C.byref(kms)))
    k_settle_ms = kms.value / kk * (env_calls / args.steps)
    _lib.check(L.qs_slow_kernel_time(env._h, kk, C.byref(kms)))
    k_slow_ms = kms.value / kk * (env_calls / args.steps)
    work1, swork1 = (C.c_uint64 * 3)(), (C.c_uint64 * 3)()
    _lib.check(L.qs_work_counters(env._h, work1, None))
    _lib.check(L.qs_settle_work_counters(env._h, swork1, None))
    _lib.check(L.qs_debug_counters(env._h, dbg, None))
    urgent = int(dbg[1])
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:     # before the e2e steps below overwrite the env's buffers
        dump_outputs(args.dump_outputs, last)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    ms_per_step = dev_ms_max / args.steps
    value = world * n * args.steps / (dev_ms_max * 1e-3)

    # ---------------- end-to-end through the host-buffer path ("e2e")
    e2e_steps = max(min(args.steps, 200), 5)
    h_out = (torch.empty(n, O, dtype=torch.float32).pin_memory(), torch.empty(n, dtype=torch.float32).pin_memory(),
             torch.empty(n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory())
    np_out = tuple(x.numpy() for x in h_out)
    if job.kind == "random":
        n_act = 16
        h_act = [torch.empty(n, A, dtype=torch.float32).pin_memory() for _ in range(n_act)]
        for i in range(n_act):
            h_act[i].copy_(job.next_input())
        np_act = [a.numpy() for a in h_act]

        def e2e_step(i):   # H2D actions, step(+resets), D2H obs/reward/done/truncated, stream sync: one C-ABI call
            env.step_host(np_act[i % n_act], np_out)
        h2d, d2h = n * A * 4, n * (O * 4 + 4 + 2)
        path = ("qs_step_host: pinned host actions -> H2D -> step kernels + settle slices -> D2H obs, reward, done, "
                "truncated -> stream sync")
    elif job.kind == "cpg":
        def e2e_step(i):   # the CPG has no per-step host input; a host consumer reads the results once per control period
            job.step(None)
            h_out[0].copy_(env._obs, non_blocking=True); h_out[1].copy_(env._reward, non_blocking=True)
            h_out[2].copy_(env._done, non_blocking=True); h_out[3].copy_(env._trunc, non_blocking=True)
            torch.cuda.synchronize(dev)
        h2d, d2h = 0, n * (O * 4 + 4 + 2)
        path = ("10 x (qs_cpg_update + qs_step) on the device, then D2H obs, reward, done, truncated of the control period "
                "-> sync (the CPG is autonomous: no per-step host input)")
    else:
        h_obs = torch.empty(n, O, dtype=torch.float32).pin_memory()
        h_obs.copy_(job.obs)
        d_obs = torch.empty(n, O, device=dev)

        def e2e_step(i):   # host observation -> device -> VecNormalize + policy -> step -> results back to the host
            d_obs.copy_(h_obs, non_blocking=True)
            a = job.policy.predict(job.vn.normalize_obs(d_obs), deterministic=False, generator=job.gen)
            o, r, d, _ = env.step(a)
            h_obs.copy_(o, non_blocking=True); h_out[1].copy_(r, non_blocking=True)
            h_out[2].copy_(env._done, non_blocking=True); h_out[3].copy_(env._trunc, non_blocking=True)
            torch.cuda.synchronize(dev)
        h2d, d2h = n * O * 4, n * (O * 4 + 4 + 2)
        path = ("pinned host obs -> H2D -> VecNormalize + MlpPolicy (torch, device) -> qs_step -> D2H obs, reward, done, "
                "truncated -> sync")
    for i in range(2):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * e2e_steps / float(t.item())

    # ---------------- rollout statistics: the only exchange of the path (one all-gather of 16 floats per shard)
    rollout = stats.gather_rollout_stats(env.rollout_stats())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline, FP32 pipe: the settle slices (dominant by time) and the step kernels
    fm = json.load(open(os.path.join(ROOT, "quadruped_springs_b200", "flop_model.json")))

    def tick_flops(w0, w1):
        ticks, cticks, csweeps = (int(w1[i] - w0[i]) for i in range(3))
        f = (ticks * fm["W0_flight_tick"] + cticks * (fm["W_per_contact"] + fm["W_any_contact"] / 4.0)
             + csweeps * fm["W_per_contact_sweep"])
        return f, ticks, cticks, csweeps

    step_flops, ticks, cticks, csweeps = tick_flops(work0, work1)
    step_flops += n * env_calls * fm["epilogue_per_control_step_estimate"]
    settle_flops, sticks, scticks, scsweeps = tick_flops(swork0, swork1)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sm_mhz_max = float(peaks.get("sm_max_mhz", 1965.0))
    fp32_peak = SM_COUNT * FP32_LANES * 2 * sm_mhz_max * 1e6 / 1e12     # TFLOP/s, non-tensor FP32 FMA
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    state_bytes = n * 4 * (2 * (37 + 12 + 12 + 4 + 1 + 29 + 12 + 3 + 3) + 24 + 9 + 1 + A + O + 2) * (env_calls / args.steps)

    def fp32_line(kernel, flops, ms, extra):
        ach = flops / args.steps / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        return {"bound": "fp32", "kernel": kernel, "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s",
                "frac": ach / fp32_peak, "kernel_ms": ms, "kernel_share_of_step": ms / ms_per_step, **extra}

    settle_line = fp32_line("k_settle_slice", settle_flops, k_settle_ms, {
        "what": "reset()'s settle of the next episodes: two slices of ticks per control step on a second stream (timed there "
                "with CUDA events; the early one runs next to k_step_contact, the late one next to k_step_slow); achieved = "
                "flops of both launches / their summed duration",
        "launches_per_step": 2 * env_calls / args.steps,
        "settle_ticks_per_step": sticks / args.steps, "algorithmic_flops_per_settle_tick": settle_flops / max(sticks, 1),
        "mean_foot_contacts_per_tick": scticks / max(sticks, 1), "mean_pgs_sweeps_per_contact_tick": scsweeps / max(scticks, 1)})
    step_line = fp32_line("k_step + k_step_contact", step_flops, k_step_ms, {
        "what": "the physics ticks of step(): k_pre, the flight variant, then the envs with foot contacts (the general-solver "
                "launch k_step_slow is timed apart: k_step_slow_ms; the epilogue kernel k_finish runs next to k_step_slow as a "
                "programmatic dependent launch and is not in this interval)",
        "algorithmic_flops_per_env_step": step_flops / args.steps / n,
        "mean_foot_contacts_per_tick": cticks / max(ticks, 1), "mean_pgs_sweeps_per_contact_tick": csweeps / max(cticks, 1),
        "hbm": {"algorithmic_bytes_per_step": state_bytes, "achieved_GBps": state_bytes / (max(k_step_ms, 1e-9) * 1e-3) / 1e9,
                "peak_GBps": hbm_peak, "frac": state_bytes / (max(k_step_ms, 1e-9) * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s"}})
    dominant, other = (settle_line, step_line) if k_settle_ms >= k_step_ms else (step_line, settle_line)
    roofline = dict(dominant)
    roofline["traffic"] = None
    roofline["traffic_source"] = None
    roofline["peak_source"] = (f"{SM_COUNT} SMs x {FP32_LANES} FP32 lanes x 2 x {sm_mhz_max:.0f} MHz (clocks.max.sm from "
                               f"{'MEASURED_PEAKS.json' if peaks else 'nominal'}); no tensor cores: per-env matrices <= 6x6")
    roofline["other_kernels"] = [other]
    roofline["k_step_slow_ms"] = k_slow_ms
    ncu_path = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    if os.path.exists(ncu_path) and args.config == 3:
        try:
            ent = json.load(open(ncu_path)).get(dominant["kernel"], {})
            roofline["traffic"] = ent.get("dram_bytes_per_launch")
            roofline["traffic_source"] = ("constant from a committed ncu --set full capture of this workload, NOT measured in "
                                          "this run: " + str(ent.get("source")))
        except Exception:
            pass
    tot_flops = settle_flops + step_flops
    steady = dict(steady)
    steady.update({
        "timed_resets_per_step": resets_timed / args.steps, "timed_settle_ticks_per_step": sticks / args.steps,
        "timed_settle_ticks_per_reset": sticks / max(resets_timed, 1), "urgent_settles_last_step": urgent,
        "settle_share_of_flops": settle_flops / max(tot_flops, 1.0),
        "note": "settle_share_of_flops of the timed region is reset() work (2500 settle ticks per finished episode), not "
                "step() physics: under random actions episodes are short, so the metric mostly measures k_settle_slice"})

    # ---------------- CPU baseline beside it (rank 0, N = 1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_dict(cpu_sample(args.cpu_seconds, args.config), args.cpu_seconds)

    conf = {"workload": cfg["name"], **cfg["env"], "envs_per_gpu": n, "envs_total": world * n,
            "action_repeat": cfg["env"].get("action_repeat", 10), "auto_reset": True, "sensor_noise": True,
            "l2": "flushed between timed iterations (192 MiB fill outside the event pair)",
            "parallelism": f"env-sharded x{world}, no per-step collective"}
    if job.kind == "random":
        conf["actions"] = "fixed-seed uniform(-1,1), fresh draw per env and step, generated on device before each timed step"
    elif job.kind == "cpg":
        conf["actions"] = ("Hopf CPG torques (k_cpg: oscillators + IK + joint PD + Cartesian impedance) computed inside the timed "
                           "region; a bench step = 10 ticks of 1 ms = one control-step equivalent")
        conf["cpg"] = cfg["cpg"]
        conf["env_ticks_per_sec"] = value * 10
    else:
        conf["actions"] = ("MlpPolicy 2x64 tanh (random init, seed 7) on VecNormalize'd observations, DiagGaussian sample, "
                           "evaluated on the device inside the timed region")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": conf, "steady_state": steady,
        "clocks": clocks, "gpu_launches": int(launches), "host_us_per_step": 1e6 * host_s / args.steps,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "path": path},
        "roofline": roofline, "cpu_baseline": cpu,
        "wall_s_timed_region": t_wall,
        "rollout_stats": {k: rollout[k] for k in ("episodes", "mean_length", "mean_max_height", "mean_max_fwd",
                                                  "mean_flip_completion", "mean_return", "terminated_fraction")},
    }
    if args.series:
        line["step_ms_series"] = [round(a.elapsed_time(b), 4) for a, b in ev]
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)   # on top of the pre-roll to the stationary regime
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--max-preroll", type=int, default=600)
    ap.add_argument("--min-preroll", type=int, default=150)
    ap.add_argument("--series", action="store_true", help="add the per-step device times to the line")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0's shard) as DIR/<name>.npy, float32, "
                         f"at most {DUMP_BYTES // 10**6} MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
