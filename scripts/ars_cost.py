"""Cost of batched ARS training (quadruped_springs_b200/ars.py) per control step and per iteration.

Per step, three arms alternated in one session on the same env, in steady state after a random pre-roll:
  a  qs_step alone
  b  qs_ars_act + qs_step + qs_obs_stats (with the episode bookkeeping): what BatchedARS runs
  c  qs_step + the same work in torch: VecNormalizeTorch-style masked statistics and normalisation, candidate weights
     materialised per env ([N, P]) and one torch.bmm per layer, bookkeeping with torch.where
for bench.py configuration 3 at 65536 envs and configuration 2 at 4096 envs, each with the linear and the MLP policy
(n_delta = 8, one candidate per N / 16 envs).  Every arm steps the same zero actions (the zero policy: the robots hold
the init pose), and b and c write the actions they compute to a buffer the step does not read.  Otherwise the physics
would differ between arms (falls, resets and their settles) and dominate the difference.  Each arm is timed with CUDA events over `--steps` steps per round,
`--rounds` rounds, a b c a b c ...; the median per step is reported, and the overheads b - a and c - a.

Then one full BatchedARS iteration of configuration 3 at 65536 envs per policy, split into reset (env.reset of every
env), rollout (act / step / statistics until every env has finished its episode) and update.

One JSON line per measurement, with the device name and its power limit.

    python scripts/ars_cost.py [--steps 200] [--rounds 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def torch_equivalent(tr, obs, alive, reward, done, ret, length, theta, deltas, delta_std, cand, stats):
    """arm c: the trainer's per-step work in torch, no host synchronisation"""
    import torch
    mean, var, count = stats
    x = obs.double()
    w = alive.double()
    bc = w.sum()
    safe = torch.clamp(bc, min=1.0)
    bm = (x * w[:, None]).sum(0) / safe
    bv = (((x - bm) ** 2) * w[:, None]).sum(0) / safe
    delta = bm - mean
    tot = count + bc
    new_mean = mean + delta * bc / tot
    new_var = (var * count + bv * bc + delta * delta * count * bc / tot) / tot
    keep = bc > 0
    mean.copy_(torch.where(keep, new_mean, mean))
    var.copy_(torch.where(keep, new_var, var))
    count.copy_(torch.where(keep, tot, count))
    a = alive.bool()
    ret.add_(torch.where(a, reward.double(), torch.zeros_like(ret)))
    length.add_(a.to(torch.int32))
    alive.copy_((a & ~done.bool()).to(torch.uint8))
    # act for the next step: normalise, candidate weights per env, one bmm per layer
    h = ((obs.double() - mean) / torch.sqrt(var + 1e-8)).clamp(-10, 10).float()
    nd = deltas.shape[0]
    sign = torch.where(cand < nd, 1.0, -1.0)
    W = theta[None] + sign[:, None] * (deltas[cand % nd] * delta_std)
    pk = tr.policy_kwargs
    sizes = pk["net_arch"] + [tr.act_dim]
    off, fan_in = 0, tr.obs_dim
    for li, out_dim in enumerate(sizes):
        wl = W[:, off:off + out_dim * fan_in].view(-1, out_dim, fan_in)
        off += out_dim * fan_in
        h = torch.bmm(wl, h.unsqueeze(-1)).squeeze(-1)
        if pk["with_bias"]:
            h = h + W[:, off:off + out_dim]
            off += out_dim
        if li < len(sizes) - 1:
            h = torch.relu(h) if pk["activation_fn"] == "ReLU" else torch.tanh(h)
        fan_in = out_dim
    if pk["squash_output"]:
        h = torch.tanh(h)
    return h.clamp(-1, 1)


def per_step(cfg_id, n, policy, steps, rounds, dev):
    import numpy as np
    import torch

    import bench
    from quadruped_springs_b200 import BatchedQuadrupedGymEnv, _lib
    from quadruped_springs_b200.ars import BatchedARS, ars_act, obs_stats
    from quadruped_springs_b200.env import _p, _stream_ptr

    env_kw = bench.CONFIGS[cfg_id]["env"]
    n_delta = 8
    tr = BatchedARS(policy, env_kw, n_delta=n_delta, n_eval_episodes=n // (2 * n_delta), device=dev, zero_policy=False)
    env = BatchedQuadrupedGymEnv(num_envs=n, device=dev, seed=0, auto_reset=True, **env_kw)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(0)
    zero_act = torch.zeros(n, env.action_dim, device=dev)
    for _ in range(150):   # pre-roll: random actions, then the zero actions every arm steps
        env.step(torch.rand(n, env.action_dim, device=dev, generator=g) * 2 - 1)
    for _ in range(50):
        env.step(zero_act)
    L, stream = env._L, _stream_ptr(dev)
    epc = n // (2 * n_delta)
    theta = tr.theta.clone()
    deltas = tr.sample_deltas(0)
    cand = torch.arange(n, device=dev) // epc
    stats = (tr.vec_normalize.obs_rms.mean, tr.vec_normalize.obs_rms.var, tr._count)
    alive = torch.ones(n, dtype=torch.uint8, device=dev)
    ret = torch.zeros(n, dtype=torch.float64, device=dev)
    length = torch.zeros(n, dtype=torch.int32, device=dev)
    actions = torch.empty(n, env.action_dim, device=dev)
    obs = env._obs

    def step(a):
        _lib.check(L.qs_step(env._h, _p(a), _p(env._obs), _p(env._reward), _p(env._done), _p(env._trunc), stream))

    def arm_a():
        step(zero_act)

    def arm_b():
        ars_act(obs, theta, tr.arch, deltas, 0.05, n_delta, 0, epc, stats[0], stats[1], out=actions)
        step(zero_act)
        obs_stats(obs, *stats, alive=alive, bookkeeping=(env._reward, env._done, ret, length))

    def arm_c():
        step(zero_act)
        actions.copy_(torch_equivalent(tr, obs, alive, env._reward, env._done, ret, length, theta, deltas, 0.05, cand,
                                       stats))

    arms = {"a": arm_a, "b": arm_b, "c": arm_c}
    for f in arms.values():   # warm-up
        for _ in range(10):
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, f in arms.items():
            alive.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / steps)
    med = {k: float(np.median(v)) for k, v in times.items()}
    env.close()
    return {"config": cfg_id, "envs": n, "policy": policy, "params": tr.n_params, "ms_per_step": med,
            "spread_ms": {k: [min(v), max(v)] for k, v in times.items()},
            "overhead_ms_b": med["b"] - med["a"], "overhead_ms_c": med["c"] - med["a"]}


def iteration(policy, dev):
    import torch

    import bench
    from quadruped_springs_b200.ars import BatchedARS, candidate_returns

    n, n_delta = 65536, 8
    tr = BatchedARS(policy, bench.CONFIGS[3]["env"], n_delta=n_delta, n_eval_episodes=n // (2 * n_delta), device=dev)
    tr.train_iteration()   # warm-up (creates the env, first settles)
    env = tr.env
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    env.reset()
    torch.cuda.synchronize()
    t_reset = time.perf_counter() - t0
    lr, ds = tr.hyperparams(1.0)
    deltas = tr.sample_deltas(tr._n_updates)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ret, length, steps = tr.rollout(deltas, ds)   # its own reset first
    torch.cuda.synchronize()
    t_rollout = time.perf_counter() - t0 - t_reset
    t0 = time.perf_counter()
    tr.update(deltas, candidate_returns(ret, length, 2 * n_delta, n // (2 * n_delta)), lr)
    torch.cuda.synchronize()
    t_update = time.perf_counter() - t0
    out = {"iteration": policy, "envs": n, "reset_s": t_reset, "rollout_s": t_rollout, "update_s": t_update,
           "control_steps": steps, "env_steps": int(length.sum()),
           "rollout_env_steps_per_s": int(length.sum()) / t_rollout}
    tr.env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--skip-iteration", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ars_cost.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    card = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit(0)}
    for cfg_id, n in ((3, 65536), (2, 4096)):
        for policy in ("LinearPolicy", "MlpPolicy"):
            print(json.dumps({**per_step(cfg_id, n, policy, args.steps, args.rounds, dev), **card}), flush=True)
    if not args.skip_iteration:
        for policy in ("LinearPolicy", "MlpPolicy"):
            print(json.dumps({**iteration(policy, dev), **card}), flush=True)


if __name__ == "__main__":
    main()
