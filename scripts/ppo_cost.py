"""Cost of batched PPO training (quadruped_springs_b200/ppo.py) per control step and per iteration.

Per step, three arms alternated in one session on the same env, in steady state after a random pre-roll:
  a  qs_step alone
  b  qs_ppo_act + qs_step + qs_obs_stats + qs_ppo_reward: what BatchedPPO runs per step
  c  qs_step + the same work in torch: VecNormalizeTorch's statistics and normalisation, MlpPolicyTorch's actor and
     critic, torch sampling and log-probability, buffer writes, the reward path, and the time-limit bootstrap by indexing
     the truncated envs (which synchronises the host)
for bench.py configuration 3 at 65536 envs and configuration 2 at 4096 envs, with the default MLP ([64, 64], tanh).
Every arm steps the same zero actions, so the physics is the same in all three; b and c write the actions they compute
to a buffer the step does not read.  Each arm is timed with CUDA events over `--steps` steps per round, `--rounds`
rounds, a b c a b c ...; the median per step is reported, and the overheads b - a and c - a.  Then each launch b adds,
and qs_step, on its own: device time per launch (CUDA events) and the host time to enqueue it.

Then `--iterations` BatchedPPO iterations per configuration (after one warm-up iteration), with n_steps 16, 8
minibatches per epoch and 5 epochs: rollout, GAE and update seconds and the end-to-end training env-steps/s.

One JSON line per measurement, with the device name and its power limit.

    python scripts/ppo_cost.py [--steps 200] [--rounds 5] [--iterations 3]
"""
import argparse
import ctypes as C
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


def per_step(cfg_id, n, steps, rounds, dev):
    import numpy as np
    import torch

    import bench
    from quadruped_springs_b200 import BatchedQuadrupedGymEnv, _lib
    from quadruped_springs_b200.ars import obs_stats
    from quadruped_springs_b200.env import _p, _stream_ptr
    from quadruped_springs_b200.ppo import BatchedPPO, ppo_act_args, ppo_reward
    from quadruped_springs_b200.vec_env import RunningMeanStdTorch

    env_kw = bench.CONFIGS[cfg_id]["env"]
    T = 16
    tr = BatchedPPO("MlpPolicy", env_kw, num_envs=n, n_steps=T, device=dev)
    env = BatchedQuadrupedGymEnv(num_envs=n, device=dev, seed=0, auto_reset=True, **env_kw)
    term = torch.zeros(n, env.obs_dim, device=dev)
    env.set_terminal_obs_buffer(term)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(0)
    zero_act = torch.zeros(n, env.action_dim, device=dev)
    for _ in range(150):
        env.step(torch.rand(n, env.action_dim, device=dev, generator=g) * 2 - 1)
    for _ in range(50):
        env.step(zero_act)
    L, stream = env._L, _stream_ptr(dev)
    O, A = env.obs_dim, env.action_dim
    buf = {"obs": torch.zeros(T, n, O, device=dev), "actions": torch.zeros(T, n, A, device=dev),
           **{k: torch.zeros(T, n, device=dev) for k in ("values", "log_probs", "episode_starts", "rewards")}}
    vn = tr.vec_normalize
    obs_count, ret_count = tr._obs_count, tr._ret_count
    ep_ret = torch.zeros(n, dtype=torch.float64, device=dev)
    ep_len = torch.zeros(n, dtype=torch.int32, device=dev)
    totals = torch.zeros(4, dtype=torch.float64, device=dev)
    actions = torch.empty(n, A, device=dev)
    theta = tr.theta()
    pol = tr.policy
    t_rms, r_rms = RunningMeanStdTorch((O,), dev), RunningMeanStdTorch((), dev)
    returns = torch.zeros(n, dtype=torch.float64, device=dev)
    gen = torch.Generator(device=dev).manual_seed(1)
    state = {"t": 0}

    def step(a):
        _lib.check(L.qs_step(env._h, _p(a), _p(env._obs), _p(env._reward), _p(env._done), _p(env._trunc), stream))

    def arm_a():
        step(zero_act)

    # one argument struct, as BatchedPPO.collect_rollouts builds it
    act_args, _ = ppo_act_args(tr.arch, env._obs, theta, stats=(vn.obs_rms.mean, vn.obs_rms.var), n_steps=T,
                               episode_start=env._done, prev_truncated=env._trunc, terminal_obs=term, actions=actions,
                               buffers=buf)
    act_ref, arch_ref = C.byref(act_args), C.byref(tr.arch)

    def act(t):
        act_args.step = t
        _lib.check(L.qs_ppo_act(act_ref, arch_ref, stream))

    def arm_b():
        t = state["t"] = (state["t"] + 1) % T
        act(t)
        step(zero_act)
        obs_stats(env._obs, vn.obs_rms.mean, vn.obs_rms.var, obs_count)
        ppo_reward(env._reward, env._done, buf["rewards"][t], ep_ret, ep_len, (vn.returns, vn.ret_rms.mean,
                   vn.ret_rms.var, ret_count), totals=totals)

    def arm_c():
        nonlocal returns
        t = state["t"] = (state["t"] + 1) % T
        with torch.no_grad():
            x = ((env._obs.double() - t_rms.mean) / torch.sqrt(t_rms.var + 1e-8)).clamp(-10, 10).float()
            mean = pol.action_net(pol.mlp_extractor.policy_net(x))
            value = pol.value_net(pol.mlp_extractor.value_net(x)).flatten()
            std = pol.log_std.exp()
            a = mean + torch.randn(mean.shape, device=dev, generator=gen) * std
            lp = torch.distributions.Normal(mean, std).log_prob(a).sum(1)
            actions.copy_(a.clamp(-1, 1))
            buf["obs"][t], buf["actions"][t], buf["values"][t], buf["log_probs"][t] = x, a, value, lp
            buf["episode_starts"][t] = env._done.float()
            step(zero_act)
            t_rms.update(env._obs)
            rew = env._reward.double()
            returns = returns * 0.99 + rew
            r_rms.update(returns)
            buf["rewards"][t] = (rew / torch.sqrt(r_rms.var + 1e-8)).clamp(-10, 10).float()
            done = env._done.bool()
            returns = torch.where(done, torch.zeros_like(returns), returns)
            idx = torch.nonzero(done & env._trunc.bool()).flatten()    # host synchronisation
            if len(idx):
                tx = ((term[idx].double() - t_rms.mean) / torch.sqrt(t_rms.var + 1e-8)).clamp(-10, 10).float()
                buf["rewards"][t, idx] += 0.99 * pol.value_net(pol.mlp_extractor.value_net(tx)).flatten()

    arms = {"a": arm_a, "b": arm_b, "c": arm_c}
    for f in arms.values():
        for _ in range(10):
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / steps)
    med = {k: float(np.median(v)) for k, v in times.items()}

    # each added launch on its own, back to back: device time per launch (CUDA events) and host time to enqueue it
    # (the loop's wall time before the synchronise); host >= device means the launch stream is host-bound
    pieces = {"qs_ppo_act": lambda: act(1), "qs_obs_stats": lambda: obs_stats(env._obs, vn.obs_rms.mean, vn.obs_rms.var,
                                                                              obs_count),
              "qs_ppo_reward": lambda: ppo_reward(env._reward, env._done, buf["rewards"][1], ep_ret, ep_len,
                                                  (vn.returns, vn.ret_rms.mean, vn.ret_rms.var, ret_count), totals=totals),
              "qs_step": arm_a}
    kernels = {}
    for name, f in pieces.items():
        f()
        dev_ms, host_ms = [], []
        for _ in range(rounds):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0 = time.perf_counter()
            e0.record()
            for _ in range(steps):
                f()
            e1.record()
            host_ms.append((time.perf_counter() - h0) * 1e3 / steps)
            e1.synchronize()
            dev_ms.append(e0.elapsed_time(e1) / steps)
        kernels[name] = {"device_ms": float(np.median(dev_ms)), "host_enqueue_ms": float(np.median(host_ms))}
    env.close()
    return {"config": cfg_id, "envs": n, "params": int(theta.numel()), "ms_per_step": med,
            "spread_ms": {k: [min(v), max(v)] for k, v in times.items()},
            "overhead_ms_b": med["b"] - med["a"], "overhead_ms_c": med["c"] - med["a"], "per_launch": kernels}


def iterations(cfg_id, n, count, dev):
    import numpy as np

    import bench
    from quadruped_springs_b200.ppo import BatchedPPO

    T = 16
    tr = BatchedPPO("MlpPolicy", bench.CONFIGS[cfg_id]["env"], num_envs=n, n_steps=T, batch_size=n * T // 8, n_epochs=5,
                    device=dev)
    tr.train_iteration()   # warm-up: creates the env, first settles, cuBLAS plans
    recs = [tr.train_iteration() for _ in range(count)]
    tr.env.close()
    med = lambda f: float(np.median([f(r) for r in recs]))
    return {"iteration": cfg_id, "envs": n, "n_steps": T, "batch_size": n * T // 8, "n_epochs": 5,
            "rollout_s": med(lambda r: r["seconds"]["rollout"]), "gae_s": med(lambda r: r["seconds"]["gae"]),
            "update_s": med(lambda r: r["seconds"]["update"]), "env_steps_per_s": med(lambda r: r["env_steps_per_s"]),
            "rollout_env_steps_per_s": med(lambda r: r["rollout_env_steps_per_s"]), "iterations": count}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iterations", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ppo_cost.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    card = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit(0)}
    for cfg_id, n in ((3, 65536), (2, 4096)):
        print(json.dumps({**per_step(cfg_id, n, args.steps, args.rounds, dev), **card}), flush=True)
    for cfg_id, n in ((3, 65536), (2, 4096)):
        print(json.dumps({**iterations(cfg_id, n, args.iterations, dev), **card}), flush=True)


if __name__ == "__main__":
    main()
