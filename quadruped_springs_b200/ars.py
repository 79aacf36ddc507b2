"""ARS training on the batched env: sb3-contrib's `ARS` (Augmented Random Search, Mania et al. 2018) with every
candidate policy of an iteration evaluated at once.

sb3-contrib evaluates its 2 * n_delta candidate policies one after another on one VecEnv.  Here one
`BatchedQuadrupedGymEnv` of N = 2 * n_delta * n_eval_episodes envs runs them side by side: env e runs candidate
e // n_eval_episodes, every env plays exactly one episode, and the candidate's return is the sum over its envs, as
`evaluate_policy(n_eval_episodes)` sums over its episodes.  Per control step the trainer launches two kernels beside
`qs_step` (csrc/qs_ars.cu): `qs_ars_act` (normalise the observation, run env e's candidate network, clip) and
`qs_obs_stats` (merge the observations of the envs still in their first episode into the running statistics, and
accumulate returns and lengths).  The update, the schedules and the parameter layout are sb3-contrib's
(`ARS._do_one_update`); what differs is listed in DESIGN.md section 7.

`save(log_dir)` writes the rl-baselines3-zoo layout that `load_model.replay` reads back (args.yml, vecnormalize.pkl,
best_model.zip), so training -> save -> replay closes inside the package.
"""
import ctypes as C
import io
import json
import os
import pickle
import time
import types
import zipfile
from collections import OrderedDict

import numpy as np
import torch
import yaml
from torch.nn.utils import parameters_to_vector, vector_to_parameters

from . import _lib
from .env import BatchedQuadrupedGymEnv, _p, _stream_ptr
from .load_model import (ENV_NAME, ArsPolicyTorch, first_episode_returns, make_vec_env, read_vecnormalize_pkl,
                         replay_env_kwargs)
from .vec_env import VecNormalizeTorch

# sb3_contrib.ars.policies: ARSLinearPolicy = ARSPolicy(net_arch=[], with_bias=False, squash_output=False)
POLICIES = {
    "LinearPolicy": ("ARSLinearPolicy", dict(net_arch=[], activation_fn="ReLU", with_bias=False, squash_output=False)),
    "MlpPolicy": ("ARSPolicy", dict(net_arch=[64, 64], activation_fn="ReLU", with_bias=True, squash_output=True)),
}
_ACTIVATIONS = {"ReLU": _lib.QS_ARS_RELU, "Tanh": _lib.QS_ARS_TANH}


def _activation_name(fn):
    """"ReLU" / "Tanh" from a name or a torch.nn class (what policy_kwargs["activation_fn"] holds in SB3)"""
    name = fn if isinstance(fn, str) else getattr(fn, "__name__", str(fn))
    for k in _ACTIVATIONS:
        if k.lower() in name.lower():
            return k
    raise ValueError(f"activation_fn {fn!r}: only ReLU and Tanh are provided")


def _schedule(v):
    return v if callable(v) else (lambda _progress_remaining, c=float(v): c)


# ----------------------------------------------------------------------------- kernels (tensor front ends)
def obs_stats(obs, mean, var, count, alive=None, bookkeeping=None):
    """qs_obs_stats: merge the rows of obs [N, O] with alive != 0 (all rows when alive is None) into the running float64
    statistics mean [O], var [O], count [1] in place (RunningMeanStd.update).  bookkeeping = (reward [N] f32, done [N]
    u8, ret [N] f64, length [N] i32) also accumulates the returns and lengths of the alive envs and then clears alive
    where done.  mean None: bookkeeping only."""
    n = int(alive.shape[0] if obs is None else obs.shape[0])
    o = 0 if obs is None else int(obs.shape[1])
    rw, dn, rt, ln = bookkeeping if bookkeeping is not None else (None,) * 4
    dev = (obs if obs is not None else alive).device
    _lib.check(_lib.lib().qs_obs_stats(_p(obs), _p(alive), n, o, _p(mean), _p(var), _p(count), _p(rw), _p(dn), _p(rt),
                                       _p(ln), _stream_ptr(dev)))


def ars_act(obs, theta, arch, deltas=None, delta_std=0.0, n_delta=1, first_candidate=0, envs_per_candidate=None,
            mean=None, var=None, clip_obs=10.0, epsilon=1e-8, out=None):
    """qs_ars_act: actions [N, A] of env e's candidate first_candidate + e // envs_per_candidate (theta itself when
    deltas is None), on observations normalised with mean / var when given."""
    n = int(obs.shape[0])
    if out is None:
        out = torch.empty(n, arch.act_dim, device=obs.device)
    epc = n if envs_per_candidate is None else int(envs_per_candidate)
    _lib.check(_lib.lib().qs_ars_act(_p(obs), _p(mean), _p(var), float(clip_obs), float(epsilon), _p(theta), _p(deltas),
                                     float(delta_std), int(n_delta), int(first_candidate), epc, C.byref(arch), _p(out), n,
                                     _stream_ptr(obs.device)))
    return out


def run_candidates(env, theta, arch, deltas, delta_std, n_delta, first_candidate, envs_per_candidate, stats=None,
                   update_stats=False, clip_obs=10.0, epsilon=1e-8, max_steps=1500, check_every=16):
    """One episode per env of `env` (auto_reset) with env e running candidate first_candidate + e // envs_per_candidate:
    reset every env, then act -> qs_step -> bookkeeping until every env has finished its first episode.
    stats = (mean, var, count) device tensors: observations are normalised with them and, when update_stats, the reset
    observations and then every step's observations of the envs still in their first episode are merged into them
    before they normalise the next action.  Returns (return [N] f64, length [N] i32, control steps run)."""
    n, dev, L = env.num_envs, env.device, env._L
    alive = torch.ones(n, dtype=torch.uint8, device=dev)
    ret = torch.zeros(n, dtype=torch.float64, device=dev)
    length = torch.zeros(n, dtype=torch.int32, device=dev)
    actions = torch.empty(n, env.action_dim, device=dev)
    mean, var, count = stats if stats is not None else (None, None, None)
    smean, svar, scount = (mean, var, count) if update_stats else (None, None, None)
    obs = env.reset()
    if update_stats:
        obs_stats(obs, mean, var, count)
    stream = _stream_ptr(dev)
    book = (env._reward, env._done, ret, length)
    steps = 0
    while steps < max_steps:
        for _ in range(min(check_every, max_steps - steps)):
            ars_act(obs, theta, arch, deltas, delta_std, n_delta, first_candidate, envs_per_candidate, mean, var,
                    clip_obs, epsilon, out=actions)
            _lib.check(L.qs_step(env._h, _p(actions), _p(env._obs), _p(env._reward), _p(env._done), _p(env._trunc),
                                 stream))
            obs_stats(obs if update_stats else None, smean, svar, scount, alive=alive, bookkeeping=book)
            steps += 1
        if not bool(alive.any()):
            break
    env._last_host_obs = None
    return ret, length, steps


def candidate_returns(ret, length, n_candidates, n_eval_episodes, alive_bonus_offset=0.0):
    """evaluate_candidates: sum(episode_rewards) + alive_bonus_offset * sum(episode_lengths) per candidate, stored in
    float32 as sb3-contrib's candidate_returns tensor"""
    r = ret.view(n_candidates, n_eval_episodes).sum(1)
    steps = length.view(n_candidates, n_eval_episodes).to(torch.float64).sum(1)
    return (r + float(alive_bonus_offset) * steps).to(torch.float32)


def ars_update(theta, deltas, returns, n_top, learning_rate):
    """ARS._do_one_update after the evaluation: keep the n_top directions with the largest max(plus, minus) (ties keep
    the lower index), scale by the standard deviation of their 2 n_top returns, step along the unscaled deltas.
    Returns (new theta, return_std, step_size)."""
    n_delta = deltas.shape[0]
    plus, minus = returns[:n_delta], returns[n_delta:]
    top = torch.maximum(plus, minus)
    idx = torch.argsort(top, descending=True, stable=True)[:n_top]
    plus, minus, d = plus[idx], minus[idx], deltas[idx]
    return_std = torch.cat([plus, minus]).std()
    step_size = learning_rate / (n_top * return_std + 1e-6)
    return theta + step_size * ((plus - minus) @ d), return_std, step_size


# ----------------------------------------------------------------------------- vecnormalize.pkl writer
class _SB3Object:
    """pickled as the stable-baselines3 class named by `_sb3_class`, its __dict__ the state (what VecNormalize.save
    writes); read_vecnormalize_pkl reads it without SB3"""

    def __init__(self, **state):
        self.__dict__.update(state)


class _VecNormalizeState(_SB3Object):
    _sb3_class = ("stable_baselines3.common.vec_env.vec_normalize", "VecNormalize")


class _RunningMeanStdState(_SB3Object):
    _sb3_class = ("stable_baselines3.common.running_mean_std", "RunningMeanStd")


class _SB3Pickler(pickle._Pickler):
    def save_global(self, obj, name=None):
        target = obj.__dict__.get("_sb3_class") if isinstance(obj, type) else None
        if target is None:
            return super().save_global(obj, name)
        self.write(pickle.GLOBAL + f"{target[0]}\n{target[1]}\n".encode("utf-8"))
        self.memoize(obj)


def write_vecnormalize_pkl(path, state, num_envs, norm_obs=True, training=True, norm_reward=False):
    """a `VecNormalize.save()`-shaped pickle of VecNormalizeTorch.state_dict() `state` (protocol 4)"""
    rms = lambda m, v, c: _RunningMeanStdState(mean=np.asarray(m, np.float64), var=np.asarray(v, np.float64), count=float(c))
    vn = _VecNormalizeState(
        obs_rms=rms(state["obs_mean"], state["obs_var"], state["obs_count"]),
        ret_rms=rms(state["ret_mean"], state["ret_var"], state["ret_count"]),
        clip_obs=float(state["clip_obs"]), clip_reward=float(state["clip_reward"]), gamma=float(state["gamma"]),
        epsilon=float(state["epsilon"]), training=bool(training), norm_obs=bool(norm_obs), norm_reward=bool(norm_reward),
        num_envs=int(num_envs), norm_obs_keys=None)
    buf = io.BytesIO()
    _SB3Pickler(buf, protocol=4).dump(vn)
    with open(path, "wb") as f:
        f.write(buf.getvalue())


# ----------------------------------------------------------------------------- the trainer
class BatchedARS:
    """sb3_contrib.ARS(policy, env, n_delta, n_top, learning_rate, delta_std, zero_policy, alive_bonus_offset,
    n_eval_episodes) over one BatchedQuadrupedGymEnv(**env_kwargs) of 2 * n_delta * n_eval_episodes envs.

    policy: "LinearPolicy" (ARSLinearPolicy) or "MlpPolicy" (ARSPolicy); policy_kwargs may set net_arch (up to two
    hidden layers of at most 64), activation_fn (ReLU or Tanh), with_bias and squash_output.  learning_rate and
    delta_std are constants or callables of progress_remaining.  normalize: rl-zoo's hyper-parameter, observation
    normalisation by VecNormalize(norm_obs=True, norm_reward=False); its statistics are `vec_normalize` (set
    `vec_normalize.training = False` to freeze them).  env_kwargs may hold num_envs, which must then equal
    2 * n_delta * n_eval_episodes.  The env is created on the first rollout; saving, loading and the update need no GPU.
    """

    def __init__(self, policy, env_kwargs=None, n_delta=8, n_top=None, learning_rate=0.02, delta_std=0.05,
                 zero_policy=True, alive_bonus_offset=0, n_eval_episodes=1, normalize=True, seed=0, device="cuda",
                 policy_kwargs=None, verbose=0):
        if policy not in POLICIES:
            raise ValueError(f"unknown policy {policy!r}: {sorted(POLICIES)}")
        n_delta, n_eval_episodes = int(n_delta), int(n_eval_episodes)
        if n_delta < 1 or n_eval_episodes < 1:
            raise ValueError("n_delta and n_eval_episodes must be at least 1")
        n_top = n_delta if n_top is None else int(n_top)
        if not 1 <= n_top <= n_delta:
            raise ValueError(f"n_top must lie in [1, n_delta = {n_delta}], got {n_top}")
        env_kwargs = dict(env_kwargs or {})
        self.num_envs = 2 * n_delta * n_eval_episodes
        n_env = env_kwargs.pop("num_envs", None)
        if n_env is not None and int(n_env) != self.num_envs:
            raise ValueError(f"the batch must hold 2 * n_delta * n_eval_episodes = {self.num_envs} envs, got {n_env}")
        for k in ("device", "seed", "auto_reset"):
            if k in env_kwargs:
                raise ValueError(f"env_kwargs[{k!r}] is set by the trainer")
        self.policy_class, pk = POLICIES[policy][0], dict(POLICIES[policy][1])
        for k, v in (policy_kwargs or {}).items():
            if k not in pk:
                raise ValueError(f"unknown policy_kwargs entry {k!r}")
            pk[k] = v
        pk["net_arch"] = [int(h) for h in pk["net_arch"]]
        pk["activation_fn"] = _activation_name(pk["activation_fn"])
        pk["with_bias"], pk["squash_output"] = bool(pk["with_bias"]), bool(pk["squash_output"])
        if len(pk["net_arch"]) > 2 or not all(1 <= h <= _lib.QS_ARS_MAX_HIDDEN for h in pk["net_arch"]):
            raise ValueError(f"net_arch {pk['net_arch']}: at most two hidden layers of 1..{_lib.QS_ARS_MAX_HIDDEN}")
        self.policy_name, self.policy_kwargs = policy, pk
        self.env_kwargs = env_kwargs
        self.n_delta, self.n_top, self.n_eval_episodes = n_delta, n_top, n_eval_episodes
        self.learning_rate, self.delta_std = learning_rate, delta_std
        self.zero_policy, self.alive_bonus_offset = bool(zero_policy), float(alive_bonus_offset)
        self.normalize, self.seed, self.verbose = bool(normalize), int(seed), verbose
        self.device = torch.device(device)

        from .ops import make_config
        cfg = make_config(**{k: env_kwargs[k] for k in ("enable_springs", "motor_control_mode", "action_space_mode",
                                                         "task_env", "observation_space_mode") if k in env_kwargs},
                          is_rl_interface=int(bool(env_kwargs.get("isRLGymInterface", True))))
        L = _lib.lib()
        self.obs_dim, self.act_dim = int(L.qs_config_obs_dim(C.byref(cfg))), int(L.qs_config_action_dim(C.byref(cfg)))
        if self.act_dim > _lib.QS_ARS_MAX_ACT:
            raise ValueError(f"the action has {self.act_dim} entries; qs_ars_act takes at most {_lib.QS_ARS_MAX_ACT}")
        self.arch = _lib.QsArsArch(self.obs_dim, self.act_dim, len(pk["net_arch"]),
                                   (C.c_int32 * 2)(*(pk["net_arch"] + [0, 0])[:2]), _ACTIVATIONS[pk["activation_fn"]],
                                   int(pk["with_bias"]), int(pk["squash_output"]))
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(self.seed)
            net = self._new_policy("cpu")
        theta = parameters_to_vector(net.parameters()).detach()
        self.theta = (torch.zeros_like(theta) if self.zero_policy else theta).to(self.device).contiguous()
        self.n_params = int(self.theta.numel())

        shim = types.SimpleNamespace(num_envs=self.num_envs, observation_space=None, action_space=None,
                                     device=self.device, env=types.SimpleNamespace(obs_dim=self.obs_dim))
        self.vec_normalize = VecNormalizeTorch(shim, training=True, norm_obs=self.normalize, norm_reward=False)
        self._count = torch.tensor([self.vec_normalize.obs_rms.count], dtype=torch.float64, device=self.device)
        self.num_timesteps, self._n_updates = 0, 0
        self.logs, self.last_rollout = [], None
        self.env = None

    # ------------------------------------------------------------------ parameters
    def _new_policy(self, device):
        pk = self.policy_kwargs
        return ArsPolicyTorch(self.obs_dim, self.act_dim, tuple(pk["net_arch"]), pk["activation_fn"].lower(),
                              pk["with_bias"], pk["squash_output"]).to(device)

    def policy_module(self, theta=None):
        """ArsPolicyTorch holding theta (the current parameters by default): vector_to_parameters"""
        net = self._new_policy(self.device)
        vector_to_parameters((self.theta if theta is None else theta).to(self.device), net.parameters())
        return net

    def hyperparams(self, progress_remaining):
        """(learning_rate, delta_std) at progress_remaining = 1 - num_timesteps / total_timesteps"""
        return (float(_schedule(self.learning_rate)(progress_remaining)),
                float(_schedule(self.delta_std)(progress_remaining)))

    def sample_deltas(self, iteration):
        """deltas ~ N(0, 1) [n_delta, P] of an iteration, from a device generator keyed by (seed, iteration)"""
        g = torch.Generator(device=self.device)
        g.manual_seed(((self.seed & 0xFFFFFFFF) << 32) | (int(iteration) & 0xFFFFFFFF))
        return torch.randn(self.n_delta, self.n_params, generator=g, device=self.device)

    def _stats(self):
        rms = self.vec_normalize.obs_rms
        return (rms.mean, rms.var, self._count) if self.normalize else None

    def _sync_count(self):
        self.vec_normalize.obs_rms.count = float(self._count.item())

    # ------------------------------------------------------------------ training
    def _get_env(self):
        if self.env is None:
            self.env = BatchedQuadrupedGymEnv(num_envs=self.num_envs, device=self.device, seed=self.seed,
                                              auto_reset=True, **self.env_kwargs)
        return self.env

    def rollout(self, deltas, delta_std):
        """evaluate_candidates: one episode per env, candidate e // n_eval_episodes -> (return [N] f64, length [N] i32,
        control steps)"""
        vn = self.vec_normalize
        return run_candidates(self._get_env(), self.theta, self.arch, deltas, delta_std, self.n_delta, 0,
                              self.n_eval_episodes, stats=self._stats(), update_stats=self.normalize and vn.training,
                              clip_obs=vn.clip_obs, epsilon=vn.epsilon)

    def update(self, deltas, returns, learning_rate):
        """the update of _do_one_update on candidate returns [2 n_delta] (float32); returns (return_std, step_size)"""
        self.theta, return_std, step_size = ars_update(self.theta, deltas, returns.to(self.device), self.n_top,
                                                       learning_rate)
        self._n_updates += 1
        return float(return_std), float(step_size)

    def train_iteration(self, progress_remaining=1.0):
        """one ARS iteration; returns its log record"""
        t0 = time.perf_counter()
        lr, dstd = self.hyperparams(progress_remaining)
        deltas = self.sample_deltas(self._n_updates)
        ret, length, steps = self.rollout(deltas, dstd)
        returns = candidate_returns(ret, length, 2 * self.n_delta, self.n_eval_episodes, self.alive_bonus_offset)
        env_steps = int(length.sum())
        self.num_timesteps += env_steps
        self.last_rollout = {"return": ret, "length": length, "deltas": deltas, "candidate_returns": returns}
        return_std, step_size = self.update(deltas, returns, lr)
        if self.normalize:
            self._sync_count()
        rec = {"iteration": self._n_updates, "num_timesteps": self.num_timesteps,
               "mean_return": float(returns.mean()), "max_return": float(returns.max()), "return_std": return_std,
               "step_size": step_size, "learning_rate": lr, "delta_std": dstd, "control_steps": steps,
               "env_steps": env_steps, "seconds": time.perf_counter() - t0}
        self.logs.append(rec)
        if self.verbose:
            print(json.dumps(rec))
        return rec

    def learn(self, total_timesteps, callback=None):
        """iterations until num_timesteps >= total_timesteps; callback(trainer, record) after each, False stops"""
        while self.num_timesteps < total_timesteps:
            rec = self.train_iteration(1.0 - float(self.num_timesteps) / float(total_timesteps))
            if callback is not None and callback(self, rec) is False:
                break
        return self

    # ------------------------------------------------------------------ evaluation
    def evaluate(self, n_envs, deterministic=True, task=None, seed=None, go_to_rest_wrapper=False, max_steps=1500):
        """the current theta through ArsPolicyTorch with the statistics frozen, one episode per env, in the env
        load_model.replay builds from the saved directory (ground randomizer, `task`, default the training task): the
        array replay(log_dir, task, algo="ars", n_envs, go_to_rest_wrapper, seed) returns.  ARS policies are
        deterministic, so `deterministic` changes nothing."""
        kw = replay_env_kwargs(self.env_kwargs, task or self.env_kwargs.get("task_env", "NO_TASK"))
        kw.pop("render", None)
        venv = make_vec_env(kw, n_envs=n_envs, device=self.device, go_to_rest_wrapper=go_to_rest_wrapper,
                            seed=self.seed if seed is None else seed)
        try:
            vn = VecNormalizeTorch(venv, training=False, norm_obs=self.normalize, norm_reward=False)
            vn.load_state_dict(self.vec_normalize.state_dict())
            return first_episode_returns(vn, self.policy_module(), max_steps)
        finally:
            venv.close()

    # ------------------------------------------------------------------ rl-zoo directory
    def save(self, log_dir):
        """log_dir/QuadrupedSpring-v0/{args.yml, vecnormalize.pkl} and log_dir/best_model.zip (rl-zoo's layout)"""
        env_dir = os.path.join(log_dir, ENV_NAME)
        os.makedirs(env_dir, exist_ok=True)
        args = OrderedDict([("algo", "ars"), ("env", ENV_NAME), ("env_kwargs", OrderedDict(sorted(self.env_kwargs.items()))),
                            ("n_timesteps", int(self.num_timesteps)), ("seed", self.seed)])
        with open(os.path.join(env_dir, "args.yml"), "w") as f:
            yaml.dump(args, f)
        if self.normalize:
            self._sync_count()
        write_vecnormalize_pkl(os.path.join(env_dir, "vecnormalize.pkl"), self.vec_normalize.state_dict(),
                               self.num_envs, norm_obs=self.normalize, training=self.vec_normalize.training)
        pk = self.policy_kwargs
        data = {"policy_class": {"__module__": "sb3_contrib.ars.policies", "__name__": self.policy_class},
                "policy_kwargs": {"net_arch": pk["net_arch"],
                                  "activation_fn": f"<class 'torch.nn.modules.activation.{pk['activation_fn']}'>",
                                  "with_bias": pk["with_bias"], "squash_output": pk["squash_output"]},
                "num_timesteps": int(self.num_timesteps), "_n_updates": int(self._n_updates), "seed": self.seed,
                "n_delta": self.n_delta, "n_top": self.n_top, "n_eval_episodes": self.n_eval_episodes,
                "alive_bonus_offset": self.alive_bonus_offset, "zero_policy": self.zero_policy}
        sd = OrderedDict((k, v.detach().cpu().clone()) for k, v in self.policy_module().state_dict().items())
        pth = io.BytesIO()
        torch.save(sd, pth)
        with zipfile.ZipFile(os.path.join(log_dir, "best_model.zip"), "w") as z:
            z.writestr("data", json.dumps(data, indent=4))
            z.writestr("policy.pth", pth.getvalue())
        return log_dir

    def load(self, log_dir):
        """resume from a directory save() wrote: parameters, statistics, num_timesteps and the iteration count"""
        path = os.path.join(log_dir, "best_model.zip")
        net = ArsPolicyTorch.from_sb3_zip(path, device=self.device)
        own = {k: tuple(v.shape) for k, v in self._new_policy("cpu").state_dict().items()}
        if {k: tuple(v.shape) for k, v in net.state_dict().items()} != own:
            raise ValueError(f"{path} holds a different policy than this trainer's {self.policy_name}")
        with zipfile.ZipFile(path) as z:
            data = json.loads(z.read("data").decode())
        self.theta = parameters_to_vector(net.parameters()).detach().to(torch.float32).contiguous()
        st = read_vecnormalize_pkl(os.path.join(log_dir, ENV_NAME, "vecnormalize.pkl"))
        self.vec_normalize.load_state_dict(st)
        self._count.fill_(float(st["obs_count"]))
        self.num_timesteps = int(data.get("num_timesteps", 0))
        self._n_updates = int(data.get("_n_updates", 0))
        return self


__all__ = ["BatchedARS", "ars_act", "obs_stats", "run_candidates", "ars_update", "candidate_returns",
           "write_vecnormalize_pkl"]
