"""PPO training on the batched env: stable-baselines3's `PPO("MlpPolicy", env, ...)` with rl-zoo's `VecNormalize`, over
one `BatchedQuadrupedGymEnv(auto_reset=True)` of `num_envs` envs.

The rollout buffer holds `n_steps x num_envs` samples: every control step of every env is one sample, so at 65536 envs
`n_steps` is small (SB3's default 2048 would be 134 M samples).  Per control step the trainer launches three kernels
beside `qs_step` (csrc/qs_ppo.cu) and synchronises nothing:
  qs_ppo_act     normalise the observation, run the actor and the critic, sample the action (Philox), write the buffer
                 row and the clipped env action, and add the time-limit bootstrap of the previous step's truncations;
  qs_obs_stats   merge the step's observations into the running observation statistics (csrc/qs_ars.cu, unchanged);
  qs_ppo_reward  discounted return, its running statistics, the normalised reward, and the episode totals for the logs.
`qs_ppo_gae` computes the advantages once per rollout.  The update (minibatches, autograd, Adam) is torch.  What
differs from SB3 is listed in DESIGN.md section 7.

`save(log_dir)` writes the rl-baselines3-zoo layout that `load_model.replay(..., algo="ppo")` reads back.
"""
import ctypes as C
import io
import json
import math
import os
import time
import types
import zipfile
from collections import OrderedDict

import numpy as np
import torch
import yaml
from torch.nn.utils import parameters_to_vector

from . import _lib
from .ars import _activation_name, _schedule, obs_stats, write_vecnormalize_pkl
from .env import BatchedQuadrupedGymEnv, _stream_ptr
from .load_model import ENV_NAME, first_episode_returns, make_vec_env, read_vecnormalize_pkl, replay_env_kwargs
from .vec_env import MlpPolicyTorch, VecNormalizeTorch

_ACTIVATIONS = {"ReLU": _lib.QS_ARS_RELU, "Tanh": _lib.QS_ARS_TANH}
DEFAULT_POLICY_KWARGS = dict(net_arch=[64, 64], activation_fn="Tanh", ortho_init=True, log_std_init=0.0)


def _a(t):
    return t.data_ptr() if t is not None else None


# ----------------------------------------------------------------------------- kernels (tensor front ends)
def ppo_act(arch, obs, theta, **kw):
    """qs_ppo_act on obs [N, O] with parameters theta (parameters_to_vector of MlpPolicyTorch); the keywords are
    ppo_act_args'.  Returns `actions` (allocated when None and needed)."""
    p, actions = ppo_act_args(arch, obs, theta, **kw)
    _lib.check(_lib.lib().qs_ppo_act(C.byref(p), C.byref(arch), _stream_ptr(obs.device)))
    return actions


def ppo_act_args(arch, obs, theta, stats=None, clip_obs=10.0, epsilon=1e-8, seed=0, env_id_offset=0, iteration=0,
                 step=0, n_steps=1, gamma=0.99, episode_start=None, prev_truncated=None, terminal_obs=None, actions=None,
                 buffers=None, last_values=None, mean_out=None, values_only=False, deterministic=False):
    """the qs_ppo_args struct of one qs_ppo_act call -> (struct, actions).  stats = (mean, var) float64 device tensors or
    None; buffers = dict of the step-major rollout arrays obs, actions, values, log_probs, episode_starts, rewards."""
    n = int(obs.shape[0])
    if actions is None and not values_only:
        actions = torch.empty(n, arch.act_dim, device=obs.device)
    b = buffers or {}
    p = _lib.QsPpoArgs()
    p.obs, p.theta = _a(obs), _a(theta)
    if stats is not None:
        p.obs_mean, p.obs_var = _a(stats[0]), _a(stats[1])
    p.episode_start, p.prev_truncated, p.terminal_obs = _a(episode_start), _a(prev_truncated), _a(terminal_obs)
    p.actions, p.last_values, p.mean_out = _a(actions), _a(last_values), _a(mean_out)
    for k in ("obs", "actions", "values", "log_probs", "episode_starts", "rewards"):
        setattr(p, "buf_" + k, _a(b.get(k)))
    p.clip_obs, p.epsilon, p.seed, p.env_id_offset = float(clip_obs), float(epsilon), int(seed), int(env_id_offset)
    p.gamma, p.iteration, p.step, p.n_steps, p.n = float(gamma), int(iteration), int(step), int(n_steps), n
    p.values_only, p.deterministic = int(bool(values_only)), int(bool(deterministic))
    return p, actions


def ppo_reward(reward, done, reward_out, ep_return, ep_length, ret_stats=None, gamma=0.99, epsilon=1e-8,
               clip_reward=10.0, totals=None):
    """qs_ppo_reward: ret_stats = (ret [N], ret_mean, ret_var, ret_count) float64 device tensors, or None for raw
    rewards; totals [4] float64 collects (episodes, sum of returns, sum of lengths) of the envs done in this step and
    the sum of every env's raw reward"""
    ret, m, v, c = ret_stats if ret_stats is not None else (None,) * 4
    _lib.check(_lib.lib().qs_ppo_reward(_a(reward), _a(done), int(reward.shape[0]), _a(ret), _a(m), _a(v), _a(c),
                                        float(gamma), float(epsilon), float(clip_reward), _a(reward_out),
                                        _a(ep_return), _a(ep_length), _a(totals), _stream_ptr(reward.device)))


def ppo_gae(rewards, values, episode_starts, last_values, last_dones, gamma, gae_lambda, advantages=None, returns=None):
    """qs_ppo_gae on step-major [n_steps, N] arrays -> (advantages, returns)"""
    T, n = int(rewards.shape[0]), int(rewards.shape[1])
    advantages = torch.empty_like(rewards) if advantages is None else advantages
    returns = torch.empty_like(rewards) if returns is None else returns
    _lib.check(_lib.lib().qs_ppo_gae(_a(rewards), _a(values), _a(episode_starts), _a(last_values), _a(last_dones), T, n,
                                     float(gamma), float(gae_lambda), _a(advantages), _a(returns),
                                     _stream_ptr(rewards.device)))
    return advantages, returns


# ----------------------------------------------------------------------------- the training half of ActorCriticPolicy
def ortho_init(policy):
    """ActorCriticPolicy._build with ortho_init: orthogonal weights with gain sqrt(2) in the extractor, 0.01 on
    action_net and 1 on value_net, zero biases; draws from torch's global CPU generator"""
    for module, gain in ((policy.mlp_extractor, math.sqrt(2)), (policy.action_net, 0.01), (policy.value_net, 1.0)):
        for m in module.modules():
            if isinstance(m, torch.nn.Linear):
                torch.nn.init.orthogonal_(m.weight, gain=gain)
                m.bias.data.fill_(0.0)


def evaluate_actions(policy, obs, actions):
    """ActorCriticPolicy.evaluate_actions with DiagGaussianDistribution: (values [B], log_prob [B], entropy [B])"""
    mean = policy.action_net(policy.mlp_extractor.policy_net(obs))
    values = policy.value_net(policy.mlp_extractor.value_net(obs)).flatten()
    dist = torch.distributions.Normal(mean, torch.ones_like(mean) * policy.log_std.exp())
    return values, dist.log_prob(actions).sum(dim=1), dist.entropy().sum(dim=1)


def explained_variance(y_pred, y_true):
    """stable_baselines3.common.utils.explained_variance (population variances)"""
    var_y = torch.var(y_true.double(), unbiased=False)
    if float(var_y) == 0.0:
        return float("nan")
    return float(1.0 - torch.var((y_true - y_pred).double(), unbiased=False) / var_y)


# ----------------------------------------------------------------------------- the trainer
class BatchedPPO:
    """stable_baselines3.PPO("MlpPolicy", env, learning_rate, n_steps, batch_size, n_epochs, gamma, gae_lambda, clip_range,
    clip_range_vf, normalize_advantage, ent_coef, vf_coef, max_grad_norm, target_kl, seed, policy_kwargs) over one
    BatchedQuadrupedGymEnv(auto_reset=True, **env_kwargs) of num_envs envs, wrapped in rl-zoo's
    VecNormalize(norm_obs=True, norm_reward=True, gamma=gamma) when `normalize`.

    The rollout buffer holds n_steps x num_envs samples (n_steps per env): keep n_steps small at large num_envs.
    learning_rate, clip_range and clip_range_vf are constants or callables of progress_remaining.  policy_kwargs:
    net_arch (one list for the actor and the critic, or {"pi": l, "vf": l} with equal lists; 0-2 hidden layers of at
    most 64), activation_fn (Tanh or ReLU), ortho_init, log_std_init.  The policy is an MlpPolicyTorch (`policy`)
    initialised from a CPU generator seeded with `seed`; its statistics are `vec_normalize`.  The env is created on
    the first rollout; the update, saving and loading need no GPU."""

    def __init__(self, policy="MlpPolicy", env_kwargs=None, num_envs=None, learning_rate=3e-4, n_steps=2048,
                 batch_size=64, n_epochs=10, gamma=0.99, gae_lambda=0.95, clip_range=0.2, clip_range_vf=None,
                 normalize_advantage=True, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, use_sde=False, target_kl=None,
                 normalize=True, seed=0, device="cuda", policy_kwargs=None, verbose=0):
        if policy != "MlpPolicy":
            raise ValueError(f"unknown policy {policy!r}: only 'MlpPolicy' is provided")
        if use_sde:
            raise ValueError("use_sde (generalised state-dependent exploration) is not provided")
        env_kwargs = dict(env_kwargs or {})
        n_env = env_kwargs.pop("num_envs", None)
        if num_envs is None:
            num_envs = n_env
        if num_envs is None or int(num_envs) < 1 or (n_env is not None and int(n_env) != int(num_envs)):
            raise ValueError(f"num_envs must be given once and be at least 1, got {num_envs} and env_kwargs {n_env}")
        for k in ("device", "seed", "auto_reset"):
            if k in env_kwargs:
                raise ValueError(f"env_kwargs[{k!r}] is set by the trainer")
        if env_kwargs.get("landing_wrapper") is not None:
            raise ValueError("landing_wrapper: the reference's landing wrappers run their scripted steps inside one "
                             "learner step, hidden from the learner; here they are ordinary control steps the policy's "
                             "samples would be credited with, so PPO does not train through them")
        n_steps, batch_size, n_epochs = int(n_steps), int(batch_size), int(n_epochs)
        if n_steps < 1 or batch_size < 1 or n_epochs < 1:
            raise ValueError("n_steps, batch_size and n_epochs must be at least 1")
        if normalize_advantage and batch_size < 2:
            raise ValueError("batch_size must be greater than 1 when advantages are normalised")
        pk = dict(DEFAULT_POLICY_KWARGS)
        for k, v in (policy_kwargs or {}).items():
            if k not in pk:
                raise ValueError(f"unknown policy_kwargs entry {k!r}")
            pk[k] = v
        na = pk["net_arch"]
        if isinstance(na, dict):
            if list(na.get("pi", [])) != list(na.get("vf", [])) or set(na) - {"pi", "vf"}:
                raise ValueError(f"net_arch {na}: the actor and the critic must share one architecture")
            na = na.get("pi", [])
        pk["net_arch"] = [int(h) for h in na]
        pk["activation_fn"] = _activation_name(pk["activation_fn"])
        pk["ortho_init"], pk["log_std_init"] = bool(pk["ortho_init"]), float(pk["log_std_init"])
        if len(pk["net_arch"]) > 2 or not all(1 <= h <= _lib.QS_ARS_MAX_HIDDEN for h in pk["net_arch"]):
            raise ValueError(f"net_arch {pk['net_arch']}: at most two hidden layers of 1..{_lib.QS_ARS_MAX_HIDDEN}")
        self.policy_kwargs, self.env_kwargs, self.num_envs = pk, env_kwargs, int(num_envs)
        self.learning_rate, self.clip_range, self.clip_range_vf = learning_rate, clip_range, clip_range_vf
        self.n_steps, self.batch_size, self.n_epochs = n_steps, batch_size, n_epochs
        self.gamma, self.gae_lambda = float(gamma), float(gae_lambda)
        self.normalize_advantage, self.ent_coef, self.vf_coef = bool(normalize_advantage), float(ent_coef), float(vf_coef)
        self.max_grad_norm, self.target_kl = float(max_grad_norm), target_kl
        self.normalize, self.seed, self.verbose = bool(normalize), int(seed), verbose
        self.device = torch.device(device)

        from .ops import make_config
        cfg = make_config(**{k: env_kwargs[k] for k in ("enable_springs", "motor_control_mode", "action_space_mode",
                                                         "task_env", "observation_space_mode") if k in env_kwargs},
                          is_rl_interface=int(bool(env_kwargs.get("isRLGymInterface", True))))
        L = _lib.lib()
        self.obs_dim, self.act_dim = int(L.qs_config_obs_dim(C.byref(cfg))), int(L.qs_config_action_dim(C.byref(cfg)))
        if self.act_dim > _lib.QS_ARS_MAX_ACT or self.obs_dim > _lib.QS_MAX_OBS:
            raise ValueError(f"the env has {self.obs_dim} observations and {self.act_dim} actions; qs_ppo_act takes at "
                             f"most {_lib.QS_MAX_OBS} and {_lib.QS_ARS_MAX_ACT}")
        self.arch = _lib.QsPpoArch(self.obs_dim, self.act_dim, len(pk["net_arch"]),
                                   (C.c_int32 * 2)(*(pk["net_arch"] + [0, 0])[:2]), _ACTIVATIONS[pk["activation_fn"]])
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(self.seed)
            net = self._new_policy("cpu")
            if pk["ortho_init"]:
                ortho_init(net)
        with torch.no_grad():
            net.log_std.fill_(pk["log_std_init"])
        self.policy = net.to(self.device)
        self.optimizer = torch.optim.Adam(self.policy.parameters(), lr=float(_schedule(learning_rate)(1.0)), eps=1e-5)

        shim = types.SimpleNamespace(num_envs=self.num_envs, observation_space=None, action_space=None,
                                     device=self.device, env=types.SimpleNamespace(obs_dim=self.obs_dim))
        self.vec_normalize = VecNormalizeTorch(shim, training=True, norm_obs=self.normalize,
                                               norm_reward=self.normalize, gamma=self.gamma)
        f64 = dict(dtype=torch.float64, device=self.device)
        self._obs_count = torch.tensor([self.vec_normalize.obs_rms.count], **f64)
        self._ret_count = torch.tensor([self.vec_normalize.ret_rms.count], **f64)
        self.num_timesteps, self._n_updates, self._iteration = 0, 0, 0
        self._progress_remaining = 1.0
        self.logs, self.buffer, self.env = [], None, None
        self._need_reset = True

    # ------------------------------------------------------------------ parameters
    def _new_policy(self, device):
        pk = self.policy_kwargs
        return MlpPolicyTorch(self.obs_dim, self.act_dim, tuple(pk["net_arch"]), pk["activation_fn"].lower()).to(device)

    def theta(self):
        """parameters_to_vector of the policy: the vector qs_ppo_act reads (layout in include/qs_b200.h)"""
        return parameters_to_vector(self.policy.parameters()).detach().contiguous()

    def schedules(self, progress_remaining):
        """(learning_rate, clip_range, clip_range_vf or None) at progress_remaining"""
        crvf = None if self.clip_range_vf is None else float(_schedule(self.clip_range_vf)(progress_remaining))
        return (float(_schedule(self.learning_rate)(progress_remaining)),
                float(_schedule(self.clip_range)(progress_remaining)), crvf)

    def permutation(self, update, epoch, size):
        """the minibatch order of one epoch: randperm(size) from a generator of the trainer's device keyed by
        (seed, update, epoch)"""
        g = torch.Generator(device=self.device)
        g.manual_seed((((self.seed & 0xFFFFFF) << 40) ^ ((int(update) & 0xFFFFFFF) << 12) ^ (int(epoch) & 0xFFF))
                      & 0x7FFFFFFFFFFFFFFF)
        return torch.randperm(size, generator=g, device=self.device)

    def _sync_counts(self):
        self.vec_normalize.obs_rms.count = float(self._obs_count.item())
        self.vec_normalize.ret_rms.count = float(self._ret_count.item())

    # ------------------------------------------------------------------ rollout
    def _get_env(self):
        if self.env is None:
            self.env = BatchedQuadrupedGymEnv(num_envs=self.num_envs, device=self.device, seed=self.seed,
                                              auto_reset=True, **self.env_kwargs)
            n, dev = self.num_envs, self.device
            self._term_obs = torch.zeros(n, self.obs_dim, device=dev)
            self.env.set_terminal_obs_buffer(self._term_obs)
            self._episode_start = torch.ones(n, dtype=torch.uint8, device=dev)
            self._ep_return = torch.zeros(n, dtype=torch.float64, device=dev)
            self._ep_length = torch.zeros(n, dtype=torch.int32, device=dev)
            self._totals = torch.zeros(4, dtype=torch.float64, device=dev)
            self._actions = torch.empty(n, self.act_dim, device=dev)
            self._last_values = torch.empty(n, device=dev)
            T, f = self.n_steps, dict(device=dev)
            self.buffer = {"obs": torch.zeros(T, n, self.obs_dim, **f), "actions": torch.zeros(T, n, self.act_dim, **f),
                           **{k: torch.zeros(T, n, **f) for k in ("rewards", "episode_starts", "values", "log_probs",
                                                                  "advantages", "returns")}}
        return self.env

    def _reset(self):
        """the first observation of learn(): env.reset(), statistics updated with it, episode starts set"""
        env = self._get_env()
        env.reset()
        if self.normalize:
            rms = self.vec_normalize.obs_rms
            obs_stats(env._obs, rms.mean, rms.var, self._obs_count)
        self.vec_normalize.returns.zero_()
        self._episode_start.fill_(1)
        self._ep_return.zero_()
        self._ep_length.zero_()
        self._need_reset = False

    def collect_rollouts(self):
        """OnPolicyAlgorithm.collect_rollouts: n_steps control steps of every env into `buffer`, then the advantages.
        Returns the rollout's totals (finished episodes, their sum of returns and of lengths, the sum of the raw rewards
        of every env and step) as a device tensor."""
        env = self._get_env()
        if self._need_reset:
            self._reset()
        vn, L, stream, T = self.vec_normalize, env._L, _stream_ptr(self.device), self.n_steps
        obs_rms, ret_rms = vn.obs_rms, vn.ret_rms
        stats = (obs_rms.mean, obs_rms.var) if self.normalize else None
        ret_stats = (vn.returns, ret_rms.mean, ret_rms.var, self._ret_count) if self.normalize else None
        b = self.buffer
        self._totals.zero_()
        theta = self.theta()
        # one argument struct for the rollout; per step only the step and two pointers change
        p, _ = ppo_act_args(self.arch, env._obs, theta, stats=stats, clip_obs=vn.clip_obs, epsilon=vn.epsilon,
                            seed=self.seed, iteration=self._iteration, n_steps=T, gamma=self.gamma,
                            terminal_obs=self._term_obs, buffers=b, actions=self._actions)
        args, arch = C.byref(p), C.byref(self.arch)
        first_start, done, trunc = _a(self._episode_start), _a(env._done), _a(env._trunc)
        step_args = [C.c_void_p(_a(x)) for x in (self._actions, env._obs, env._reward, env._done, env._trunc)]
        rows = list(b["rewards"])
        for t in range(T):
            p.step, p.episode_start, p.prev_truncated = t, first_start if t == 0 else done, None if t == 0 else trunc
            _lib.check(L.qs_ppo_act(args, arch, stream))
            _lib.check(L.qs_step(env._h, *step_args, stream))
            if self.normalize:
                obs_stats(env._obs, obs_rms.mean, obs_rms.var, self._obs_count)
            ppo_reward(env._reward, env._done, rows[t], self._ep_return, self._ep_length, ret_stats, self.gamma,
                       vn.epsilon, vn.clip_reward, self._totals)
        p.step, p.episode_start, p.prev_truncated, p.values_only = T, done, trunc, 1
        p.last_values = _a(self._last_values)
        _lib.check(L.qs_ppo_act(args, arch, stream))
        self._episode_start.copy_(env._done)
        env._last_host_obs = None
        self.num_timesteps += self.num_envs * T
        self._iteration += 1
        return self._totals

    def compute_advantages(self):
        """RolloutBuffer.compute_returns_and_advantage(last_values, dones) on the device (qs_ppo_gae)"""
        b = self.buffer
        ppo_gae(b["rewards"], b["values"], b["episode_starts"], self._last_values, self._episode_start, self.gamma,
                self.gae_lambda, b["advantages"], b["returns"])

    # ------------------------------------------------------------------ update
    def train(self):
        """PPO.train on `buffer` (step-major [n_steps, N] arrays; flat sample i is env i // n_steps, step
        i % n_steps, as SB3's swap_and_flatten orders them) at the current progress_remaining; returns the logs"""
        b, T = self.buffer, self.buffer["values"].shape[0]
        flat = {k: v.transpose(0, 1).reshape(v.shape[0] * v.shape[1], *v.shape[2:])
                for k, v in b.items() if k in ("obs", "actions", "values", "log_probs", "advantages", "returns")}
        size = flat["values"].shape[0]
        lr, clip_range, clip_range_vf = self.schedules(self._progress_remaining)
        for group in self.optimizer.param_groups:
            group["lr"] = lr
        pg_losses, value_losses, entropy_losses, clip_fractions = [], [], [], []
        approx_kl_divs, continue_training, loss = [], True, None
        params = list(self.policy.parameters())
        update = self._n_updates
        for epoch in range(self.n_epochs):
            approx_kl_divs = []
            perm = self.permutation(update, epoch, size)
            for start in range(0, size, self.batch_size):
                idx = perm[start:start + self.batch_size]
                obs, actions = flat["obs"][idx], flat["actions"][idx]
                old_values, old_log_prob = flat["values"][idx], flat["log_probs"][idx]
                advantages, returns = flat["advantages"][idx], flat["returns"][idx]
                values, log_prob, entropy = evaluate_actions(self.policy, obs, actions)
                if self.normalize_advantage and len(advantages) > 1:
                    advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
                ratio = torch.exp(log_prob - old_log_prob)
                policy_loss_1 = advantages * ratio
                policy_loss_2 = advantages * torch.clamp(ratio, 1 - clip_range, 1 + clip_range)
                policy_loss = -torch.min(policy_loss_1, policy_loss_2).mean()
                pg_losses.append(policy_loss.detach())
                clip_fractions.append(torch.mean((torch.abs(ratio - 1) > clip_range).float()).detach())
                if clip_range_vf is None:
                    values_pred = values
                else:
                    values_pred = old_values + torch.clamp(values - old_values, -clip_range_vf, clip_range_vf)
                value_loss = torch.nn.functional.mse_loss(returns, values_pred)
                value_losses.append(value_loss.detach())
                entropy_loss = -torch.mean(entropy)
                entropy_losses.append(entropy_loss.detach())
                loss = policy_loss + self.ent_coef * entropy_loss + self.vf_coef * value_loss
                with torch.no_grad():
                    log_ratio = log_prob - old_log_prob
                    approx_kl_div = torch.mean((torch.exp(log_ratio) - 1) - log_ratio)
                approx_kl_divs.append(approx_kl_div)
                if self.target_kl is not None and float(approx_kl_div) > 1.5 * self.target_kl:
                    continue_training = False
                    break
                self.optimizer.zero_grad()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(params, self.max_grad_norm)
                self.optimizer.step()
            self._n_updates += 1
            if not continue_training:
                break
        mean = lambda xs: float(torch.stack(xs).double().mean())
        logs = {"entropy_loss": mean(entropy_losses), "policy_gradient_loss": mean(pg_losses),
                "value_loss": mean(value_losses), "approx_kl": mean(approx_kl_divs),
                "clip_fraction": mean(clip_fractions), "loss": float(loss.detach()),
                "explained_variance": explained_variance(b["values"].flatten(), b["returns"].flatten()),
                "std": float(self.policy.log_std.detach().exp().mean()), "n_updates": self._n_updates,
                "learning_rate": lr, "clip_range": clip_range}
        if clip_range_vf is not None:
            logs["clip_range_vf"] = clip_range_vf
        return logs

    def train_iteration(self, total_timesteps=None):
        """one PPO iteration (collect_rollouts, GAE, train); progress_remaining = 1 - num_timesteps / total_timesteps
        after the rollout (1 when total_timesteps is None).  Returns its log record."""
        sync = torch.cuda.synchronize if self.device.type == "cuda" else (lambda: None)
        sync()
        t0 = time.perf_counter()
        totals = self.collect_rollouts()
        sync()
        t1 = time.perf_counter()
        self.compute_advantages()
        sync()
        t2 = time.perf_counter()
        if total_timesteps is not None:
            self._progress_remaining = 1.0 - float(self.num_timesteps) / float(total_timesteps)
        logs = self.train()
        sync()
        t3 = time.perf_counter()
        if self.normalize:
            self._sync_counts()
        episodes, ret_sum, len_sum, rew_sum = totals.tolist()
        env_steps = self.num_envs * self.n_steps
        rec = {"iteration": self._iteration, "num_timesteps": self.num_timesteps, "episodes": int(episodes),
               "ep_rew_mean": ret_sum / episodes if episodes else float("nan"),
               "ep_len_mean": len_sum / episodes if episodes else float("nan"),
               "reward_per_step": rew_sum / env_steps,
               **logs, "seconds": {"rollout": t1 - t0, "gae": t2 - t1, "update": t3 - t2},
               "env_steps_per_s": env_steps / (t3 - t0), "rollout_env_steps_per_s": env_steps / (t1 - t0)}
        self.logs.append(rec)
        if self.verbose:
            print(json.dumps(rec))
        return rec

    def learn(self, total_timesteps, callback=None, reset_num_timesteps=True):
        """PPO.learn: reset the env once, then iterations until num_timesteps >= total_timesteps (counted from the
        current num_timesteps when reset_num_timesteps is False); callback(trainer, record) after each, False stops"""
        if reset_num_timesteps:
            self.num_timesteps = 0
        else:
            total_timesteps += self.num_timesteps
        if reset_num_timesteps or self.env is None:
            self._need_reset = True
        while self.num_timesteps < total_timesteps:
            rec = self.train_iteration(total_timesteps)
            if callback is not None and callback(self, rec) is False:
                break
        return self

    # ------------------------------------------------------------------ evaluation
    def evaluate(self, n_envs, task=None, seed=None, go_to_rest_wrapper=False, max_steps=1500):
        """the deterministic policy with the statistics frozen, one episode per env, in the env load_model.replay builds
        from the saved directory (ground randomizer, `task`, default the training task): the array
        replay(log_dir, task, algo="ppo", n_envs, go_to_rest_wrapper, seed) returns"""
        kw = replay_env_kwargs(self.env_kwargs, task or self.env_kwargs.get("task_env", "NO_TASK"))
        kw.pop("render", None)
        venv = make_vec_env(kw, n_envs=n_envs, device=self.device, go_to_rest_wrapper=go_to_rest_wrapper,
                            seed=self.seed if seed is None else seed)
        try:
            if self.normalize:
                self._sync_counts()
            vn = VecNormalizeTorch(venv, training=False, norm_obs=self.normalize, norm_reward=False)
            vn.load_state_dict(self.vec_normalize.state_dict())
            return first_episode_returns(vn, self.policy, max_steps)
        finally:
            venv.close()

    # ------------------------------------------------------------------ rl-zoo directory
    def save(self, log_dir):
        """log_dir/QuadrupedSpring-v0/{args.yml, vecnormalize.pkl} and log_dir/best_model.zip (rl-zoo's layout, with
        SB3's policy.pth, policy.optimizer.pth and data)"""
        env_dir = os.path.join(log_dir, ENV_NAME)
        os.makedirs(env_dir, exist_ok=True)
        args = OrderedDict([("algo", "ppo"), ("env", ENV_NAME), ("env_kwargs", OrderedDict(sorted(self.env_kwargs.items()))),
                            ("n_timesteps", int(self.num_timesteps)), ("seed", self.seed)])
        with open(os.path.join(env_dir, "args.yml"), "w") as f:
            yaml.dump(args, f)
        if self.normalize:
            self._sync_counts()
        write_vecnormalize_pkl(os.path.join(env_dir, "vecnormalize.pkl"), self.vec_normalize.state_dict(),
                               self.num_envs, norm_obs=self.normalize, training=self.vec_normalize.training,
                               norm_reward=self.normalize)
        pk = self.policy_kwargs
        data = {"policy_class": {"__module__": "stable_baselines3.common.policies", "__name__": "ActorCriticPolicy"},
                "policy_kwargs": {"net_arch": {"pi": pk["net_arch"], "vf": pk["net_arch"]},
                                  "activation_fn": f"<class 'torch.nn.modules.activation.{pk['activation_fn']}'>",
                                  "ortho_init": pk["ortho_init"], "log_std_init": pk["log_std_init"]},
                "num_timesteps": int(self.num_timesteps), "_n_updates": int(self._n_updates),
                "iteration": int(self._iteration), "seed": self.seed, "n_envs": self.num_envs,
                "n_steps": self.n_steps, "batch_size": self.batch_size, "n_epochs": self.n_epochs,
                "gamma": self.gamma, "gae_lambda": self.gae_lambda, "ent_coef": self.ent_coef,
                "vf_coef": self.vf_coef, "max_grad_norm": self.max_grad_norm,
                "normalize_advantage": self.normalize_advantage, "target_kl": self.target_kl}
        sd = OrderedDict((k, v.detach().cpu().clone()) for k, v in self.policy.state_dict().items())
        pth, opt = io.BytesIO(), io.BytesIO()
        torch.save(sd, pth)
        torch.save(self.optimizer.state_dict(), opt)
        with zipfile.ZipFile(os.path.join(log_dir, "best_model.zip"), "w") as z:
            z.writestr("data", json.dumps(data, indent=4))
            z.writestr("policy.pth", pth.getvalue())
            z.writestr("policy.optimizer.pth", opt.getvalue())
        return log_dir

    def load(self, log_dir):
        """resume from a directory save() wrote: parameters, statistics, optimiser state and counters (the env and
        VecNormalize's per-env discounted returns are not part of the directory, as in SB3)"""
        path = os.path.join(log_dir, "best_model.zip")
        net = MlpPolicyTorch.from_sb3_zip(path, device="cpu")
        with zipfile.ZipFile(path) as z:
            data = json.loads(z.read("data").decode())
            opt = torch.load(io.BytesIO(z.read("policy.optimizer.pth")), map_location="cpu", weights_only=True)
        own = {k: tuple(v.shape) for k, v in self.policy.state_dict().items()}
        act = str(data.get("policy_kwargs", {}).get("activation_fn", ""))
        if {k: tuple(v.shape) for k, v in net.state_dict().items()} != own or self.policy_kwargs["activation_fn"] not in act:
            raise ValueError(f"{path} holds a different policy than this trainer's")
        self.policy.load_state_dict(net.state_dict())
        self.optimizer.load_state_dict(opt)
        st = read_vecnormalize_pkl(os.path.join(log_dir, ENV_NAME, "vecnormalize.pkl"))
        self.vec_normalize.load_state_dict(st)
        self._obs_count.fill_(float(st["obs_count"]))
        self._ret_count.fill_(float(st["ret_count"]))
        self.num_timesteps = int(data.get("num_timesteps", 0))
        self._n_updates = int(data.get("_n_updates", 0))
        self._iteration = int(data.get("iteration", 0))
        return self


__all__ = ["BatchedPPO", "ppo_act", "ppo_reward", "ppo_gae", "ortho_init", "evaluate_actions", "explained_variance"]
