"""stable-baselines3-shaped front ends of the batched env (SURVEY.md section 8f rank 3).

The reference trains and replays its policies through SB3: `make_vec_env(callable_env, n_envs=1)` (a DummyVecEnv of
`ObsFlatteningWrapper(GoToRestWrapper(QuadrupedGymEnv(**kwargs)))`), `VecNormalize.load(stats_path, env)` with
`training = False`, `norm_reward = False`, and `PPO.load(...).predict(obs, deterministic=True)` in a loop
(/root/reference/quadruped_spring/load_model.py:88-138).  stable-baselines3 is not a dependency of this package
(and is not installed on the build image), so the three pieces are restated here against SB3's documented contracts:

* `BatchedVecEnv`       -- the VecEnv protocol (`reset`, `step_async`/`step_wait`, `step`, `get_attr`, `env_method`,
                           `infos[i]["terminal_observation"]`, `infos[i]["TimeLimit.truncated"]`) over ONE
                           `BatchedQuadrupedGymEnv`; numpy in / numpy out through `qs_step_host` (the end-to-end path),
                           or torch tensors in / out with no host round trip (`step_tensor`).
* `VecNormalizeTorch`   -- VecNormalize on the device: running mean / variance of the observations and of the discounted
                           return, clipping, `training` / `norm_obs` / `norm_reward` switches, state import / export.
* `MlpPolicyTorch`      -- the inference half of SB3's `ActorCriticPolicy` with the default `MlpExtractor`
                           (2 x 64 tanh, separate value net); loads the `policy.pth` of a `PPO.save()` zip without SB3.

None of this is on the measured hot path; the step itself is the C ABI's `qs_step` / `qs_step_host`.
"""
import io
import json
import zipfile

import numpy as np
import torch

from .env import BatchedQuadrupedGymEnv
from .render import tile_images


class BatchedVecEnv:
    """VecEnv protocol of stable-baselines3 (`stable_baselines3.common.vec_env.base_vec_env.VecEnv`) over a
    BatchedQuadrupedGymEnv.  `callable_env` of load_model.py:88-99 maps to kwargs: `go_to_rest_wrapper=True`,
    `landing_wrapper="LandingWrapper2"`, ...; the observation is already flat (ObsFlatteningWrapper)."""

    metadata = {"render.modes": ["rgb_array"]}

    def __init__(self, env=None, num_envs=None, device="cuda", render_env_ids=(0,), **env_kwargs):
        """render_env_ids: the envs whose follow-camera images get_images() / render() return."""
        if env is None:
            env = BatchedQuadrupedGymEnv(num_envs=num_envs, device=device, auto_reset=True, **env_kwargs)
        if not env._auto_reset:
            raise ValueError("a VecEnv resets finished envs inside step_wait: build the env with auto_reset=True")
        self.env = env
        self.num_envs = env.num_envs
        self.observation_space = env.observation_space
        self.action_space = env.action_space
        self.device = env.device
        self.render_env_ids = [int(i) for i in render_env_ids]
        if not self.render_env_ids or not all(0 <= i < env.num_envs for i in self.render_env_ids):
            raise ValueError(f"render_env_ids must be a non-empty list of env indices in [0, {env.num_envs})")
        n, o = env.num_envs, env.obs_dim
        self._term_obs = torch.zeros(n, o, device=env.device)
        env.set_terminal_obs_buffer(self._term_obs)
        pin = torch.cuda.is_available()
        self._host = (torch.empty(n, o, pin_memory=pin).numpy(), torch.empty(n, pin_memory=pin).numpy(),
                      torch.empty(n, dtype=torch.uint8, pin_memory=pin).numpy(),
                      torch.empty(n, dtype=torch.uint8, pin_memory=pin).numpy())
        self._actions = None

    # ------------------------------------------------------------------ numpy protocol
    def reset(self):
        return self.env.reset_host().copy()

    def step_async(self, actions):
        self._actions = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.num_envs, self.env.action_dim)

    def step_wait(self):
        obs, rew, done, trunc = self.env.step_host(self._actions, out=self._host)
        done = done.astype(bool)
        infos = [{} for _ in range(self.num_envs)]
        idx = np.flatnonzero(done)
        if len(idx):
            # only the finished rows cross the bus
            sel = torch.as_tensor(idx, device=self.device)
            term = self._term_obs.index_select(0, sel).cpu().numpy()
            for j, i in enumerate(idx):
                infos[i]["terminal_observation"] = term[j]
                infos[i]["TimeLimit.truncated"] = bool(trunc[i])
        return obs.copy(), rew.copy(), done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    # ------------------------------------------------------------------ tensor path (no host round trip)
    def reset_tensor(self):
        return self.env.reset()

    def step_tensor(self, actions):
        """actions [N, A] cuda tensor -> (obs, reward, done, infos) of tensors; infos["terminal_observation"] is the
        [N, O] buffer whose rows are valid where done."""
        obs, rew, done, infos = self.env.step(actions)
        infos = dict(infos)
        infos["terminal_observation"] = self._term_obs
        return obs, rew, done, infos

    # ------------------------------------------------------------------ the rest of the protocol
    def close(self):
        self.env.close()

    def seed(self, seed=None):
        """SB3 calls it once; the Philox key is fixed at construction (results are keyed by (seed, env id, episode))"""
        return [None] * self.num_envs

    def _indices(self, indices):
        if indices is None:
            return list(range(self.num_envs))
        if isinstance(indices, int):
            return [indices]
        return list(indices)

    def get_attr(self, attr_name, indices=None):
        v = getattr(self.env, attr_name)
        return [v for _ in self._indices(indices)]

    def _all_or_raise(self, indices, what):
        # one handle holds every env: an attribute or a method call cannot apply to a strict subset of them
        idx = self._indices(indices)
        if sorted(set(idx)) != list(range(self.num_envs)):
            raise ValueError(f"{what} applies to all {self.num_envs} envs of the batch; a subset of indices is not supported")
        return idx

    def set_attr(self, attr_name, value, indices=None):
        self._all_or_raise(indices, "set_attr")
        setattr(self.env, attr_name, value)

    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        idx = self._all_or_raise(indices, "env_method")
        r = getattr(self.env, method_name)(*method_args, **method_kwargs)
        return [r for _ in idx]

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False for _ in self._indices(indices)]

    def get_images(self):
        """One follow-camera image (numpy uint8 [360, 480, 3]) per env of render_env_ids (VecVideoRecorder's source)."""
        return list(self.env.render_images(self.render_env_ids)["rgb"].cpu().numpy())

    def render(self, mode="rgb_array"):
        """The images of get_images() tiled as stable-baselines3's VecEnv.render does (render.tile_images).  There is
        no GUI, so "rgb_array" is the only mode."""
        if mode != "rgb_array":
            raise NotImplementedError(f"render mode {mode!r} needs a GUI; only 'rgb_array' is provided")
        return tile_images(self.get_images())

    @property
    def unwrapped(self):
        return self


class RunningMeanStdTorch:
    """stable_baselines3.common.running_mean_std.RunningMeanStd (parallel-variance update, Chan et al.) in float64
    on the device."""

    def __init__(self, shape=(), device="cuda", epsilon=1e-4):
        self.mean = torch.zeros(shape, dtype=torch.float64, device=device)
        self.var = torch.ones(shape, dtype=torch.float64, device=device)
        self.count = float(epsilon)

    def update(self, x):
        x = x.to(torch.float64)
        if x.dim() == self.mean.dim():
            x = x[None]
        bv, bm = torch.var_mean(x, dim=0, unbiased=False)
        bc = x.shape[0]
        delta = bm - self.mean
        tot = self.count + bc
        m_a, m_b = self.var * self.count, bv * bc
        self.mean = self.mean + delta * bc / tot
        self.var = (m_a + m_b + delta * delta * self.count * bc / tot) / tot
        self.count = tot


class VecNormalizeTorch:
    """stable_baselines3.common.vec_env.VecNormalize on device tensors (load_model.py:113-116): observations
    `clip((obs - mean) / sqrt(var + eps), +-clip_obs)`, rewards `clip(r / sqrt(var_ret + eps), +-clip_reward)` with
    `ret = ret * gamma + r` zeroed on done; statistics update only while `training`."""

    def __init__(self, venv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8):
        self.venv = venv
        self.num_envs = venv.num_envs
        self.observation_space, self.action_space = venv.observation_space, venv.action_space
        dev = venv.device
        self.obs_rms = RunningMeanStdTorch((venv.env.obs_dim,), dev)
        self.ret_rms = RunningMeanStdTorch((), dev)
        self.returns = torch.zeros(self.num_envs, dtype=torch.float64, device=dev)
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.old_obs = self.old_reward = None

    def normalize_obs(self, obs):
        if not self.norm_obs:
            return obs
        o = (obs.to(torch.float64) - self.obs_rms.mean) / torch.sqrt(self.obs_rms.var + self.epsilon)
        return o.clamp(-self.clip_obs, self.clip_obs).to(torch.float32)

    def unnormalize_obs(self, obs):
        if not self.norm_obs:
            return obs
        return (obs.to(torch.float64) * torch.sqrt(self.obs_rms.var + self.epsilon) + self.obs_rms.mean).to(torch.float32)

    def normalize_reward(self, reward):
        if not self.norm_reward:
            return reward
        r = reward.to(torch.float64) / torch.sqrt(self.ret_rms.var + self.epsilon)
        return r.clamp(-self.clip_reward, self.clip_reward).to(torch.float32)

    def get_original_obs(self):
        return self.old_obs

    def get_original_reward(self):
        return self.old_reward

    def reset(self):
        obs = self.venv.reset_tensor()
        self.old_obs = obs.clone()
        self.returns.zero_()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)

    def step(self, actions):
        obs, rew, done, infos = self.venv.step_tensor(actions)
        self.old_obs, self.old_reward = obs.clone(), rew.clone()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        if self.training:
            self.returns = self.returns * self.gamma + rew.to(torch.float64)
            self.ret_rms.update(self.returns)
        out_rew = self.normalize_reward(rew)
        infos = dict(infos)
        infos["terminal_observation"] = self.normalize_obs(infos["terminal_observation"])
        self.returns = torch.where(done, torch.zeros_like(self.returns), self.returns)
        return self.normalize_obs(obs), out_rew, done, infos

    # ---- statistics I/O (the fields of SB3's vecnormalize.pkl)
    def state_dict(self):
        return {"obs_mean": self.obs_rms.mean.cpu().numpy(), "obs_var": self.obs_rms.var.cpu().numpy(),
                "obs_count": self.obs_rms.count, "ret_mean": float(self.ret_rms.mean), "ret_var": float(self.ret_rms.var),
                "ret_count": self.ret_rms.count, "clip_obs": self.clip_obs, "clip_reward": self.clip_reward,
                "gamma": self.gamma, "epsilon": self.epsilon}

    def load_state_dict(self, d):
        dev = self.returns.device
        self.obs_rms.mean = torch.as_tensor(np.asarray(d["obs_mean"], np.float64), device=dev)
        self.obs_rms.var = torch.as_tensor(np.asarray(d["obs_var"], np.float64), device=dev)
        self.obs_rms.count = float(d["obs_count"])
        self.ret_rms.mean = torch.as_tensor(float(d["ret_mean"]), dtype=torch.float64, device=dev)
        self.ret_rms.var = torch.as_tensor(float(d["ret_var"]), dtype=torch.float64, device=dev)
        self.ret_rms.count = float(d["ret_count"])
        for k in ("clip_obs", "clip_reward", "gamma", "epsilon"):
            if k in d:
                setattr(self, k, float(d[k]))


class MlpPolicyTorch(torch.nn.Module):
    """Inference half of SB3's ActorCriticPolicy with the default MlpExtractor: `net_arch` hidden layers with
    `activation_fn` for the actor (`mlp_extractor.policy_net`) and the critic (`mlp_extractor.value_net`), linear heads
    `action_net` / `value_net`, state-independent `log_std` (DiagGaussian).  `predict(obs, deterministic=True)` returns
    the clipped mean action like `BasePolicy.predict` (actions are clipped to the Box bounds, here +-1).
    Parameter names match SB3's state dict so that `policy.pth` of a `PPO.save()` archive loads unchanged."""

    def __init__(self, obs_dim, act_dim, net_arch=(64, 64), activation="tanh"):
        super().__init__()
        act = {"tanh": torch.nn.Tanh, "relu": torch.nn.ReLU}[activation]

        def mlp(sizes):
            layers, last = [], obs_dim
            for s in sizes:
                layers += [torch.nn.Linear(last, s), act()]
                last = s
            return torch.nn.Sequential(*layers), last

        class _Extractor(torch.nn.Module):
            pass

        self.mlp_extractor = _Extractor()
        self.mlp_extractor.policy_net, lp = mlp(net_arch)
        self.mlp_extractor.value_net, lv = mlp(net_arch)
        self.action_net = torch.nn.Linear(lp, act_dim)
        self.value_net = torch.nn.Linear(lv, 1)
        self.log_std = torch.nn.Parameter(torch.zeros(act_dim))

    @torch.no_grad()
    def predict(self, obs, deterministic=True, generator=None):
        mean = self.action_net(self.mlp_extractor.policy_net(obs))
        if not deterministic:
            mean = mean + torch.randn(mean.shape, device=mean.device, generator=generator) * self.log_std.exp()
        return mean.clamp(-1.0, 1.0)

    @torch.no_grad()
    def predict_values(self, obs):
        return self.value_net(self.mlp_extractor.value_net(obs)).squeeze(-1)

    forward = predict

    @classmethod
    def from_sb3_zip(cls, path, device="cuda"):
        """Load the policy of a `PPO.save(path)` archive: `policy.pth` (a torch state dict) and the `data` JSON
        (net_arch / activation_fn when present).  SB3 itself is not needed."""
        with zipfile.ZipFile(path) as z:
            sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
            arch, activation = None, "tanh"
            if "data" in z.namelist():
                data = json.loads(z.read("data").decode())
                pk = data.get("policy_kwargs", {})
                if isinstance(pk, dict):
                    na = pk.get("net_arch")
                    if isinstance(na, dict):
                        arch = tuple(na.get("pi", ()))
                    elif isinstance(na, list) and na and isinstance(na[-1], dict):
                        arch = tuple(na[-1].get("pi", ()))      # SB3 < 1.8: [dict(pi=[..], vf=[..])]
                    elif isinstance(na, list) and na:
                        arch = tuple(int(x) for x in na)
                    if "ReLU" in str(pk.get("activation_fn", "")):
                        activation = "relu"
        pi = sorted((k for k in sd if k.startswith("mlp_extractor.policy_net.") and k.endswith(".weight")),
                    key=lambda k: int(k.split(".")[2]))   # numeric layer order ("10" after "2")
        if arch is None:
            arch = tuple(sd[k].shape[0] for k in pi)
        obs_dim = sd[pi[0]].shape[1] if pi else sd["action_net.weight"].shape[1]
        act_dim = sd["action_net.weight"].shape[0]
        pol = cls(obs_dim, act_dim, arch, activation)
        own = pol.state_dict()
        pol.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=False)
        return pol.to(device)


class EvaluationWrapper:
    """env/wrappers/evaluation_wrapper.py:6-61 on the batch: `infos["feet_forces"]` (mean normal force over the four feet),
    `infos["max_height"]` and `infos["max_fwd"]` (running maxima of the base height and of the task's jumping distance;
    the height maximum restarts at reset, the distance maximum never does, as upstream :18-20,57-59).  The reference
    samples them at every substep through `set_sub_step_callback`; here they are sampled once per control step, from
    the state the step kernel leaves (a fused kernel cannot call back into Python between substeps)."""

    def __init__(self, env):
        if getattr(env, "_auto_reset", False):
            # with auto_reset the state read after step() already belongs to the next episode: the terminal height and
            # distance would be lost and max_height would run over episode boundaries
            raise ValueError("EvaluationWrapper evaluates episode by episode: build the env with auto_reset=False")
        self.env = env
        n, dev = env.num_envs, env.device
        self.max_h = torch.zeros(n, device=dev)
        self.max_fwd = torch.zeros(n, device=dev)

    def __getattr__(self, k):
        return getattr(self.env, k)

    def reset(self, mask=None, **k):
        if mask is None:
            self.max_h.zero_()
        else:
            self.max_h[torch.as_tensor(mask, device=self.env.device).bool()] = 0.0
        return self.env.reset(mask=mask, **k)

    def step(self, action):
        obs, reward, done, infos = self.env.step(action)
        infos = dict(infos)
        _, _, feet_forces, _ = self.env.robot.GetContactInfo()
        self.max_fwd = torch.maximum(self.max_fwd, self.env.task.compute_jumping_distance())
        self.max_h = torch.maximum(self.max_h, self.env.robot.GetBasePosition()[:, 2])
        infos["feet_forces"] = feet_forces.sum(-1) / 4
        infos["max_height"] = self.max_h
        infos["max_fwd"] = self.max_fwd
        return obs, reward, done, infos
