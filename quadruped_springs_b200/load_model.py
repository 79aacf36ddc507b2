"""Replaying trained policies on the batched env: the reference's `load_model.py` without its dependencies.

/root/reference/quadruped_spring/load_model.py:66-134 reads an rl-baselines3-zoo log directory

    <src>/<env name>/args.yml          the env kwargs the policy was trained with            (:66-85)
    <src>/<env name>/vecnormalize.pkl  a pickled stable-baselines3 VecNormalize              (:58,114-116)
    <src>/best_model.zip               a PPO (stable-baselines3) or ARS (sb3-contrib) model  (:59,124)

builds `ObsFlatteningWrapper(GoToRestWrapper(QuadrupedGymEnv(**kwargs)))` through `make_vec_env`, and rolls
`model.predict(obs, deterministic=True)` (:88-134).  Neither stable-baselines3, sb3-contrib nor gym is a dependency of
this package, so the three files are read directly:

* `args.yml` with a YAML loader that knows the one Python tag rl-zoo writes (`collections.OrderedDict`) and nothing else;
* `vecnormalize.pkl` with a restricted unpickler: numpy arrays are rebuilt, every other class (VecNormalize,
  RunningMeanStd, gym spaces, random generators ...) becomes an inert attribute bag, so no foreign code runs;
* the model zip by key name (`policy.pth`): `MlpPolicyTorch` for PPO, `ArsPolicyTorch` for ARS.

Host-side glue over the C ABI; not part of the measured path.
"""
import io
import json
import os
import pickle
import zipfile
from collections import OrderedDict

import numpy as np
import torch
import yaml

from .vec_env import BatchedVecEnv, MlpPolicyTorch, VecNormalizeTorch

ENV_NAME = "QuadrupedSpring-v0"                      # load_model.py:42


# ----------------------------------------------------------------------------- args.yml (load_model.py:66-107)
class _ZooLoader(yaml.SafeLoader):
    """SafeLoader + `!!python/object/apply:collections.OrderedDict` (what rl-zoo's `yaml.dump(OrderedDict(...))` writes);
    the reference uses yaml.UnsafeLoader (:70), which would run arbitrary constructors"""


def _ordered_dict(loader, node):
    seq = loader.construct_sequence(node, deep=True)
    return OrderedDict((k, v) for k, v in (seq[0] if seq else []))


_ZooLoader.add_constructor("tag:yaml.org,2002:python/object/apply:collections.OrderedDict", _ordered_dict)
_ZooLoader.add_constructor("tag:yaml.org,2002:python/tuple", lambda l, n: tuple(l.construct_sequence(n, deep=True)))


def load_env_kwargs(src, env_name=ENV_NAME):
    """load_model.py:66-74: the args rl-zoo saved next to the model"""
    args_path = os.path.join(src, env_name, "args.yml")
    if not os.path.isfile(args_path):
        raise RuntimeError(f"{args_path} file not found.")
    with open(args_path, "r") as f:
        return yaml.load(f, Loader=_ZooLoader)


def adapt_args(kwargs):
    """load_model.py:102-106"""
    for e in ("add_noise", "enable_env_randomization", "aux_seed"):
        kwargs.pop(e, None)


def replay_env_kwargs(training_kwargs, task, render=False):
    """load_model.py:79-85: training kwargs -> the kwargs of the replay env (ground randomizer, the given task)"""
    env_kwargs = dict(training_kwargs)
    env_kwargs["render"] = render
    env_kwargs["env_randomizer_mode"] = "GROUND_RANDOMIZER"
    env_kwargs["task_env"] = task
    adapt_args(env_kwargs)
    return env_kwargs


def get_env_kwargs(src, task, render=False, env_name=ENV_NAME):
    """load_model.py:77-85: the training kwargs with the task / randomizer the replay wants"""
    env_kwargs = {}
    loaded_args = load_env_kwargs(src, env_name)
    if loaded_args.get("env_kwargs") is not None:
        env_kwargs = replay_env_kwargs(loaded_args["env_kwargs"], task, render)
    return env_kwargs


def make_vec_env(env_kwargs, n_envs=1, go_to_rest_wrapper=True, landing_wrapper=None, device="cuda", seed=0):
    """`make_vec_env(callable_env(kwargs), n_envs)` of load_model.py:88-99,113: one batched env stands for the DummyVecEnv of
    `n_envs` wrapped envs (GoToRestWrapper by default as upstream; the landing wrappers are the commented alternatives)"""
    return BatchedVecEnv(num_envs=n_envs, device=device, seed=seed, go_to_rest_wrapper=go_to_rest_wrapper,
                         landing_wrapper=landing_wrapper, **env_kwargs)


# ----------------------------------------------------------------------------- vecnormalize.pkl (load_model.py:114-116)
class _Bag:
    """what every non-numpy class of the pickle becomes: it keeps the attributes and runs nothing"""

    def __init__(self, *a, **k):
        pass

    def __setstate__(self, state):
        if isinstance(state, dict):
            self.__dict__.update(state)
        elif isinstance(state, tuple) and len(state) == 2 and isinstance(state[1], dict):   # (dict, slots)
            self.__dict__.update(state[0] or {})
            self.__dict__.update(state[1])
        else:
            self.__dict__["_state"] = state

    def __call__(self, *a, **k):          # a pickled function reference used as a constructor
        return _Bag()


def _bag_class(module, name):
    return type(name, (_Bag,), {"__module__": module})


class _RestrictedUnpickler(pickle.Unpickler):
    _NUMPY_OK = {
        ("numpy.core.multiarray", "_reconstruct"), ("numpy._core.multiarray", "_reconstruct"),
        ("numpy.core.multiarray", "scalar"), ("numpy._core.multiarray", "scalar"),
        ("numpy", "ndarray"), ("numpy", "dtype"), ("numpy.core.numeric", "_frombuffer"), ("numpy._core.numeric", "_frombuffer"),
    }

    def find_class(self, module, name):
        if (module, name) in self._NUMPY_OK:
            import importlib
            for mod in (module.replace("numpy.core", "numpy._core"), module.replace("numpy._core", "numpy.core")):
                try:
                    return getattr(importlib.import_module(mod), name)
                except (ImportError, AttributeError):
                    continue
            raise pickle.UnpicklingError(f"numpy has no {module}.{name}")
        if module == "collections" and name == "OrderedDict":
            return OrderedDict
        if module == "builtins" and name in ("dict", "list", "tuple", "set", "frozenset", "float", "int", "bool", "str",
                                               "bytes", "bytearray", "complex", "slice", "range", "object"):
            return getattr(__import__("builtins"), name)
        if module == "copyreg" and name == "_reconstructor":
            return lambda cls, base, state: cls()
        return _bag_class(module, name)


def read_vecnormalize_pkl(path):
    """-> dict of the statistics `VecNormalizeTorch.load_state_dict` takes, from an SB3 `VecNormalize.save()` pickle"""
    with open(path, "rb") as f:
        vn = _RestrictedUnpickler(f).load()
    g = vn.__dict__

    def rms(o):
        d = o.__dict__
        return np.asarray(d["mean"], np.float64), np.asarray(d["var"], np.float64), float(d["count"])

    om, ov, oc = rms(g["obs_rms"])
    rm, rv, rc = rms(g["ret_rms"])
    out = {"obs_mean": om, "obs_var": ov, "obs_count": oc, "ret_mean": float(rm), "ret_var": float(rv), "ret_count": rc}
    for k in ("clip_obs", "clip_reward", "gamma", "epsilon"):
        if k in g:
            out[k] = float(g[k])
    for k in ("norm_obs", "norm_reward", "training"):
        if k in g:
            out[k] = bool(g[k])
    return out


def load_vecnormalize(stats_path, venv, training=False, norm_reward=False):
    """`VecNormalize.load(stats_path, env)` + `env.training = False; env.norm_reward = False` (load_model.py:114-116)"""
    st = read_vecnormalize_pkl(stats_path)
    vn = VecNormalizeTorch(venv, training=training, norm_obs=st.get("norm_obs", True), norm_reward=norm_reward)
    if vn.obs_rms.mean.shape != tuple(np.shape(st["obs_mean"])):
        raise ValueError(f"vecnormalize.pkl holds statistics for observations of shape {np.shape(st['obs_mean'])}, "
                         f"the env produces {tuple(vn.obs_rms.mean.shape)}")
    vn.load_state_dict(st)
    return vn


# ----------------------------------------------------------------------------- ARS policies (sb3_contrib.ars.policies)
class ArsPolicyTorch(torch.nn.Module):
    """Inference of sb3-contrib's `ARSPolicy` / `ARSLinearPolicy`: `action_net = Sequential(create_mlp(obs_dim, act_dim,
    net_arch, activation_fn, squash_output))` -- Linear layers at the even indices (with or without bias), the
    activation between them, an optional final Tanh -- and `predict` = the network's output clipped to the action
    box.  Parameter names match the state dict of `ARS.save()` (`action_net.<i>.weight`)."""

    def __init__(self, obs_dim, act_dim, net_arch=(), activation="relu", with_bias=True, squash_output=False):
        super().__init__()
        act = {"tanh": torch.nn.Tanh, "relu": torch.nn.ReLU}[activation]
        layers, last = [], obs_dim
        for s in net_arch:
            layers += [torch.nn.Linear(last, s, bias=with_bias), act()]
            last = s
        layers.append(torch.nn.Linear(last, act_dim, bias=with_bias))
        if squash_output:
            layers.append(torch.nn.Tanh())
        self.action_net = torch.nn.Sequential(*layers)

    @torch.no_grad()
    def predict(self, obs, deterministic=True, generator=None):
        return self.action_net(obs).clamp(-1.0, 1.0)

    forward = predict

    @classmethod
    def from_sb3_zip(cls, path, device="cuda"):
        with zipfile.ZipFile(path) as z:
            sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
            data = json.loads(z.read("data").decode()) if "data" in z.namelist() else {}
        w = sorted((k for k in sd if k.startswith("action_net.") and k.endswith(".weight")), key=lambda k: int(k.split(".")[1]))
        if not w:
            raise ValueError("not an ARS policy: no action_net.<i>.weight in policy.pth")
        arch = tuple(int(sd[k].shape[0]) for k in w[:-1])
        obs_dim, act_dim = int(sd[w[0]].shape[1]), int(sd[w[-1]].shape[0])
        with_bias = w[0].replace(".weight", ".bias") in sd
        pk = data.get("policy_kwargs") if isinstance(data.get("policy_kwargs"), dict) else {}
        pclass = str(data.get("policy_class", ""))
        squash = bool(pk.get("squash_output", "Linear" not in pclass and bool(arch)))   # ARSPolicy: True, ARSLinearPolicy: False
        activation = "tanh" if "Tanh" in str(pk.get("activation_fn", "")) else "relu"
        pol = cls(obs_dim, act_dim, arch, activation, with_bias, squash)
        pol.load_state_dict({k: v for k, v in sd.items() if k in pol.state_dict()}, strict=True)
        return pol.to(device)


LEARNING_ALGS = {"ars": ArsPolicyTorch, "ppo": MlpPolicyTorch}      # load_model.py:35


def load_policy(model_path, algo="ppo", device="cuda"):
    """`LEARNING_ALGS[ALGO].load(model_path, env)` (load_model.py:124), inference half only"""
    return LEARNING_ALGS[algo].from_sb3_zip(model_path, device=device)


def replay(source_path, task, algo="ppo", model="best_model.zip", n_envs=1, device="cuda", max_steps=1500, **make_kwargs):
    """load_model.py:109-138 end to end: env from args.yml, VecNormalize statistics, policy; one deterministic episode
    per env.  Returns the undiscounted return of every env's first episode [n_envs] (numpy)."""
    env_kwargs = get_env_kwargs(source_path, task)
    env_kwargs.pop("render", None)
    venv = make_vec_env(env_kwargs, n_envs=n_envs, device=device, **make_kwargs)
    vn = load_vecnormalize(os.path.join(source_path, ENV_NAME, "vecnormalize.pkl"), venv)
    policy = load_policy(os.path.join(source_path, model), algo, device)
    ret = first_episode_returns(vn, policy, max_steps)
    venv.close()
    return ret


def first_episode_returns(vn, policy, max_steps=1500):
    """`model.predict(obs, deterministic=True)` on the normalised env until every env has finished its first episode
    (load_model.py:126-134): the undiscounted return of that episode per env [num_envs] (numpy)"""
    obs = vn.reset()
    ret = torch.zeros(vn.num_envs, device=obs.device)
    alive = torch.ones(vn.num_envs, dtype=torch.bool, device=obs.device)
    for _ in range(max_steps):
        obs, reward, done, _ = vn.step(policy.predict(obs, deterministic=True))
        ret += torch.where(alive, vn.get_original_reward(), torch.zeros_like(ret))
        alive &= ~done
        if not bool(alive.any()):
            break
    return ret.cpu().numpy()
