"""Batched PPO training (quadruped_springs_b200/ppo.py, csrc/qs_ppo.cu) against stable-baselines3's PPO, RolloutBuffer and
VecNormalize restated here in numpy / torch, MlpPolicyTorch and load_model.replay."""
import copy
import io
import math
import pickle

import numpy as np
import pytest
import torch

from quadruped_springs_b200 import load_model as lm
from quadruped_springs_b200.ars import _RunningMeanStdState, _SB3Pickler, _VecNormalizeState, write_vecnormalize_pkl
from quadruped_springs_b200.ppo import BatchedPPO, evaluate_actions, ppo_act, ppo_gae

ENV_KW = dict(task_env="JUMPING_IN_PLACE_PPO", observation_space_mode="PPO_BASIC", action_space_mode="SYMMETRIC",
              enable_springs=True, motor_control_mode="PD")
# bench.py configuration 3
CONFIG3 = dict(enable_springs=True, task_env="JUMPING_FORWARD", motor_control_mode="CARTESIAN_PD",
               action_space_mode="SYMMETRIC", observation_space_mode="ARS_BASIC")


def _cpu_trainer(**kw):
    kw.setdefault("env_kwargs", ENV_KW)
    kw.setdefault("num_envs", 8)
    return BatchedPPO("MlpPolicy", device="cpu", **kw)


# ----------------------------------------------------------------------------- numpy restatement of SB3
def _np_gae(rewards, values, episode_starts, last_values, dones, gamma, gae_lambda):
    """RolloutBuffer.compute_returns_and_advantage, as SB3 writes it, on float32 [n_steps, n_envs] arrays"""
    rewards, values, episode_starts = (np.asarray(x, np.float32) for x in (rewards, values, episode_starts))
    last_values, dones = np.asarray(last_values, np.float32), np.asarray(dones)
    buffer_size = rewards.shape[0]
    advantages = np.zeros_like(rewards)
    last_gae_lam = 0
    for step in reversed(range(buffer_size)):
        if step == buffer_size - 1:
            next_non_terminal = 1.0 - dones.astype(np.float32)
            next_values = last_values
        else:
            next_non_terminal = 1.0 - episode_starts[step + 1]
            next_values = values[step + 1]
        delta = rewards[step] + gamma * next_values * next_non_terminal - values[step]
        last_gae_lam = delta + gamma * gae_lambda * next_non_terminal * last_gae_lam
        advantages[step] = last_gae_lam
    return advantages, advantages + values


def _random_rollout(rng, T, n):
    rewards = rng.normal(0, 1, (T, n)).astype(np.float32)
    values = rng.normal(0, 1, (T, n)).astype(np.float32)
    starts = (rng.random((T, n)) < 0.15).astype(np.float32)
    last_values = rng.normal(0, 1, n).astype(np.float32)
    dones = rng.random(n) < 0.3
    dones[0] = True          # a done on the last step
    starts[:, 1] = 0.0       # an env with no episode boundary at all
    dones[1] = False
    return rewards, values, starts, last_values, dones


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_gae_restatement_closed_forms(seed):
    rng = np.random.default_rng(seed)
    T, n, gamma = 24, 40, 0.97
    rewards, values, starts, last_values, dones = _random_rollout(rng, T, n)
    # where the episode of (t, e) ends inside the buffer: the first later step that starts an episode
    for lam in (1.0, 0.0):
        adv, ret = _np_gae(rewards, values, starts, last_values, dones, gamma, lam)
        assert np.array_equal(ret, adv + values)
        for e in range(n):
            for t in range(T):
                if lam == 0.0:   # one-step TD error
                    if t == T - 1:
                        nxt = 0.0 if dones[e] else float(last_values[e])
                    else:
                        nxt = 0.0 if starts[t + 1, e] else float(values[t + 1, e])
                    want = float(rewards[t, e]) + gamma * nxt - float(values[t, e])
                else:            # discounted return to the episode's end (or the bootstrap) minus the value
                    g, k, want = 1.0, t, 0.0
                    while True:
                        want += g * float(rewards[k, e])
                        g *= gamma
                        if k == T - 1:
                            want += 0.0 if dones[e] else g * float(last_values[e])
                            break
                        if starts[k + 1, e]:
                            break
                        k += 1
                    want -= float(values[t, e])
                assert abs(float(adv[t, e]) - want) <= 2e-5 * (1 + abs(want)), (lam, t, e)


def _sb3_train(policy, opt, flat, perms, hp):
    """PPO.train's loop as SB3 writes it, over flat samples and given per-epoch permutations; returns its logs"""
    entropy_losses, pg_losses, value_losses, clip_fractions = [], [], [], []
    continue_training, n_updates = True, 0
    for group in opt.param_groups:
        group["lr"] = hp["lr"]
    clip_range, clip_range_vf = hp["clip_range"], hp["clip_range_vf"]
    for epoch in range(hp["n_epochs"]):
        approx_kl_divs = []
        indices = perms[epoch]
        start_idx = 0
        while start_idx < len(indices):
            idx = indices[start_idx:start_idx + hp["batch_size"]]
            start_idx += hp["batch_size"]
            obs, actions = flat["obs"][idx], flat["actions"][idx]
            mean = policy.action_net(policy.mlp_extractor.policy_net(obs))
            values = policy.value_net(policy.mlp_extractor.value_net(obs)).flatten()
            dist = torch.distributions.Normal(mean, torch.ones_like(mean) * policy.log_std.exp())
            log_prob, entropy = dist.log_prob(actions).sum(dim=1), dist.entropy().sum(dim=1)
            advantages = flat["advantages"][idx]
            if hp["normalize_advantage"] and len(advantages) > 1:
                advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
            ratio = torch.exp(log_prob - flat["log_probs"][idx])
            policy_loss_1 = advantages * ratio
            policy_loss_2 = advantages * torch.clamp(ratio, 1 - clip_range, 1 + clip_range)
            policy_loss = -torch.min(policy_loss_1, policy_loss_2).mean()
            pg_losses.append(policy_loss.item())
            clip_fractions.append(torch.mean((torch.abs(ratio - 1) > clip_range).float()).item())
            if clip_range_vf is None:
                values_pred = values
            else:
                old = flat["values"][idx]
                values_pred = old + torch.clamp(values - old, -clip_range_vf, clip_range_vf)
            value_loss = torch.nn.functional.mse_loss(flat["returns"][idx], values_pred)
            value_losses.append(value_loss.item())
            entropy_loss = -torch.mean(entropy)
            entropy_losses.append(entropy_loss.item())
            loss = policy_loss + hp["ent_coef"] * entropy_loss + hp["vf_coef"] * value_loss
            with torch.no_grad():
                log_ratio = log_prob - flat["log_probs"][idx]
                approx_kl_div = torch.mean((torch.exp(log_ratio) - 1) - log_ratio).cpu().numpy()
                approx_kl_divs.append(approx_kl_div)
            if hp["target_kl"] is not None and approx_kl_div > 1.5 * hp["target_kl"]:
                continue_training = False
                break
            opt.zero_grad()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(policy.parameters(), hp["max_grad_norm"])
            opt.step()
        n_updates += 1
        if not continue_training:
            break
    return {"entropy_loss": np.mean(entropy_losses), "policy_gradient_loss": np.mean(pg_losses),
            "value_loss": np.mean(value_losses), "approx_kl": np.mean(approx_kl_divs),
            "clip_fraction": np.mean(clip_fractions), "n_updates": n_updates}


TRAIN_CASES = {
    "partial_minibatch": dict(batch_size=16),
    "clip_range_vf": dict(batch_size=24, clip_range_vf=0.05),
    "target_kl_stops_first_epoch": dict(batch_size=16, learning_rate=3e-2, target_kl=1e-5),
    "schedules": dict(batch_size=32, learning_rate=lambda p: 1e-3 * p, clip_range=lambda p: 0.1 + 0.1 * p,
                      clip_range_vf=lambda p: 0.2 * p),
    "no_advantage_normalisation": dict(batch_size=16, normalize_advantage=False, ent_coef=0.01),
}


@pytest.mark.parametrize("case", sorted(TRAIN_CASES))
def test_train_matches_sb3_restatement(case):
    kw = dict(TRAIN_CASES[case])
    T, n = 5, 13                                        # 65 samples: minibatches of 16 leave a partial one of 1
    tr = _cpu_trainer(num_envs=n, n_steps=T, n_epochs=2, seed=4, **kw)
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for p in tr.policy.parameters():
            p.add_(torch.randn(p.shape, generator=g) * 0.05)
    O, A = tr.obs_dim, tr.act_dim
    obs = torch.randn(T, n, O, generator=g)
    actions = torch.randn(T, n, A, generator=g)
    with torch.no_grad():
        v0, lp0, _ = evaluate_actions(tr.policy, obs.reshape(-1, O), actions.reshape(-1, A))
    buf = {"obs": obs, "actions": actions, "values": v0.view(T, n) + 0.1 * torch.randn(T, n, generator=g),
           "log_probs": lp0.view(T, n) + (0.0 if "target_kl" in case else 0.05 * torch.randn(T, n, generator=g)),
           "advantages": torch.randn(T, n, generator=g), "returns": torch.randn(T, n, generator=g),
           "rewards": torch.zeros(T, n), "episode_starts": torch.zeros(T, n)}
    tr.buffer = buf
    tr._progress_remaining = 0.625
    policy = copy.deepcopy(tr.policy)
    opt = torch.optim.Adam(policy.parameters(), lr=1.0, eps=1e-5)
    # SB3's swap_and_flatten: [n_steps, n_envs, ...] -> [n_envs * n_steps, ...]
    flat = {k: torch.from_numpy(np.ascontiguousarray(v.numpy().swapaxes(0, 1).reshape(T * n, *v.shape[2:])))
            for k, v in buf.items()}
    perms = [tr.permutation(0, epoch, T * n) for epoch in range(2)]
    lr, cr, crvf = tr.schedules(0.625)
    if case == "schedules":
        assert (lr, cr, crvf) == (1e-3 * 0.625, 0.1 + 0.1 * 0.625, 0.2 * 0.625)
    hp = dict(lr=lr, clip_range=cr, clip_range_vf=crvf, n_epochs=2, batch_size=tr.batch_size,
              normalize_advantage=tr.normalize_advantage, ent_coef=tr.ent_coef, vf_coef=tr.vf_coef,
              max_grad_norm=tr.max_grad_norm, target_kl=tr.target_kl)
    ref = _sb3_train(policy, opt, flat, perms, hp)
    logs = tr.train()
    if "target_kl" in case:
        assert ref["n_updates"] == 1                # stopped in the first epoch, after at least one step
    assert logs["n_updates"] == ref["n_updates"] == tr._n_updates
    for k in ("entropy_loss", "policy_gradient_loss", "value_loss", "approx_kl", "clip_fraction"):
        np.testing.assert_allclose(logs[k], ref[k], rtol=1e-6, atol=1e-9, err_msg=k)
    for (name, a), b in zip(tr.policy.named_parameters(), policy.parameters()):
        np.testing.assert_allclose(a.detach().numpy(), b.detach().numpy(), rtol=1e-6, atol=1e-8, err_msg=name)
    assert logs["learning_rate"] == lr and logs["clip_range"] == cr
    assert logs["std"] == pytest.approx(float(policy.log_std.exp().mean()), rel=1e-6)


def parameters(policy):
    return torch.cat([p.detach().reshape(-1) for p in policy.parameters()])


def test_target_kl_stops_before_the_step():
    """a target_kl below the first minibatch's divergence: no optimiser step at all"""
    tr = _cpu_trainer(num_envs=4, n_steps=4, batch_size=8, target_kl=1e-12)
    g = torch.Generator().manual_seed(1)
    tr.buffer = {"obs": torch.randn(4, 4, tr.obs_dim, generator=g), "actions": torch.randn(4, 4, tr.act_dim, generator=g),
                 **{k: torch.randn(4, 4, generator=g) for k in ("values", "log_probs", "advantages", "returns")}}
    before = parameters(tr.policy).clone()
    logs = tr.train()
    assert torch.equal(parameters(tr.policy), before) and logs["n_updates"] == 1 and logs["approx_kl"] > 1.5e-12


@pytest.mark.parametrize("net_arch,act", [([64, 64], "Tanh"), ([32], "ReLU"), ([], "Tanh")])
def test_ortho_init(net_arch, act):
    tr = _cpu_trainer(policy_kwargs={"net_arch": net_arch, "activation_fn": act})
    pol = tr.policy
    checked = 0
    for module, gain in ((pol.mlp_extractor, math.sqrt(2)), (pol.action_net, 0.01), (pol.value_net, 1.0)):
        for m in module.modules():
            if isinstance(m, torch.nn.Linear):
                W = m.weight.detach().double()
                G = W @ W.T if W.shape[0] <= W.shape[1] else W.T @ W
                torch.testing.assert_close(G, gain ** 2 * torch.eye(G.shape[0], dtype=torch.float64), atol=1e-5 * gain ** 2,
                                           rtol=0)
                assert torch.count_nonzero(m.bias) == 0
                checked += 1
    assert checked == 2 * len(net_arch) + 2
    assert torch.count_nonzero(pol.log_std) == 0
    assert torch.equal(parameters(pol), parameters(_cpu_trainer(policy_kwargs={"net_arch": net_arch,
                                                                                "activation_fn": act}).policy))
    assert not torch.equal(parameters(pol), parameters(_cpu_trainer(seed=1, policy_kwargs={
        "net_arch": net_arch, "activation_fn": act}).policy))


@pytest.mark.parametrize("net_arch,act", [([64, 64], "Tanh"), ([48], "ReLU")])
def test_save_round_trip(tmp_path, net_arch, act):
    tr = _cpu_trainer(policy_kwargs={"net_arch": net_arch, "activation_fn": act}, seed=11)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for p in tr.policy.parameters():
            p.add_(torch.randn(p.shape, generator=g) * 0.1)
    tr.policy.log_std.grad = None
    loss = sum((p ** 2).sum() for p in tr.policy.parameters())
    loss.backward()
    tr.optimizer.step()                                  # Adam state to round-trip
    vn = tr.vec_normalize
    vn.obs_rms.mean = torch.randn(tr.obs_dim, generator=g, dtype=torch.float64)
    vn.obs_rms.var = torch.rand(tr.obs_dim, generator=g, dtype=torch.float64) + 0.1
    vn.ret_rms.mean = torch.tensor(0.3712345678901, dtype=torch.float64)
    vn.ret_rms.var = torch.tensor(2.7182818284590, dtype=torch.float64)
    tr._obs_count.fill_(123457.0001)
    tr._ret_count.fill_(9876.5)
    tr.num_timesteps, tr._n_updates, tr._iteration = 98765, 70, 7
    tr.save(str(tmp_path))

    net = lm.MlpPolicyTorch.from_sb3_zip(str(tmp_path / "best_model.zip"), device="cpu")
    for (k, v), (k2, v2) in zip(net.state_dict().items(), tr.policy.state_dict().items()):
        assert k == k2 and torch.equal(v, v2)
    x = torch.randn(16, tr.obs_dim, generator=g) * 3
    assert torch.equal(net.predict(x), tr.policy.predict(x))          # the activation is read back from `data`
    st = lm.read_vecnormalize_pkl(str(tmp_path / lm.ENV_NAME / "vecnormalize.pkl"))
    assert np.array_equal(st["obs_mean"], vn.obs_rms.mean.numpy()) and np.array_equal(st["obs_var"], vn.obs_rms.var.numpy())
    assert st["obs_count"] == 123457.0001 and st["ret_count"] == 9876.5
    assert st["ret_mean"] == 0.3712345678901 and st["ret_var"] == 2.7182818284590 and st["gamma"] == 0.99
    assert st["norm_obs"] is True and st["norm_reward"] is True
    args = lm.load_env_kwargs(str(tmp_path))
    assert args["algo"] == "ppo" and dict(args["env_kwargs"]) == ENV_KW

    back = _cpu_trainer(policy_kwargs={"net_arch": net_arch, "activation_fn": act}, seed=11).load(str(tmp_path))
    assert torch.equal(parameters(back.policy), parameters(tr.policy))
    sa, sb = back.optimizer.state_dict(), tr.optimizer.state_dict()
    assert sa["param_groups"] == sb["param_groups"]
    for k in sb["state"]:
        for f in sb["state"][k]:
            assert torch.equal(sa["state"][k][f], sb["state"][k][f]), (k, f)
    bvn = back.vec_normalize
    assert torch.equal(bvn.obs_rms.mean, vn.obs_rms.mean) and torch.equal(bvn.obs_rms.var, vn.obs_rms.var)
    assert float(bvn.ret_rms.mean) == 0.3712345678901 and float(bvn.ret_rms.var) == 2.7182818284590
    assert float(back._obs_count) == 123457.0001 and float(back._ret_count) == 9876.5
    assert (back.num_timesteps, back._n_updates, back._iteration) == (98765, 70, 7)
    with pytest.raises(ValueError):
        _cpu_trainer(policy_kwargs={"net_arch": [16]}).load(str(tmp_path))
    with pytest.raises(ValueError):
        _cpu_trainer(policy_kwargs={"net_arch": net_arch, "activation_fn": "ReLU" if act == "Tanh" else "Tanh"}).load(
            str(tmp_path))


def _parent_write_vecnormalize_pkl(path, state, num_envs, norm_obs=True, training=True):
    """write_vecnormalize_pkl as it was before the norm_reward keyword"""
    rms = lambda m, v, c: _RunningMeanStdState(mean=np.asarray(m, np.float64), var=np.asarray(v, np.float64), count=float(c))
    vn = _VecNormalizeState(
        obs_rms=rms(state["obs_mean"], state["obs_var"], state["obs_count"]),
        ret_rms=rms(state["ret_mean"], state["ret_var"], state["ret_count"]),
        clip_obs=float(state["clip_obs"]), clip_reward=float(state["clip_reward"]), gamma=float(state["gamma"]),
        epsilon=float(state["epsilon"]), training=bool(training), norm_obs=bool(norm_obs), norm_reward=False,
        num_envs=int(num_envs), norm_obs_keys=None)
    buf = io.BytesIO()
    _SB3Pickler(buf, protocol=4).dump(vn)
    with open(path, "wb") as f:
        f.write(buf.getvalue())


def test_ars_pickle_is_unchanged(tmp_path):
    from quadruped_springs_b200.ars import BatchedARS
    tr = BatchedARS("LinearPolicy", dict(ENV_KW, observation_space_mode="ARS_BASIC"), device="cpu")
    tr.vec_normalize.obs_rms.mean = torch.linspace(-1, 1, tr.obs_dim, dtype=torch.float64)
    st = tr.vec_normalize.state_dict()
    for norm_obs, training in ((True, True), (False, False)):
        _parent_write_vecnormalize_pkl(tmp_path / "a.pkl", st, 16, norm_obs, training)
        write_vecnormalize_pkl(tmp_path / "b.pkl", st, 16, norm_obs, training)
        assert (tmp_path / "a.pkl").read_bytes() == (tmp_path / "b.pkl").read_bytes()
    tr.save(str(tmp_path / "ars"))
    assert lm.read_vecnormalize_pkl(str(tmp_path / "ars" / lm.ENV_NAME / "vecnormalize.pkl"))["norm_reward"] is False


def test_bad_arguments_raise():
    _cpu_trainer()
    bad = [dict(use_sde=True), dict(env_kwargs=dict(ENV_KW, landing_wrapper="LandingWrapper2")),
           dict(policy_kwargs={"net_arch": [64, 64, 64]}), dict(policy_kwargs={"net_arch": [128]}),
           dict(policy_kwargs={"net_arch": {"pi": [64], "vf": [32]}}), dict(policy_kwargs={"activation_fn": "ELU"}),
           dict(policy_kwargs={"use_expln": True}), dict(num_envs=0), dict(n_steps=0), dict(batch_size=1),
           dict(env_kwargs=dict(ENV_KW, num_envs=16)), dict(env_kwargs=dict(ENV_KW, seed=3))]
    for kw in bad:
        with pytest.raises(ValueError):
            _cpu_trainer(**kw)
    with pytest.raises(ValueError, match="landing"):
        _cpu_trainer(env_kwargs=dict(ENV_KW, landing_wrapper="LandingWrapperBackflip"))
    with pytest.raises(ValueError):
        BatchedPPO("CnnPolicy", ENV_KW, num_envs=8, device="cpu")
    assert _cpu_trainer(policy_kwargs={"net_arch": {"pi": [32], "vf": [32]}}).policy_kwargs["net_arch"] == [32]
    assert _cpu_trainer(num_envs=None, env_kwargs=dict(ENV_KW, num_envs=16)).num_envs == 16


# ----------------------------------------------------------------------------- GPU
def _normalise(obs, mean, var, clip=10.0, eps=1e-8):
    """VecNormalizeTorch.normalize_obs"""
    return ((obs.double() - mean) / torch.sqrt(var + eps)).clamp(-clip, clip).float()


def _bits(t):
    return t.contiguous().view(torch.int32)


ARCHS = [([64, 64], "Tanh"), ([64, 64], "ReLU"), ([37], "Tanh"), ([], "Tanh")]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["PPO_BASIC", "ARS_BASIC"])
@pytest.mark.parametrize("action_mode", ["SYMMETRIC_NO_HIP", "SYMMETRIC", "DEFAULT"])
@pytest.mark.parametrize("net_arch,act", ARCHS)
def test_ppo_act_matches_torch(mode, action_mode, net_arch, act):
    dev = "cuda"
    tr = BatchedPPO("MlpPolicy", dict(ENV_KW, observation_space_mode=mode, action_space_mode=action_mode), num_envs=8,
                    policy_kwargs={"net_arch": net_arch, "activation_fn": act}, device=dev)
    assert tr.act_dim == {"SYMMETRIC_NO_HIP": 4, "SYMMETRIC": 6, "DEFAULT": 12}[action_mode]
    g = torch.Generator(device=dev).manual_seed(7)
    with torch.no_grad():
        for p in tr.policy.parameters():
            p.copy_(torch.randn(p.shape, device=dev, generator=g) * 0.1)
    n, O, A = 1000, tr.obs_dim, tr.act_dim
    obs = torch.randn(n, O, device=dev, generator=g) * 1.5 + 1
    mean = torch.randn(O, device=dev, dtype=torch.float64, generator=g) * 0.5
    var = torch.rand(O, device=dev, dtype=torch.float64, generator=g) + 0.5
    var[:2] = 0.01                                           # these columns often exceed clip_obs = 10
    buf = {"obs": torch.zeros(2, n, O, device=dev), "actions": torch.zeros(2, n, A, device=dev),
           **{k: torch.zeros(2, n, device=dev) for k in ("values", "log_probs", "episode_starts", "rewards")}}
    starts = (torch.rand(n, device=dev, generator=g) < 0.5).to(torch.uint8)
    mu = torch.empty(n, A, device=dev)
    acts = ppo_act(tr.arch, obs, tr.theta(), stats=(mean, var), seed=3, iteration=2, step=1, n_steps=2,
                   episode_start=starts, buffers=buf, mean_out=mu)
    x = _normalise(obs, mean, var)
    assert (x.abs() == 10).any()
    assert torch.equal(_bits(buf["obs"][1]), _bits(x))                       # bit-identical normalisation
    pol = tr.policy
    with torch.no_grad():
        ref_mean = pol.action_net(pol.mlp_extractor.policy_net(x))
        ref_v = pol.predict_values(x)
        torch.testing.assert_close(mu, ref_mean, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(buf["values"][1], ref_v, rtol=1e-5, atol=1e-6)
        a = buf["actions"][1]
        lp = torch.distributions.Normal(ref_mean, pol.log_std.exp()).log_prob(a).sum(1)
        torch.testing.assert_close(buf["log_probs"][1], lp, rtol=1e-5, atol=1e-5)
    assert torch.equal(acts, a.clamp(-1, 1))
    assert torch.equal(buf["episode_starts"][1], starts.float())
    assert torch.count_nonzero(buf["obs"][0]) == 0 and torch.count_nonzero(buf["rewards"]) == 0
    det = ppo_act(tr.arch, obs, tr.theta(), stats=(mean, var), deterministic=True)
    assert torch.equal(det, mu.clamp(-1, 1))                                  # clipped mean, the same rounding
    # no normalisation: the raw observation goes into the networks
    lv = torch.empty(n, device=dev)
    ppo_act(tr.arch, obs, tr.theta(), values_only=True, step=2, n_steps=2, last_values=lv)
    with pytest.raises(ValueError):   # the bootstrap row step - 1 would lie past the buffer
        ppo_act(tr.arch, obs, tr.theta(), values_only=True, step=3, n_steps=2, last_values=lv)
    with pytest.raises(ValueError):
        ppo_act(tr.arch, obs, tr.theta(), step=2, n_steps=2, episode_start=starts, buffers=buf)
    torch.testing.assert_close(lv, pol.predict_values(obs), rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_noise_is_batch_and_shard_invariant_and_normal():
    dev, n, T = "cuda", 65536, 16
    tr = BatchedPPO("MlpPolicy", dict(ENV_KW, action_space_mode="DEFAULT"), num_envs=n, device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    with torch.no_grad():
        tr.policy.log_std.copy_(torch.randn(tr.act_dim, device=dev, generator=g) * 0.3)
    theta = tr.theta()
    obs = torch.randn(n, tr.obs_dim, device=dev, generator=g)
    starts = torch.zeros(n, dtype=torch.uint8, device=dev)
    std = tr.policy.log_std.detach().exp()

    def eps(rows, step, offset=0, iteration=0):
        m = len(rows) if not isinstance(rows, slice) else obs[rows].shape[0]
        buf = {"obs": torch.empty(1, m, tr.obs_dim, device=dev), "actions": torch.empty(1, m, tr.act_dim, device=dev),
               **{k: torch.empty(1, m, device=dev) for k in ("values", "log_probs", "episode_starts", "rewards")}}
        mu = torch.empty(m, tr.act_dim, device=dev)
        ppo_act(tr.arch, obs[rows].contiguous(), theta, seed=5, env_id_offset=offset, iteration=iteration, step=0,
                n_steps=1, episode_start=starts[:m], buffers=buf, mean_out=mu)
        return buf["actions"][0], mu

    full, mu_full = eps(slice(0, n), 0)
    for e in torch.randint(0, n, (32,), generator=torch.Generator().manual_seed(2)).tolist() + [0, n - 1]:
        alone, mu = eps(slice(e, e + 1), 0, offset=e)
        assert torch.equal(_bits(alone[0]), _bits(full[e])) and torch.equal(_bits(mu[0]), _bits(mu_full[e])), e
    half = n // 2
    hi, _ = eps(slice(half, n), 0, offset=half)
    assert torch.equal(_bits(hi), _bits(full[half:]))
    assert not torch.equal(eps(slice(0, n), 0, iteration=1)[0], full)
    draws = []
    for t in range(T):
        a, mu = eps(slice(0, n), 0, iteration=t)   # (iteration, step) both key the stream; steps are checked below
        draws.append(((a - mu) / std).double())
    E = torch.stack(draws)                           # [T, n, A]
    assert abs(float(E.mean())) < 0.01 and abs(float(E.std()) - 1) < 0.01
    corr = lambda u, v: float(((u - u.mean()) * (v - v.mean())).mean() / (u.std() * v.std()))
    assert abs(corr(E[:, :-1], E[:, 1:])) < 0.01          # adjacent envs
    assert abs(corr(E[:-1], E[1:])) < 0.01                # adjacent iterations
    assert abs(corr(E[..., :-1], E[..., 1:])) < 0.01      # adjacent action entries
    steps = []
    for t in range(T):
        buf = {"obs": torch.empty(T, n, tr.obs_dim, device=dev), "actions": torch.empty(T, n, tr.act_dim, device=dev),
               **{k: torch.empty(T, n, device=dev) for k in ("values", "log_probs", "episode_starts", "rewards")}}
        ppo_act(tr.arch, obs, theta, seed=5, step=t, n_steps=T, episode_start=starts, buffers=buf, mean_out=mu_full)
        steps.append(((buf["actions"][t] - mu_full) / std).double())
    S = torch.stack(steps)
    assert abs(float(S.mean())) < 0.01 and abs(float(S.std()) - 1) < 0.01 and abs(corr(S[:-1], S[1:])) < 0.01


@pytest.mark.gpu
def test_rollout_matches_sb3_collect_rollouts():
    """one rollout of a 4096-env configuration-3 env with time limits of 0.25 s against a twin env driven by SB3's
    collect_rollouts + VecNormalize restated in torch, fed the kernel's actions"""
    from quadruped_springs_b200.vec_env import BatchedVecEnv, VecNormalizeTorch
    dev, n, T, gamma = "cuda", 4096, 64, 0.99
    kw = dict(CONFIG3, solver={"max_episode_time": 0.25})
    tr = BatchedPPO("MlpPolicy", kw, num_envs=n, n_steps=T, gamma=gamma, seed=3, device=dev)
    g = torch.Generator(device=dev).manual_seed(2)
    with torch.no_grad():                                   # actions of order one, so robots fall as well
        tr.policy.action_net.weight.copy_(torch.randn(tr.policy.action_net.weight.shape, device=dev, generator=g) * 0.5)
    totals = tr.collect_rollouts().clone()
    tr.compute_advantages()
    b = tr.buffer

    twin = BatchedVecEnv(num_envs=n, device=dev, seed=3, **kw)
    vn = VecNormalizeTorch(twin, gamma=gamma)
    obs = vn.reset()
    pol = tr.policy
    rewards = torch.zeros(T, n, device=dev)
    starts = torch.ones(n, device=dev)
    ep_ret = torch.zeros(n, dtype=torch.float64, device=dev)
    ep_len = torch.zeros(n, dtype=torch.int64, device=dev)
    n_trunc = n_done = 0
    ep_count, ep_sum, len_sum, rew_sum = 0, 0.0, 0, 0.0
    with torch.no_grad():
        for t in range(T):
            torch.testing.assert_close(b["obs"][t], obs, rtol=1e-5, atol=1e-6)
            assert torch.equal(b["episode_starts"][t], starts), t
            mean = pol.action_net(pol.mlp_extractor.policy_net(obs))
            torch.testing.assert_close(b["values"][t], pol.predict_values(obs), rtol=1e-5, atol=1e-6)
            a = b["actions"][t]
            lp = torch.distributions.Normal(mean, pol.log_std.exp()).log_prob(a).sum(1)
            torch.testing.assert_close(b["log_probs"][t], lp, rtol=1e-5, atol=1e-5)
            obs, rew, done, infos = vn.step(a.clamp(-1, 1))
            trunc = done & infos["TimeLimit.truncated"]
            tv = pol.predict_values(infos["terminal_observation"])
            rewards[t] = torch.where(trunc, rew + gamma * tv, rew)
            ep_ret += vn.get_original_reward().double()
            rew_sum += float(vn.get_original_reward().double().sum())
            ep_len += 1
            ep_count += int(done.sum())
            ep_sum += float(ep_ret[done].sum())
            len_sum += int(ep_len[done].sum())
            ep_ret[done], ep_len[done] = 0, 0
            n_trunc += int(trunc.sum())
            n_done += int(done.sum())
            starts = done.float()
        torch.testing.assert_close(tr._last_values, pol.predict_values(obs), rtol=1e-5, atol=1e-6)
    assert n_trunc > 0 and n_done > n_trunc, (n_trunc, n_done)
    torch.testing.assert_close(b["rewards"], rewards, rtol=1e-5, atol=1e-5)
    tr._sync_counts()
    for mine, ref in ((tr.vec_normalize.ret_rms, vn.ret_rms), (tr.vec_normalize.obs_rms, vn.obs_rms)):
        assert torch.allclose(mine.mean, ref.mean, rtol=1e-12, atol=1e-12 * float(ref.var.sqrt().max()))
        assert torch.allclose(mine.var, ref.var, rtol=1e-12, atol=0)
        assert mine.count == ref.count
    assert int(totals[0]) == ep_count == n_done
    assert float(totals[1]) == pytest.approx(ep_sum, rel=1e-9) and int(totals[2]) == len_sum
    assert float(totals[3]) == pytest.approx(rew_sum, rel=1e-9)
    # GAE of the rollout against the restatement
    adv, ret = _np_gae(b["rewards"].cpu().numpy(), b["values"].cpu().numpy(), b["episode_starts"].cpu().numpy(),
                       tr._last_values.cpu().numpy(), tr._episode_start.cpu().numpy().astype(bool), gamma, tr.gae_lambda)
    np.testing.assert_allclose(b["advantages"].cpu().numpy(), adv, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(b["returns"].cpu().numpy(), ret, rtol=1e-6, atol=1e-7)
    twin.close()
    tr.env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("T,n", [(32, 4096), (7, 1000), (1, 33)])
def test_gae_kernel_matches_restatement(T, n):
    rng = np.random.default_rng(T * n)
    rewards, values, starts, last_values, dones = _random_rollout(rng, T, n)
    d = lambda x: torch.as_tensor(x, device="cuda").contiguous()
    adv, ret = ppo_gae(d(rewards), d(values), d(starts), d(last_values), d(dones.astype(np.uint8)), 0.99, 0.95)
    ref_adv, ref_ret = _np_gae(rewards, values, starts, last_values, dones, 0.99, 0.95)
    np.testing.assert_allclose(adv.cpu().numpy(), ref_adv, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(ret.cpu().numpy(), ref_ret, rtol=1e-6, atol=1e-7)


def _state(tr):
    vn = tr.vec_normalize
    return (parameters(tr.policy).cpu(), vn.obs_rms.mean.cpu(), vn.obs_rms.var.cpu(), vn.obs_rms.count,
            float(vn.ret_rms.mean), float(vn.ret_rms.var), vn.ret_rms.count)


def _same(a, b):
    return all(torch.equal(x, y) if torch.is_tensor(x) else x == y for x, y in zip(a, b))


SMALL = dict(num_envs=1024, n_steps=16, batch_size=2048, n_epochs=3)
_LOG_KEYS = ("ep_rew_mean", "episodes", "policy_gradient_loss", "value_loss", "entropy_loss", "approx_kl",
             "clip_fraction", "explained_variance", "std")


@pytest.mark.gpu
def test_training_is_deterministic_and_resumes(tmp_path):
    def trainer(seed):
        return BatchedPPO("MlpPolicy", ENV_KW, seed=seed, device="cuda", **SMALL)

    a, b, c = trainer(1), trainer(1), trainer(2)
    la = [a.train_iteration() for _ in range(2)]
    lb = [b.train_iteration() for _ in range(2)]
    c.train_iteration()
    c.train_iteration()
    assert _same(_state(a), _state(b)) and not _same(_state(a), _state(c))
    for ra, rb in zip(la, lb):
        assert all(ra[k] == rb[k] or (ra[k] != ra[k] and rb[k] != rb[k]) for k in _LOG_KEYS)
    # save after one iteration, disturb the trainer (one more update), load, train one more: as two straight
    d = trainer(1)
    d.train_iteration()
    d.save(str(tmp_path))
    d.train()
    assert not _same(_state(d), _state(a))
    d.load(str(tmp_path))
    rd = d.train_iteration()
    assert _same(_state(d), _state(a))
    assert all(rd[k] == la[1][k] or (rd[k] != rd[k]) for k in _LOG_KEYS)
    for t in (a, b, c, d):
        t.env.close()


@pytest.mark.gpu
def test_save_then_replay_equals_evaluate(tmp_path):
    tr = BatchedPPO("MlpPolicy", ENV_KW, seed=5, device="cuda", **SMALL)
    tr.learn(2 * SMALL["num_envs"] * SMALL["n_steps"])
    tr.save(str(tmp_path))
    for task, seed in (("JUMPING_IN_PLACE_PPO", 7), ("JUMPING_IN_PLACE", 8)):
        rep = lm.replay(str(tmp_path), task, algo="ppo", n_envs=48, go_to_rest_wrapper=False, seed=seed)
        ev = tr.evaluate(48, task=task, seed=seed)
        assert rep.shape == (48,) and np.isfinite(rep).all()
        assert np.array_equal(rep.view(np.int32), ev.view(np.int32)), task
    tr.env.close()


# The learning smoke, measured on one B200 (1000 W; DESIGN.md section 7): JUMPING_IN_PLACE, PPO_BASIC, SYMMETRIC, PD with
# springs, 4096 envs, n_steps 32, batch_size 8192, n_epochs 5, learning_rate 1e-3, SB3's other defaults, seed 0, against
# a control with learning_rate 0 and the same seed (the same envs and noise; its policy never changes).  After 20
# iterations: raw reward per control step over the last 5 rollouts 8.0e-4 trained, 7.5e-5 control; the last rollout's
# ep_rew_mean 0.0746 trained, 0.0076 control; the deterministic evaluation over 256 envs 0.0 before, 0.0729 trained,
# 0.0 control.  The test takes about 10 s.
SMOKE = dict(env_kwargs=dict(ENV_KW, task_env="JUMPING_IN_PLACE"), num_envs=4096, n_steps=32, batch_size=8192,
             n_epochs=5, learning_rate=1e-3, seed=0, iterations=20)
SMOKE_MIN_GAIN = dict(reward_per_step=4e-4, ep_rew_mean=0.03, evaluation=0.03)   # measured 7.2e-4, 0.067, 0.073


@pytest.mark.gpu
def test_learning_smoke():
    import time
    t0 = time.perf_counter()
    cfg = dict(SMOKE)
    iters = cfg.pop("iterations")
    lr = cfg.pop("learning_rate")
    out = {}
    for name, rate in (("trained", lr), ("control", 0.0)):
        tr = BatchedPPO("MlpPolicy", device="cuda", learning_rate=rate, **cfg)
        before = float(tr.evaluate(256).mean())
        recs = [tr.train_iteration() for _ in range(iters)]
        out[name] = {"eval_before": before, "eval_after": float(tr.evaluate(256).mean()),
                     "reward_per_step": float(np.mean([r["reward_per_step"] for r in recs[-5:]])),
                     "ep_rew_mean": recs[-1]["ep_rew_mean"]}
        tr.env.close()
    took = time.perf_counter() - t0
    print({**out, "iterations": iters, "seconds": took})
    t, c = out["trained"], out["control"]
    assert t["eval_before"] == c["eval_before"]
    assert t["reward_per_step"] - c["reward_per_step"] > SMOKE_MIN_GAIN["reward_per_step"]
    assert t["ep_rew_mean"] - c["ep_rew_mean"] > SMOKE_MIN_GAIN["ep_rew_mean"]
    assert t["eval_after"] - t["eval_before"] > SMOKE_MIN_GAIN["evaluation"]
    assert t["eval_after"] - c["eval_after"] > SMOKE_MIN_GAIN["evaluation"]
    assert took < 60
