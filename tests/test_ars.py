"""Batched ARS training (quadruped_springs_b200/ars.py, csrc/qs_ars.cu) against sb3-contrib's ARS restated in numpy,
ArsPolicyTorch, RunningMeanStdTorch and load_model.replay."""
import numpy as np
import pytest
import torch
from torch.nn.utils import parameters_to_vector

from quadruped_springs_b200 import load_model as lm
from quadruped_springs_b200.ars import (BatchedARS, ars_act, candidate_returns, obs_stats, run_candidates)

ENV_KW = dict(task_env="JUMPING_IN_PLACE_PPO", observation_space_mode="ARS_BASIC", action_space_mode="SYMMETRIC",
              enable_springs=True, motor_control_mode="PD")
POLICY_VARIANTS = [("LinearPolicy", {}), ("LinearPolicy", {"with_bias": True}), ("MlpPolicy", {}),
                   ("MlpPolicy", {"with_bias": False}), ("MlpPolicy", {"activation_fn": "Tanh", "net_arch": [48]})]


def _cpu_trainer(policy="LinearPolicy", **kw):
    kw.setdefault("env_kwargs", ENV_KW)
    return BatchedARS(policy, device="cpu", **kw)


# ----------------------------------------------------------------------------- numpy restatement of sb3-contrib
def _np_do_one_update(theta, deltas, ret, lengths, n_delta, n_eval, n_top, lr, alive_bonus_offset):
    """ARS.evaluate_candidates (return bookkeeping) + ARS._do_one_update (the update), in numpy"""
    R = np.array([sum(ret[c * n_eval:(c + 1) * n_eval]) + alive_bonus_offset * sum(lengths[c * n_eval:(c + 1) * n_eval])
                  for c in range(2 * n_delta)], np.float32)
    plus, minus = R[:n_delta], R[n_delta:]
    top = np.maximum(plus, minus)
    idx = np.argsort(-top, kind="stable")[:n_top]
    plus, minus, d = plus[idx].astype(np.float64), minus[idx].astype(np.float64), deltas[idx].astype(np.float64)
    std = np.concatenate([plus, minus]).std(ddof=1)
    step = lr / (n_top * std + 1e-6)
    return theta.astype(np.float64) + step * ((plus - minus) @ d), std, step


@pytest.mark.parametrize("case", ["full", "top3", "top2_tied", "schedules_bonus"])
def test_update_matches_sb3_restatement(case):
    n_delta, n_eval = 8, 3
    kw = {"n_delta": n_delta, "n_eval_episodes": n_eval}
    if case == "top3":
        kw["n_top"] = 3
    if case == "top2_tied":
        kw["n_top"] = 2
    if case == "schedules_bonus":
        kw.update(n_top=5, learning_rate=lambda p: 0.02 * p, delta_std=lambda p: 0.01 + 0.04 * p, alive_bonus_offset=-0.5)
    tr = _cpu_trainer("MlpPolicy", **kw)
    rng = np.random.default_rng(3)
    theta0 = rng.normal(0, 0.3, tr.n_params).astype(np.float32)
    tr.theta = torch.tensor(theta0)
    deltas = rng.normal(0, 1, (n_delta, tr.n_params)).astype(np.float32)
    N = 2 * n_delta * n_eval
    ret = rng.normal(5, 2, N)
    lengths = rng.integers(50, 1000, N).astype(np.int32)
    if case == "top2_tied":
        # candidates 1 and 2 tie on max(plus, minus) at the n_top boundary, behind candidate 0
        ret[:] = 0.0
        ret[0 * n_eval] = 9.0
        ret[1 * n_eval] = 4.0
        ret[(n_delta + 2) * n_eval] = 4.0
        ret[(n_delta + 5) * n_eval] = 1.0
    progress = 0.375
    lr, dstd = tr.hyperparams(progress)
    if case == "schedules_bonus":
        assert (lr, dstd) == (0.02 * progress, 0.01 + 0.04 * progress)
    else:
        assert (lr, dstd) == (0.02, 0.05)
    R = candidate_returns(torch.tensor(ret), torch.tensor(lengths), 2 * n_delta, n_eval, tr.alive_bonus_offset)
    std, step = tr.update(torch.tensor(deltas), R, lr)
    ref, ref_std, ref_step = _np_do_one_update(theta0, deltas, ret, lengths, n_delta, n_eval, tr.n_top, lr,
                                               tr.alive_bonus_offset)
    assert tr._n_updates == 1
    np.testing.assert_allclose(std, ref_std, rtol=1e-6)
    np.testing.assert_allclose(step, ref_step, rtol=1e-6)
    np.testing.assert_allclose(tr.theta.numpy(), ref, rtol=1e-6, atol=1e-6 * np.abs(ref).max())
    if case == "top2_tied":   # the tie keeps the lower index: directions 0 and 1, not 2
        exp = theta0 + np.float32(step) * (9.0 * deltas[0] + 4.0 * deltas[1])
        np.testing.assert_allclose(tr.theta.numpy(), exp, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("policy,pk", POLICY_VARIANTS)
def test_parameter_vector_layout(policy, pk):
    """theta <-> ArsPolicyTorch state dict, both ways, bit for bit: layer by layer, weight [out, in] row-major, then bias"""
    tr = _cpu_trainer(policy, policy_kwargs=pk)
    theta = torch.randn(tr.n_params, generator=torch.Generator().manual_seed(1))
    sd = tr.policy_module(theta).state_dict()
    names = list(sd)
    layers = sorted({int(k.split(".")[1]) for k in names})
    expect = []
    for i in layers:
        expect.append(f"action_net.{i}.weight")
        if tr.policy_kwargs["with_bias"]:
            expect.append(f"action_net.{i}.bias")
    assert names == expect
    flat = torch.cat([sd[k].reshape(-1) for k in names])
    assert torch.equal(flat.view(torch.int32), theta.view(torch.int32))
    # and back: a policy's parameters_to_vector is the same concatenation
    net = tr._new_policy("cpu")
    assert torch.equal(parameters_to_vector(net.parameters()), torch.cat([v.reshape(-1) for v in net.state_dict().values()]))
    # the size qs_ars_act addresses deltas with
    a = tr.arch
    P, fan_in = 0, a.obs_dim
    for h in list(a.hidden)[:a.n_hidden] + [a.act_dim]:
        P += h * fan_in + (h if a.bias else 0)
        fan_in = h
    assert P == tr.n_params


@pytest.mark.parametrize("policy,pk", [POLICY_VARIANTS[0], POLICY_VARIANTS[2], POLICY_VARIANTS[4]])
def test_save_round_trip(tmp_path, policy, pk):
    tr = _cpu_trainer(policy, policy_kwargs=pk, n_delta=4, n_top=2, seed=11)
    g = torch.Generator().manual_seed(5)
    tr.theta = torch.randn(tr.n_params, generator=g)
    rms = tr.vec_normalize.obs_rms
    rms.mean = torch.randn(tr.obs_dim, generator=g, dtype=torch.float64)
    rms.var = torch.rand(tr.obs_dim, generator=g, dtype=torch.float64) + 0.1
    tr._count.fill_(123457.0001)
    tr.num_timesteps, tr._n_updates = 98765, 7
    tr.save(str(tmp_path))

    net = lm.ArsPolicyTorch.from_sb3_zip(str(tmp_path / "best_model.zip"), device="cpu")
    own = tr.policy_module()
    for (k, v), (k2, v2) in zip(net.state_dict().items(), own.state_dict().items()):
        assert k == k2 and torch.equal(v, v2)
    x = torch.randn(16, tr.obs_dim, generator=g) * 3
    assert torch.equal(net.predict(x), own.predict(x))   # same activation and squash read back from `data`
    st = lm.read_vecnormalize_pkl(str(tmp_path / lm.ENV_NAME / "vecnormalize.pkl"))
    assert np.array_equal(st["obs_mean"], rms.mean.numpy()) and np.array_equal(st["obs_var"], rms.var.numpy())
    assert st["obs_count"] == 123457.0001 and st["norm_obs"] is True and st["norm_reward"] is False
    assert dict(lm.load_env_kwargs(str(tmp_path))["env_kwargs"]) == ENV_KW
    assert lm.get_env_kwargs(str(tmp_path), "JUMPING_IN_PLACE")["task_env"] == "JUMPING_IN_PLACE"

    back = _cpu_trainer(policy, policy_kwargs=pk, n_delta=4, n_top=2, seed=11).load(str(tmp_path))
    assert torch.equal(back.theta, tr.theta)
    assert torch.equal(back.vec_normalize.obs_rms.mean, rms.mean) and torch.equal(back.vec_normalize.obs_rms.var, rms.var)
    assert float(back._count) == 123457.0001 and back.vec_normalize.obs_rms.count == 123457.0001
    assert (back.num_timesteps, back._n_updates) == (98765, 7)
    with pytest.raises(ValueError):
        _cpu_trainer("MlpPolicy" if policy == "LinearPolicy" else "LinearPolicy").load(str(tmp_path))


def test_bad_arguments_raise():
    with pytest.raises(ValueError):
        _cpu_trainer("CnnPolicy")
    for n_top in (0, 9):
        with pytest.raises(ValueError):
            _cpu_trainer(n_delta=8, n_top=n_top)
    with pytest.raises(ValueError):
        _cpu_trainer(n_delta=8, n_eval_episodes=2, env_kwargs=dict(ENV_KW, num_envs=16))
    assert _cpu_trainer(n_delta=8, n_eval_episodes=2, env_kwargs=dict(ENV_KW, num_envs=32)).num_envs == 32
    with pytest.raises(ValueError):
        _cpu_trainer("MlpPolicy", policy_kwargs={"net_arch": [64, 64, 64]})
    with pytest.raises(ValueError):
        _cpu_trainer("MlpPolicy", policy_kwargs={"net_arch": [128]})
    with pytest.raises(ValueError):
        _cpu_trainer("MlpPolicy", policy_kwargs={"activation_fn": "ELU"})
    with pytest.raises(ValueError):
        _cpu_trainer(env_kwargs=dict(ENV_KW, action_space_mode="DEFAULT", isRLGymInterface=True, seed=3))


# ----------------------------------------------------------------------------- GPU
def _normalise(obs, mean, var, clip=10.0, eps=1e-8):
    """VecNormalizeTorch.normalize_obs"""
    return ((obs.double() - mean) / torch.sqrt(var + eps)).clamp(-clip, clip).float()


def _candidate_theta(theta, deltas, delta_std, c):
    n_delta = deltas.shape[0]
    return theta + deltas[c] * delta_std if c < n_delta else theta - deltas[c - n_delta] * delta_std


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["ARS_BASIC", "ARS_SENSOR", "ARS_BACKFLIP"])
@pytest.mark.parametrize("policy,pk", POLICY_VARIANTS)
def test_ars_act_matches_ars_policy_torch(mode, policy, pk):
    dev = "cuda"
    tr = BatchedARS(policy, dict(ENV_KW, observation_space_mode=mode), n_delta=4, policy_kwargs=pk, device=dev)
    g = torch.Generator(device=dev).manual_seed(7)
    O, n_delta, epc, ds = tr.obs_dim, 4, 37, 0.05
    n = 2 * n_delta * epc - 5                      # the last candidate's group is cut short
    # activations of order 1, so that fp32 summation order stays far below the tolerance
    theta = torch.randn(tr.n_params, device=dev, generator=g) * 0.1
    deltas = torch.randn(n_delta, tr.n_params, device=dev, generator=g)
    obs = torch.randn(n, O, device=dev, generator=g) * 1.5 + 1
    mean = torch.randn(O, device=dev, dtype=torch.float64, generator=g) * 0.5
    var = torch.rand(O, device=dev, dtype=torch.float64, generator=g) + 0.5
    var[:2] = 0.01                                                 # these columns often exceed clip_obs = 10
    acts = ars_act(obs, theta, tr.arch, deltas, ds, n_delta, 0, epc, mean, var)
    x = _normalise(obs, mean, var)
    assert (x.abs() == 10).any()
    for c in range(2 * n_delta):
        rows = slice(c * epc, min((c + 1) * epc, n))
        net = tr.policy_module(_candidate_theta(theta, deltas, ds, c))
        raw = net.action_net(x[rows])
        ref = raw.clamp(-1, 1)
        torch.testing.assert_close(acts[rows], ref, rtol=1e-5, atol=1e-6)
        clipped = raw.abs() > 1 + 1e-4
        assert torch.equal(acts[rows][clipped], ref[clipped])   # clipping is exact
    # no normalisation, theta itself
    a0 = ars_act(obs, theta, tr.arch)
    torch.testing.assert_close(a0, tr.policy_module(theta).predict(obs), rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["LinearPolicy", "MlpPolicy"])
def test_ars_act_is_batch_invariant(policy):
    dev = "cuda"
    tr = BatchedARS(policy, ENV_KW, n_delta=8, device=dev)
    g = torch.Generator(device=dev).manual_seed(9)
    n, n_delta, epc = 65536, 8, 4096
    theta = torch.randn(tr.n_params, device=dev, generator=g) * 0.3
    deltas = torch.randn(n_delta, tr.n_params, device=dev, generator=g)
    obs = torch.randn(n, tr.obs_dim, device=dev, generator=g) * 2
    mean = torch.randn(tr.obs_dim, device=dev, dtype=torch.float64, generator=g) * 0.1
    var = torch.rand(tr.obs_dim, device=dev, dtype=torch.float64, generator=g) + 0.5
    full = ars_act(obs, theta, tr.arch, deltas, 0.05, n_delta, 0, epc, mean, var)
    bits = lambda t: t.view(torch.int32)
    for e in torch.randint(0, n, (48,), generator=torch.Generator().manual_seed(1)).tolist() + [0, n - 1, epc - 1, epc]:
        alone = ars_act(obs[e:e + 1].contiguous(), theta, tr.arch, deltas, 0.05, n_delta, e // epc, 1, mean, var)
        assert torch.equal(bits(alone[0]), bits(full[e])), e
    # two candidates' groups cut to 3000 envs each, started at candidate 5: every env keeps its bits
    part = torch.cat([torch.arange(5 * epc, 5 * epc + 3000), torch.arange(6 * epc, 6 * epc + 3000)]).to(dev)
    out = ars_act(obs[part].contiguous(), theta, tr.arch, deltas, 0.05, n_delta, 5, 3000, mean, var)
    assert torch.equal(bits(out), bits(full[part]))
    # rows shuffled within one candidate
    perm = torch.randperm(n, device=dev, generator=g)
    same = ars_act(obs[perm].contiguous(), theta, tr.arch, None, 0.0, n_delta, 0, n, mean, var)
    ref = ars_act(obs, theta, tr.arch, None, 0.0, n_delta, 0, n, mean, var)
    assert torch.equal(bits(same), bits(ref[perm]))


@pytest.mark.gpu
@pytest.mark.parametrize("n,O", [(65536, 20), (1000, 32), (7, 1)])
def test_obs_stats_matches_running_mean_std(n, O):
    from quadruped_springs_b200.vec_env import RunningMeanStdTorch
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(n + O)
    ref = RunningMeanStdTorch((O,), dev)
    mean, var = ref.mean.clone(), ref.var.clone()
    count = torch.tensor([ref.count], dtype=torch.float64, device=dev)
    offset = torch.randn(O, device=dev, generator=g) * 5
    scale = torch.rand(O, device=dev, generator=g) * 3 + 1e-3
    for it in range(5):
        obs = (torch.randn(n, O, device=dev, generator=g) * scale + offset).contiguous()
        alive = (torch.rand(n, device=dev, generator=g) < (1.0 if it == 0 else 0.3 + 0.15 * it)).to(torch.uint8)
        if it == 0:
            obs_stats(obs, mean, var, count)                 # alive None: every row
        else:
            obs_stats(obs, mean, var, count, alive=alive)
        rows = obs if it == 0 else obs[alive.bool()]
        if rows.shape[0]:
            ref.update(rows)
        col = ref.mean.abs() + ref.var.sqrt()
        assert (torch.abs(mean - ref.mean) <= 1e-12 * col).all(), (it, (mean - ref.mean).abs().max())
        assert (torch.abs(var - ref.var) <= 1e-12 * ref.var).all(), (it, ((var - ref.var) / ref.var).abs().max())
        assert float(count) == ref.count
    before = (mean.clone(), var.clone(), count.clone())
    obs_stats(obs, mean, var, count, alive=torch.zeros(n, dtype=torch.uint8, device=dev))
    for a, b in zip((mean, var, count), before):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_obs_stats_bookkeeping():
    dev, n = "cuda", 50000
    g = torch.Generator(device=dev).manual_seed(2)
    alive = (torch.rand(n, device=dev, generator=g) < 0.6).to(torch.uint8)
    ret = torch.randn(n, dtype=torch.float64, device=dev, generator=g)
    length = torch.randint(0, 100, (n,), dtype=torch.int32, device=dev, generator=g)
    reward = torch.randn(n, device=dev, generator=g)
    done = (torch.rand(n, device=dev, generator=g) < 0.2).to(torch.uint8)
    a0, r0, l0 = alive.bool().clone(), ret.clone(), length.clone()
    obs_stats(None, None, None, None, alive=alive, bookkeeping=(reward, done, ret, length))
    assert torch.equal(ret, torch.where(a0, r0 + reward.double(), r0))
    assert torch.equal(length, torch.where(a0, l0 + 1, l0))
    assert torch.equal(alive.bool(), a0 & ~done.bool())


def _small_env(tr, n_envs, offset):
    from quadruped_springs_b200 import BatchedQuadrupedGymEnv
    return BatchedQuadrupedGymEnv(num_envs=n_envs, device=tr.device, seed=tr.seed, env_id_offset=offset, auto_reset=True,
                                  **tr.env_kwargs)


@pytest.mark.gpu
@pytest.mark.parametrize("frozen_stats", [False, True])
def test_candidate_alone_matches_batched_iteration(frozen_stats):
    n_delta, n_eval = 4, 8
    tr = BatchedARS("MlpPolicy", ENV_KW, n_delta=n_delta, n_eval_episodes=n_eval, normalize=frozen_stats,
                    zero_policy=False, seed=3, device="cuda")
    if frozen_stats:
        g = torch.Generator(device="cuda").manual_seed(4)
        rms = tr.vec_normalize.obs_rms
        rms.mean = torch.randn(tr.obs_dim, dtype=torch.float64, device="cuda", generator=g) * 0.2
        rms.var = torch.rand(tr.obs_dim, dtype=torch.float64, device="cuda", generator=g) + 0.2
        tr.vec_normalize.training = False
    theta0 = tr.theta.clone()
    stats0 = tuple(t.clone() for t in tr._stats()) if frozen_stats else None
    tr.train_iteration()
    ro = tr.last_rollout
    if frozen_stats:   # frozen: the iteration did not touch them
        assert all(torch.equal(a, b) for a, b in zip(tr._stats(), stats0))
    _, dstd = tr.hyperparams(1.0)
    for c in (0, 3, 5, 2 * n_delta - 1):
        env = _small_env(tr, n_eval, c * n_eval)
        ret, length, _ = run_candidates(env, theta0, tr.arch, ro["deltas"], dstd, n_delta, c, n_eval, stats=stats0)
        rows = slice(c * n_eval, (c + 1) * n_eval)
        assert torch.equal(length, ro["length"][rows]), c
        assert torch.equal(ret.view(torch.int64), ro["return"][rows].view(torch.int64)), c
        env.close()
    assert (ro["length"] > 0).all()


@pytest.mark.gpu
def test_training_is_deterministic():
    def run(seed):
        tr = BatchedARS("LinearPolicy", ENV_KW, n_delta=4, n_eval_episodes=16, seed=seed, device="cuda")
        for _ in range(3):
            tr.train_iteration()
        rms = tr.vec_normalize.obs_rms
        out = (tr.theta.clone(), rms.mean.clone(), rms.var.clone(), rms.count, tr.num_timesteps)
        tr.env.close()
        return out

    a, b, c = run(1), run(1), run(2)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    assert a[3] == b[3] and a[4] == b[4]
    assert not torch.equal(a[0], c[0])


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["LinearPolicy", "MlpPolicy"])
def test_save_then_replay_equals_evaluate(tmp_path, policy):
    tr = BatchedARS(policy, ENV_KW, n_delta=4, n_eval_episodes=8, seed=5, device="cuda")
    tr.learn(1)   # one iteration
    tr.train_iteration()
    tr.save(str(tmp_path))
    for task, seed in (("JUMPING_IN_PLACE_PPO", 7), ("JUMPING_IN_PLACE", 8)):
        rep = lm.replay(str(tmp_path), task, algo="ars", n_envs=48, go_to_rest_wrapper=False, seed=seed)
        ev = tr.evaluate(48, task=task, seed=seed)
        assert rep.shape == (48,) and np.isfinite(rep).all()
        assert np.array_equal(rep.view(np.int32), ev.view(np.int32)), task


# The learning smoke, chosen on one B200 (1000 W; DESIGN.md section 7): JUMPING_IN_PLACE, ARS_BASIC, SYMMETRIC, PD with
# springs, the linear policy, n_delta = 8, n_eval_episodes = 256 (4096 envs), sb3-contrib's other defaults, seed 0.
# The deterministic evaluation over 256 envs returned 0.0 for the zero policy and 0.1308 after 10 iterations, in 12 s.
# (On JUMPING_IN_PLACE_PPO the zero policy, which holds the init pose, out-scores every candidate of the first 20
# iterations, so that task does not show learning this early.)
SMOKE = dict(policy="LinearPolicy", env_kwargs=dict(ENV_KW, task_env="JUMPING_IN_PLACE"), n_delta=8, n_eval_episodes=256,
             seed=0, iterations=10)


@pytest.mark.gpu
def test_learning_smoke():
    import time
    t0 = time.perf_counter()
    cfg = dict(SMOKE)
    iters = cfg.pop("iterations")
    tr = BatchedARS(cfg.pop("policy"), cfg.pop("env_kwargs"), device="cuda", **cfg)
    zero = tr.evaluate(256).mean()
    for _ in range(iters):
        tr.train_iteration()
    trained = tr.evaluate(256).mean()
    took = time.perf_counter() - t0
    print({"zero_policy_return": float(zero), "trained_return": float(trained), "iterations": iters, "seconds": took})
    assert trained > zero
    assert took < 60
