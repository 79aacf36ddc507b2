"""The step at the benchmark's size (65536 envs of configuration 3 on one GPU) and the routes that only run there.

At that size the step takes routes that the smaller tests never see: more airborne envs than one wave of the flight
kernel takes (the rest ride with k_step_contact, which runs the contact instantiation of the tick), the general solver
with 32 envs per warp, settle-conveyor windows that wrap the queue, and the host path's side buffer at n / 16 rows.
Which envs overflow the flight list follows the order of k_pre's atomics, so it changes from run to run: results are
deterministic and shard-invariant only if every route gives the same bits.  These tests force each route with the
library's environment switches and require bit-identical results, and hold the step's ticks and the conveyor's
episode starts at that size against the oracle.  Each test prints one JSON line with what it covered."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

from conftest import load_golden
from test_substep_trace import CFG3, FOOT_LINKS, OracleTicks, _TickCompare

pytestmark = pytest.mark.gpu

N_FULL = 65536
OUT_NAMES = ("obs", "reward", "done", "truncated")
STATE_KEYS = ("state", "tau_motor", "tau_spring", "foot_force", "contact", "task", "env_steps")
URDF_LO = np.array([-1.0471975512, -0.663225115758, -2.72271363311] * 4)   # go1.urdf joint limits
URDF_HI = np.array([1.0471975512, 2.96705972839, -0.837758040957] * 4)


@pytest.fixture(scope="module")
def qs():
    import quadruped_springs_b200 as m
    assert torch.cuda.is_available()
    return m


def _flight_cap():
    """the flight kernel's default list length: one wave of its blocks (2 blocks of 128 threads per SM)"""
    return torch.cuda.get_device_properties(0).multi_processor_count * 2 * 128


def _counters(env):
    """qs_debug_counters: envs in the general solver, urgent settles, conveyor entries in flight, last slice"""
    out = (C.c_int32 * 4)()
    env._L.qs_debug_counters(env._h, out, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    return list(out)


def _make(qs, monkeypatch, env_vars=None, **kw):
    """an env of configuration 3 created under the library switches `env_vars` (qs_create reads them)"""
    env_vars = env_vars or {}
    for k, v in env_vars.items():
        monkeypatch.setenv(k, str(v))
    try:
        return qs.BatchedQuadrupedGymEnv(auto_reset=True, enable_noise=True, **CFG3, **kw)
    finally:
        for k in env_vars:
            monkeypatch.delenv(k)


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b):
    """bit equality (a NaN equals the same NaN)"""
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _first_diff(a, b):
    """where two equally shaped tensors first differ (flat index into a's shape) and the two values"""
    d = (_bits(a) != _bits(b)).flatten().nonzero()
    if len(d) == 0:
        return None
    i = int(d[0])
    idx = np.unravel_index(i, tuple(a.shape))
    return dict(index=[int(x) for x in idx], got=float(b.flatten()[i]), want=float(a.flatten()[i]), count=len(d))


def _step(env, path, a_dev, a_np):
    """one control step through the device-buffer graph ("graph") or the end-to-end numpy path ("host"): the
    outputs as device tensors"""
    if path == "graph":
        o, r, d, info = env.step(a_dev)
        return o, r, d, info["TimeLimit.truncated"]
    o, r, d, t = env.step_host(a_np)
    dev = env.device
    return (torch.from_numpy(o).to(dev), torch.from_numpy(r).to(dev), torch.from_numpy(d).to(dev).bool(),
            torch.from_numpy(t).to(dev).bool())


class _Lockstep:
    """Steps a reference env and followers with the same actions.  A follower covers the global env ids `sl` of the
    reference (a shard) and gets those rows of the actions.  After every step its obs, reward, done and truncated must
    equal the reference's rows bit for bit; every `every` steps and when it stops, its state, torques, foot forces,
    contact words, task slots and step counters too.  With traces set (`trace`), the tick rows of every traced env must
    be equal as well, so that a failure names the env, the tick and the quantity.  The envs run side by side: 65536
    envs times 150 steps of outputs would not fit in host memory."""

    def __init__(self, ref, every=25):
        self.ref, self.every, self.t = ref, every, 0
        self.followers = []
        self.ref_trace = None

    def add(self, name, env, sl=None, path="graph", steps=None, watch=None, trace=None):
        """steps: the follower stops after that many steps, once `watch` (called with the env after each of its steps)
        has returned True"""
        self.followers.append(dict(name=name, env=env, sl=sl if sl is not None else slice(0, env.num_envs), path=path,
                                   steps=steps, watch=watch, trace=trace))

    def check_state(self, f):
        for key in STATE_KEYS:
            want, got = self.ref._views[key][..., f["sl"]], f["env"]._views[key]
            assert _same(want, got), (f["name"], self.t, key, _first_diff(want, got))

    def step(self, a_np, ref_path="graph"):
        a_dev = torch.from_numpy(a_np).to(self.ref.device)
        out = _step(self.ref, ref_path, a_dev, a_np)
        for f in self.followers:
            if f["env"] is None:
                continue
            sl = f["sl"]
            got = _step(f["env"], f["path"], a_dev[sl].contiguous(), np.ascontiguousarray(a_np[sl]))
            for name, x, y in zip(OUT_NAMES, out, got):
                assert _same(x[sl], y), (f["name"], self.t, name, _first_diff(x[sl], y))
            if f["trace"] is not None:
                want = self.ref_trace[:, :, sl]
                if not _same(want, f["trace"]):
                    tick, row, col = _first_diff(want, f["trace"])["index"]
                    raise AssertionError(dict(variant=f["name"], step=self.t, tick=tick, row=row, env=sl.start + col,
                                              got=float(f["trace"][tick, row, col]), want=float(want[tick, row, col])))
        self.t += 1
        for f in self.followers:
            if f["env"] is None:
                continue
            ok = f["watch"](f["env"]) if f["watch"] is not None else True
            last = f["steps"] is not None and self.t >= f["steps"] and ok
            if self.t % self.every == 0 or last:
                self.check_state(f)
            if last:
                f["env"].close()
                f["env"] = None
        return out

    def finish(self):
        for f in self.followers:
            if f["env"] is not None:
                self.check_state(f)


def _actions(rng, n, adim):
    return rng.uniform(-1, 1, (n, adim)).astype(np.float32)


# ------------------------------------------------------------------ routes
def test_dispatch_routes_are_bit_identical(qs, monkeypatch):
    """4096 envs, 200 steps, every env traced: the default dispatch against each forced route -- everything through
    k_step_contact (flight cap 0), a flight cap that cuts inside a warp and off a block boundary (1000), the general
    solver at 1, 2, 8 and 32 envs per warp, the epilogue without programmatic dependent launch, direct launches
    instead of the step's graph.  Results and tick rows are bit-identical."""
    n, steps = 4096, 200
    variants = [("flight_cap_0", {"QS_FLIGHT_CAP": 0}), ("flight_cap_1000", {"QS_FLIGHT_CAP": 1000})] + \
               [(f"slow_spread_{k}", {"QS_SLOW_SPREAD": k}) for k in (1, 2, 8, 32)] + \
               [("finish_pdl_0", {"QS_FINISH_PDL": 0}), ("graph_0", {"QS_GRAPH": 0})]
    ref = _make(qs, monkeypatch, num_envs=n, seed=41)
    ls = _Lockstep(ref)
    envs = [(name, _make(qs, monkeypatch, v, num_envs=n, seed=41)) for name, v in variants]
    o0 = ref.reset().clone()
    ls.ref_trace = ref.set_substep_trace(torch.arange(n))
    for name, e in envs:
        assert _same(o0, e.reset()), name
        ls.add(name, e, trace=e.set_substep_trace(torch.arange(n)))
    rng = np.random.default_rng(5)
    over = general = dones = general_steps = 0
    for _ in range(steps):
        airborne = int(((ref._views["contact"] & 15) == 0).sum())
        over += airborne > 1000
        _, _, d, _ = ls.step(_actions(rng, n, ref.action_dim))
        g = _counters(ref)[0]
        general += g
        general_steps += g > 0
        dones += int(d.sum())
    ls.finish()
    print(json.dumps(dict(test="dispatch_routes", envs=n, steps=steps, variants=[v for v, _ in variants],
                          steps_over_cap_1000=over, general=general, steps_with_general=general_steps, dones=dones)))
    assert over > steps // 2 and general > 0 and dones > 0


# ------------------------------------------------------------------ the benchmark's size
def test_benchmark_size_is_deterministic(qs, monkeypatch):
    """65536 envs, 150 steps, three runs side by side: the step's graph, the end-to-end host path (side buffer of
    4096 rows) and, until urgent settles have happened (at least 60 steps), a run whose settle slices are one tick
    long.  Each run overflows the flight list with its own set of envs: all three are bit-identical.

    Random actions alone never empty a ring of settled episodes at this size: the one-tick slices let the queue grow
    past the conveyor's window within about 70 steps, and a backlog is then settled whole.  So that episodes also
    start on the urgent path (k_settle_urgent, and the host path's second observation copy), 256 envs are cut off by
    the NaN guard on 20 consecutive steps, in every run alike: each of them ends more episodes than its ring holds."""
    n, steps, cap = N_FULL, 150, _flight_cap()
    ref = _make(qs, monkeypatch, num_envs=n, seed=43)
    host = _make(qs, monkeypatch, num_envs=n, seed=43)
    starved = _make(qs, monkeypatch, {"QS_SETTLE_SLICE_MIN": 1, "QS_SETTLE_SLICE_MAX": 1}, num_envs=n, seed=43)
    o0 = ref.reset().clone()
    assert np.array_equal(host.reset_host(), o0.cpu().numpy())
    assert _same(o0, starved.reset())
    urgent, starved_steps = [0], [0]

    def watch(e):
        urgent[0] += _counters(e)[1]
        starved_steps[0] += 1
        return urgent[0] > 0

    ls = _Lockstep(ref)
    ls.add("host_path", host, path="host")
    ls.add("settle_slice_1", starved, steps=60, watch=watch)
    rng = np.random.default_rng(7)
    cut = torch.arange(0, n, n // 256, device=ref.device)
    over = general = dones = urgent_ref = 0
    for t in range(steps):
        airborne = int(((ref._views["contact"] & 15) == 0).sum())
        over += airborne > cap
        _, _, d, _ = ls.step(_actions(rng, n, ref.action_dim))
        c = _counters(ref)
        general += c[0]
        urgent_ref += c[1]
        dones += int(d.sum())
        if 10 <= t < 30:   # a non-finite base height: the next step ends the episode (done, reward 0)
            for e in [ref] + [f["env"] for f in ls.followers if f["env"] is not None]:
                e._views["state"][2, cut] = float("nan")
    ls.finish()
    print(json.dumps(dict(test="benchmark_size_deterministic", envs=n, steps=steps, flight_cap=cap, steps_over_cap=over,
                          general=general, dones=dones, starved_steps=starved_steps[0], urgent=urgent[0],
                          urgent_default=urgent_ref)))
    assert over > steps // 2 and general > 0 and dones > 0 and urgent[0] > 0


def test_benchmark_size_matches_its_shards(qs, monkeypatch):
    """65536 envs against the same envs in 2 shards of 32768 (general solver at 32 envs per warp, no flight-list
    overflow) and in 8 shards of 8192 (one env per warp), bit for bit after every step, and the shards' rollout
    statistics add up to the full run's"""
    n, steps, cap = N_FULL, 150, _flight_cap()
    ref = _make(qs, monkeypatch, num_envs=n, seed=47)
    ls = _Lockstep(ref)
    shards = []
    for k in (2, 8):
        m = n // k
        for i in range(k):
            e = _make(qs, monkeypatch, num_envs=m, seed=47, env_id_offset=i * m)
            shards.append((k, e))
            ls.add(f"{k}x{m}[{i}]", e, sl=slice(i * m, (i + 1) * m))
    o0 = ref.reset().clone()
    for f in ls.followers:
        assert _same(o0[f["sl"]], f["env"].reset()), f["name"]
    rng = np.random.default_rng(11)
    over = general = general_half = dones = 0
    for _ in range(steps):
        airborne = int(((ref._views["contact"] & 15) == 0).sum())
        over += airborne > cap
        _, _, d, _ = ls.step(_actions(rng, n, ref.action_dim))
        general += _counters(ref)[0]
        general_half += _counters(shards[0][1])[0]
        dones += int(d.sum())
    ls.finish()
    full = ref.rollout_stats().double().cpu()
    for k in (2, 8):
        parts = torch.stack([e.rollout_stats() for kk, e in shards if kk == k]).double().cpu()
        tot = parts.sum(0)
        for r in (3, 6):   # the two maxima
            tot[r] = parts[:, r].max()
        for r in (0, 1, 3, 6):   # env count, finished episodes, maxima: exact
            assert float(tot[r]) == float(full[r]), (k, r, float(tot[r]), float(full[r]))
        # the sums: k_stats adds in atomic order
        np.testing.assert_allclose(tot.numpy(), full.numpy(), rtol=1e-5, atol=0)
    print(json.dumps(dict(test="benchmark_size_shards", envs=n, steps=steps, flight_cap=cap, steps_over_cap=over,
                          general=general, general_in_half_shard=general_half, dones=dones,
                          episodes=float(full[1]))))
    assert over > steps // 2 and general > 0 and general_half > 0 and dones > 0


# ------------------------------------------------------------------ against the oracle at size
class _OracleTicksGeneral(OracleTicks):
    """OracleTicks that also records, per tick, whether the oracle's solver had joint-limit rows (World.last_rows) or
    contacts of non-foot shapes: the ticks the library runs on the general solver"""

    def step(self, action):
        world, general = self.world, []

        class _Recording:
            def __getattr__(self, name):
                return getattr(world, name)

            def step(self, tau):
                world.step(tau)
                general.append(world.last_rows[0] > 0 or any(c[0] not in FOOT_LINKS for c in world.contacts()))

        self.world = _Recording()
        try:
            rows = super().step(action)
        finally:
            self.world = world
        self.general = general
        return rows


def test_benchmark_size_ticks_match_oracle(qs, monkeypatch):
    """65536 envs after 40 steps of random actions, restarted from their own state with a cold contact history (as the
    teacher-forced tests do): every env starts the step in the flight list, so about 27 k of them overflow into
    k_step_contact and every grounded env is handed over at tick 0.  One traced step, tick by tick against the oracle:
    envs the oracle needs the general solver for (up to 256), envs airborne for the whole step, envs that touch down
    in it and envs grounded at tick 0 (128 each)."""
    n, cap = N_FULL, _flight_cap()
    env = _make(qs, monkeypatch, num_envs=n, seed=53)
    env.reset()
    rng = np.random.default_rng(13)
    for _ in range(40):
        env.step(torch.from_numpy(_actions(rng, n, env.action_dim)).cuda())
    env.set_state(env.get_state())   # clears the contact bits and impulses: a cold contact history
    S = env.get_state().double().cpu().numpy()
    mu = env._views["mu"].double().cpu().numpy()
    assert int(((env._views["contact"] & 15) == 0).sum()) == n > cap
    tr = env.set_substep_trace(torch.arange(n))
    act = _actions(rng, n, env.action_dim)
    env.step(torch.from_numpy(act).cuda())
    general_gpu = _counters(env)[0]
    got = tr.cpu().numpy()                           # [10, 66, n]
    feet = got[:, 65].astype(np.int64) & 15          # [10, n]
    invalid = got[:, 65].astype(np.int64) >> 8
    q = np.concatenate([S[None, :, 13:25], got[:, 13:25].transpose(0, 2, 1)])   # [11, n, 12]
    near_limit = ((q <= URDF_LO + 0.02) | (q >= URDF_HI - 0.02)).any(axis=(0, 2))
    candidates = (invalid > 0).any(0) | near_limit
    pick = np.random.default_rng(17)
    ref = _OracleTicksGeneral(**CFG3)

    def oracle(i):
        ref.world.set_params(mu_ground=mu[i])
        ref.world.set_state(S[i])
        rows = ref.step(act[i].astype(np.float64))
        return rows, any(ref.general)

    strata = {"general": _TickCompare(), "airborne": _TickCompare(), "touchdown": _TickCompare(),
              "grounded": _TickCompare()}
    count = dict.fromkeys(strata, 0)

    def compare(i, stratum):
        rows, general = oracle(i)
        name = "general" if general else stratum
        if name == "general" and count["general"] >= 256:
            return
        strata[name].add(got[:, :, i].astype(np.float64), rows, general)
        count[name] += 1

    cand = np.flatnonzero(candidates)
    for i in pick.permutation(cand)[:1024]:
        rows, general = oracle(i)
        if general and count["general"] < 256:
            strata["general"].add(got[:, :, i].astype(np.float64), rows, True)
            count["general"] += 1
    pools = {"airborne": (feet == 0).all(0), "touchdown": (feet[0] == 0) & (feet != 0).any(0),
             "grounded": feet[0] != 0}
    for name, pool in pools.items():
        for i in pick.permutation(np.flatnonzero(pool & ~candidates))[:128]:
            compare(i, name)
    print(json.dumps(dict(test="benchmark_size_ticks_oracle", envs=n, flight_cap=cap, general_gpu=general_gpu,
                          candidates=int(candidates.sum()), compared=count,
                          pools={k: int(v.sum()) for k, v in pools.items()})))
    assert general_gpu > 0
    for name, cmp in strata.items():
        assert count[name] > 0, name
        cmp.check()


def test_conveyor_settled_starts_match_oracle(qs, monkeypatch):
    """65536 envs, at least 100 steps: 24 envs whose episode ended in the last step start the next one from a slot the
    settle conveyor filled (k_settle_slice); that start against the oracle's reset with the env's friction draw"""
    from oracle import oracle as O
    from test_gpu_parity import ATOL, RTOL
    n = N_FULL
    env = _make(qs, monkeypatch, num_envs=n, seed=59)
    env.reset()
    rng = np.random.default_rng(19)
    t = 0
    while True:
        _, _, d, _ = env.step(torch.from_numpy(_actions(rng, n, env.action_dim)).cuda())
        t += 1
        c = _counters(env)
        if t >= 100 and int(d.sum()) >= 24 and c[1] == 0:   # no urgent settle in this step: every start is a slot's
            break
        assert t < 200
    ended = np.flatnonzero(d.cpu().numpy())
    ids = np.random.default_rng(23).permutation(ended)[:24]
    assert (env._views["env_steps"][ids] == 0).all() and (env._views["sim_steps"][ids] == 0).all()
    S = env.get_state().cpu().numpy()
    obs = env.get_observation(with_noise=False).cpu().numpy()
    mu = env._views["mu"].cpu().numpy()
    last = env.get_last_action().cpu().numpy()
    g = load_golden("analytic.npz")
    init_action = g["s1_CARTESIAN_PD_SYMMETRIC_init_action"]
    o = O.Env(**CFG3)
    worst = 0.0
    for i in ids:
        ref_obs = o.reset(mu=float(mu[i]))
        np.testing.assert_allclose(S[i], o.world.get_state(), atol=1e-3)       # 2500 fp32 ticks vs fp64
        np.testing.assert_allclose(obs[i], ref_obs, atol=1e-3)
        np.testing.assert_allclose(last[i], init_action, rtol=RTOL, atol=ATOL)
        worst = max(worst, float(np.abs(S[i] - o.world.get_state()).max()))
    print(json.dumps(dict(test="conveyor_settled_starts", envs=n, steps=t, ended_in_last_step=len(ended),
                          compared=len(ids), worst_state_err=worst)))
