"""Per-substep trace (qs_set_substep_trace, BatchedQuadrupedGymEnv.set_substep_trace, SubstepRecorder) and the oracle's
per-tick record it is checked against.  The CPU tests pin that record and the recorder's views; the GPU tests
(-m gpu, on the B200) check that tracing changes no result, that the rows are complete and end on the step, and that
every tick matches the oracle's.  The oracle's Env records nothing between ticks; OracleTicks runs its tick loop from
here, on its World, and is pinned bit for bit to Env.step."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

from conftest import ROLLOUTS, load_golden

JIP = dict(enable_springs=True, task_env="JUMPING_IN_PLACE", observation_space_mode="ARS_BASIC")
CFG3 = dict(enable_springs=True, task_env="JUMPING_FORWARD", motor_control_mode="CARTESIAN_PD",
            action_space_mode="SYMMETRIC", observation_space_mode="ARS_BASIC")   # bench.py configuration 3


# ------------------------------------------------------------------ the oracle, tick by tick
CALF_LINKS, FOOT_LINKS = (4, 8, 12, 16), (5, 9, 13, 17)   # pybullet link ids (quadruped.py:236-241,545-596)


class OracleTicks:
    """The tick loop of the oracle's qso_env_step (ApplyAction + stepSimulation, quadruped_gym_env.py:207-219: action
    filter, action -> motor command, then per tick PD + spring torque and World.step), run here on the World of an
    oracle Env so that every tick can be recorded with what the substep trace holds: state 37, motor torque 12, spring
    torque 12, foot normal forces 4 (0 off contact), contact word mask | invalid << 8 (GetContactInfo,
    quadruped.py:224-258).  Only the oracle's public functions are used; test_oracle_ticks_are_the_env_step pins it
    bit for bit to Env.step."""

    def __init__(self, mu=1.0, enable_springs=True, motor_control_mode="PD", action_space_mode="SYMMETRIC",
                 task_env="NO_TASK", enable_action_filter=False, action_repeat=10, time_step=0.001, demo=None,
                 **env_kw):
        from oracle import oracle as O
        from quadruped_springs_b200.configs import go1_config
        self.O = O
        self.env = O.Env(enable_springs=enable_springs, motor_control_mode=motor_control_mode,
                         action_space_mode=action_space_mode, task_env=task_env, action_repeat=action_repeat,
                         enable_action_filter=enable_action_filter, time_step=time_step, **env_kw)
        if demo is not None:   # the *_DEMO tasks' demonstration (rows start with the action)
            self.env.set_demo(demo[:, :self.env.action_dim])
        self.env.reset(mu=mu)
        self.world = self.env.world
        c = go1_config(enable_springs)
        self.kp, self.kd = np.array(c.MOTOR_KP, float), np.array(c.MOTOR_KD, float)
        self.tau_max = np.array(c.TORQUE_LIMITS, float)
        self.springs = (np.array(c.SPRINGS_STIFFNESS, float), np.array(c.SPRINGS_DAMPING, float),
                        np.array(c.SPRINGS_REST_ANGLE, float)) if enable_springs else None
        self.map = dict(enable_springs=enable_springs, control=motor_control_mode, action_mode=action_space_mode,
                        task=task_env)
        self.repeat, self.adim = action_repeat, self.env.action_dim
        self.filt = None
        if enable_action_filter:   # action_filter.py:110-127: butter(2, 3 Hz) at the control rate, history = last action
            fs = 1.0 / (action_repeat * time_step)
            K = np.tan(np.pi * 3.0 / fs)
            nrm = 1.0 / (1 + np.sqrt(2.0) * K + K * K)
            b0 = K * K * nrm
            self.fb, self.fa = (b0, 2 * b0, b0), (1.0, 2 * (K * K - 1) * nrm, (1 - np.sqrt(2.0) * K + K * K) * nrm)
            a0 = self.env.last_action()
            self.filt = [a0.copy(), a0.copy(), a0.copy(), a0.copy()]   # x[t-1], x[t-2], y[t-1], y[t-2]

    def set_springs(self, k3, b3, rest3):
        self.springs = (np.asarray(k3, float), np.asarray(b3, float), np.asarray(rest3, float))

    def step(self, action):
        """one control step from the World's current state; returns the rows [action_repeat, 66]"""
        a = np.asarray(action, float)[:self.adim].copy()
        if self.filt is not None:
            x1, x2, y1, y2 = self.filt
            fb, fa = self.fb, self.fa
            y = a * fb[0] + x1 * fb[1] + x2 * fb[2] - (y1 * fa[1] + y2 * fa[2])
            self.filt = [a.copy(), x1, y, y1]
            a = y
        a12 = np.zeros(12)
        a12[:self.adim] = a
        cmd = self.O.action_to_command(a12, **self.map)
        rows = np.zeros((self.repeat, 66))
        for t in range(self.repeat):
            s = self.world.get_state()
            q, qd = s[13:25], s[25:37]
            tm = self.O.pd_torque(self.kp, self.kd, self.tau_max, cmd, q, qd)
            ts = self.O.spring_torque(*self.springs, q, qd) if self.springs else np.zeros(12)
            self.world.step(tm + ts)
            r = rows[t]
            r[:37] = self.world.get_state()
            r[37:49], r[49:61] = tm, ts
            mask, ninv = 0, 0
            for link, nf, dist, pos in self.world.contacts():
                if link in FOOT_LINKS:
                    k = FOOT_LINKS.index(link)
                    mask |= 1 << k
                    r[61 + k] += nf
                else:
                    ninv += 1
            ninv += sum(1 for la, lb, _ in self.world.self_contacts() if la in CALF_LINKS or lb in CALF_LINKS)
            r[65] = mask | ninv << 8
        return rows


ORACLE_CFGS = [
    dict(enable_springs=True, task_env="JUMPING_IN_PLACE"),
    dict(enable_springs=False, task_env="JUMPING_IN_PLACE", action_space_mode="DEFAULT"),
    dict(enable_springs=True, task_env="JUMPING_FORWARD", motor_control_mode="CARTESIAN_PD"),
    dict(enable_springs=True, task_env="JUMPING_IN_PLACE_PPO_HP", enable_action_filter=True),
    dict(enable_springs=True, task_env="BACKFLIP"),
]


@pytest.mark.parametrize("cfg", ORACLE_CFGS, ids=lambda c: "-".join(str(v) for v in c.values()))
def test_oracle_ticks_are_the_env_step(cfg):
    """the recorded tick loop is the oracle's Env.step bit for bit: from the same state (a cold contact history on both
    sides), its last row equals the Env's post-step state, torques and contact summary exactly, over a random rollout
    that flies, lands and crashes"""
    from oracle import oracle as O
    ticks = OracleTicks(mu=0.8, **cfg)
    env = O.Env(**{k: v for k, v in cfg.items()})
    env.reset(mu=0.8)
    rng = np.random.default_rng(0)
    flights = contacts = 0
    for _ in range(60):
        s0 = env.world.get_state()
        env.world.set_state(s0)
        ticks.world.set_state(s0)
        a = rng.uniform(-1, 1, env.action_dim)
        rec = ticks.step(a)
        o, r, d, t = env.step(a)
        tm, ts = env.torques()
        assert np.array_equal(rec[-1, :37], env.world.get_state())
        assert np.array_equal(rec[-1, 37:49], tm) and np.array_equal(rec[-1, 49:61], ts)
        mask, force, ninv = 0, np.zeros(4), 0
        for link, nf, dist, pos in env.world.contacts():
            if link in FOOT_LINKS:
                mask |= 1 << FOOT_LINKS.index(link)
                force[FOOT_LINKS.index(link)] += nf
            else:
                ninv += 1
        ninv += sum(1 for la, lb, _ in env.world.self_contacts() if la in CALF_LINKS or lb in CALF_LINKS)
        assert np.array_equal(rec[-1, 61:65], force) and rec[-1, 65] == mask | ninv << 8
        feet = rec[:, 65].astype(int) & 15
        flights += int((feet == 0).sum())
        contacts += int((feet != 0).sum())
        if d:
            break
    # (the 3 Hz action filter smooths random actions into a stand: no flight phase there)
    assert contacts > 10 and (flights > 10 or cfg.get("enable_action_filter"))


def test_oracle_tick_rows_are_world_steps():
    """row t = World.step applied to row t-1's world with row t's torques (to 1e-12)"""
    from oracle import oracle as O
    ticks = OracleTicks(mu=0.8, **ORACLE_CFGS[0])
    p = ticks.world.params()
    w = O.World(**{k: getattr(p, k) for k, _ in p._fields_})
    rng = np.random.default_rng(3)
    worst, n_contact_ticks = 0.0, 0
    for _ in range(60):
        s0 = ticks.world.get_state()
        ticks.world.set_state(s0)
        w.set_state(s0)
        rec = ticks.step(rng.uniform(-1, 1, 6))
        for k in range(10):
            w.step(rec[k, 37:49] + rec[k, 49:61])
            worst = max(worst, float(np.abs(w.get_state() - rec[k, :37]).max()))
            n_contact_ticks += int(rec[k, 65]) & 15 != 0
    assert worst < 1e-12 and n_contact_ticks > 20


# ------------------------------------------------------------------ CPU: the recorder's views
class _FakeEnv:
    """what SubstepRecorder uses of an env: set_substep_trace, step, the sim_steps view, sim_time_step"""

    def __init__(self, n_envs=5, repeat=3):
        self.sim_time_step = 0.001
        self._views = {"sim_steps": torch.arange(n_envs, dtype=torch.int32) * 100}
        self.repeat, self.calls = repeat, 0

    def set_substep_trace(self, env_ids):
        self.ids = list(env_ids)
        self.buf = torch.zeros(self.repeat, 66, len(self.ids))
        return self.buf

    def step(self, action):
        # hand-filled rows: value = 1000 * call + 100 * tick + row + column / 10; contact word: mask 5, 2 invalid
        c = self.calls
        t = torch.arange(self.repeat)[:, None, None]
        r = torch.arange(66)[None, :, None]
        j = torch.arange(len(self.ids))[None, None, :]
        self.buf.copy_((1000 * c + 100 * t + r + j / 10).float())
        self.buf[:, 65] = 5 | 2 << 8
        self._views["sim_steps"] += self.repeat
        self.calls += 1
        return action


def test_recorder_views_and_save(tmp_path):
    from quadruped_springs_b200.substep import SubstepRecorder
    env = _FakeEnv()
    rec = SubstepRecorder(env, [4, 1], steps=4)
    for i in range(3):
        assert rec.step(i) == i
    assert rec.count == 3 and rec.data.shape == (4, 3, 66, 2)
    expect = lambda first, k: torch.stack([torch.stack([torch.stack(
        [torch.tensor([1000 * s + 100 * t + first + q + j / 10 for q in range(k)]) for j in range(2)])
        for t in range(3)]) for s in range(3)]).float()
    for name, (first, k) in {"base_position": (0, 3), "base_orientation": (3, 4), "base_linear_velocity": (7, 3),
                             "base_angular_velocity": (10, 3), "motor_angles": (13, 12), "motor_velocities": (25, 12),
                             "motor_torques": (37, 12), "spring_torques": (49, 12), "feet_normal_forces": (61, 4)}.items():
        v = getattr(rec, name)
        assert v.shape == (3, 3, 2, k), name
        assert torch.equal(v, expect(first, k)), name
    assert torch.equal(rec.feet_in_contact, torch.tensor([True, False, True, False]).expand(3, 3, 2, 4))
    assert torch.equal(rec.invalid_contacts, torch.full((3, 3, 2), 2, dtype=torch.int32))
    # env 4 starts at tick 400, env 1 at tick 100; three ticks per step
    st = rec.sim_time
    assert st.dtype == torch.float64 and st.shape == (3, 3, 2)
    np.testing.assert_allclose(st[:, :, 0].numpy(), (400 + 3 * np.arange(3)[:, None] + np.arange(1, 4)[None]) * 1e-3)
    np.testing.assert_allclose(st[:, :, 1].numpy(), (100 + 3 * np.arange(3)[:, None] + np.arange(1, 4)[None]) * 1e-3)
    rec.save(tmp_path / "trace.npz")
    z = np.load(tmp_path / "trace.npz")
    for name in ("base_position", "motor_torques", "feet_in_contact", "invalid_contacts", "sim_time"):
        assert np.array_equal(z[name], getattr(rec, name).numpy()), name
    assert list(z["env_ids"]) == [4, 1]
    rec.step(3)
    with pytest.raises(RuntimeError):
        rec.step(4)


# ------------------------------------------------------------------ GPU
def cuda(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32, device="cuda")


@pytest.fixture(scope="module")
def qs():
    import quadruped_springs_b200 as m
    assert torch.cuda.is_available()
    return m


def _counters(env):
    out = (C.c_int32 * 4)()
    env._L.qs_debug_counters(env._h, out, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    return list(out)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["graph", "host"])
def test_trace_is_invisible_complete_and_ends_on_the_step(qs, path):
    """4096 envs of configuration 3 (noise, auto_reset) for 300 steps, one env tracing all envs and one tracing none:
    every result is bit-identical; every tick row of every traced env is written; the last row is the step"""
    n, steps = 4096, 300
    kw = dict(num_envs=n, seed=21, auto_reset=True, enable_noise=True, **CFG3)
    a, b = qs.BatchedQuadrupedGymEnv(**kw), qs.BatchedQuadrupedGymEnv(**kw)
    a.reset(), b.reset()
    tr = a.set_substep_trace(torch.arange(n))
    assert tr.shape == (10, 66, n) and tr.dtype == torch.float32
    rng = np.random.default_rng(2)
    dones = general = urgent = mid_contact = 0
    for step in range(steps):
        act = rng.uniform(-1, 1, (n, a.action_dim)).astype(np.float32)
        tr.fill_(float("nan"))
        contact0 = a._views["contact"].clone()
        if path == "graph":
            oa, ra, da, ia = a.step(cuda(act))
            ob, rb, db, ib = b.step(cuda(act))
            assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
            assert torch.equal(ia["TimeLimit.truncated"], ib["TimeLimit.truncated"])
            done = da
        else:
            oa, ra, da, ta = a.step_host(act)
            ob, rb, db, tb = b.step_host(act)
            assert np.array_equal(oa, ob) and np.array_equal(ra, rb) and np.array_equal(da, db) and np.array_equal(ta, tb)
            done = torch.as_tensor(da, device="cuda").bool()
        for key in ("state", "tau_motor", "tau_spring", "foot_force", "contact"):
            assert torch.equal(a._views[key], b._views[key]), (step, key)
        # complete: every tick row was written (the contact word of a written row is always finite), and every row of
        # an env that did not end its episode (a state that stops being finite ends it) is finite
        assert torch.isfinite(tr[:, 65]).all(), step
        assert torch.isfinite(tr[:, :, ~done]).all(), step
        # the last row is the step, for the envs that were not reset in it
        keep = ~done
        cnt, inv, forces, _ = a.robot.GetContactInfo()
        last = tr[-1][:, keep]
        assert torch.equal(last[0:37], a._views["state"][:, keep])
        assert torch.equal(last[37:49], a._views["tau_motor"][:, keep])
        assert torch.equal(last[49:61], a._views["tau_spring"][:, keep])
        assert torch.equal(last[61:65], forces.t()[:, keep].float())
        assert torch.equal(last[65], a._views["contact"][keep].float())
        # hard cases: flight -> contact inside the step, the general solver, episode ends, urgent settles
        bits = tr[:, 65].to(torch.int32) & 15
        first = torch.where((bits != 0).any(0), (bits != 0).int().argmax(0), torch.full_like(bits[0], -1))
        mid_contact += int((((contact0 & 15) == 0) & (first > 0)).sum())
        c = _counters(a)
        general += c[0]
        urgent += c[1]
        dones += int(done.sum())
    print(json.dumps(dict(path=path, dones=dones, general=general, urgent=urgent, mid_contact=mid_contact)))
    assert dones > 0 and general > 0 and mid_contact > 0


def _oracle_ticks_for(g, cfg):
    """OracleTicks with a rollout fixture's configuration and draws (friction, springs, masses)"""
    keys = ("enable_springs", "motor_control_mode", "action_space_mode", "task_env", "enable_action_filter")
    demo = np.asarray(g["demo"]) if "demo" in g.files else None
    ot = OracleTicks(mu=float(g["mu"]), demo=demo, **{k: v for k, v in cfg.items() if k in keys})
    if "springs" in g.files:
        s = np.asarray(g["springs"], dtype=np.float64)
        ot.set_springs(s[0:3], s[3:6], s[6:9])
    if "masses" in g.files:
        m = g["masses"]
        for leg in range(4):
            for j in range(3):
                ot.world.set_mass(2 + 4 * leg + j, m[j])
        ot.world.set_mass(0, m[3])
        ot.world.set_payload(m[4], m[5:8])
    return ot


class _TickCompare:
    """per-tick comparison of trace columns [10, 66] with oracle records [10, 66].  The fast solver is held to the
    single-tick fp32 tolerances (TOL_F32) widened linearly with the tick index to the 10-tick factor 3 of
    test_physics_tick_matches_oracle; ticks of a step that went through the general solver to the bounds of the
    teacher-forced replay's crash steps.  A tick is compared while the foot-contact bits agree up to it."""

    def __init__(self):
        from test_gpu_parity import TOL_F32
        self.tol = TOL_F32
        self.ticks = self.same = self.compared = 0
        self.worst = {}

    def add(self, got, ref, general):
        sl = (slice(0, 3), slice(3, 7), slice(7, 10), slice(10, 13), slice(13, 25), slice(25, 37))
        gb, rb = got[:, 65].astype(int) & 15, ref[:, 65].astype(int) & 15
        agree = np.cumprod(gb == rb).astype(bool)
        self.ticks += len(gb)
        self.same += int((gb == rb).sum())
        for t in np.nonzero(agree)[0]:
            self.compared += 1
            scale = 1.0 + 2.0 * t / 9.0
            if general:
                bounds = (2e-3, 2e-3, 5e-2, 5e-2, 2e-3, 1.0)
            else:
                bounds = tuple(x * scale for x in self.tol)
            for q, (s, tol) in enumerate(zip(sl, bounds)):
                err = float(np.abs(got[t, s] - ref[t, s]).max())
                self.worst[(general, q)] = max(self.worst.get((general, q), 0.0), err / tol)
                assert err < tol, (general, t, s, err, tol)
            np.testing.assert_allclose(got[t, 37:61], ref[t, 37:61], rtol=1e-3, atol=5e-2 if not general else 2.0)
            if not general:
                np.testing.assert_allclose(got[t, 61:65], ref[t, 61:65], rtol=2e-3, atol=0.2)

    def check(self):
        print(json.dumps(dict(ticks=self.ticks, same_bits=self.same / self.ticks, compared=self.compared,
                              worst_over_tol={f"{'general' if k[0] else 'fast'}_{k[1]}": v for k, v in self.worst.items()})))
        assert self.same / self.ticks > 0.98


@pytest.mark.gpu
def test_tick_rows_match_oracle_teacher_forced(qs):
    """every control step of every reference rollout (ROLLOUTS), from the reference's pre-step state with a cold contact
    history on both sides: each of the ten tick rows against the oracle's per-tick record"""
    cmp = _TickCompare()
    from test_gpu_parity import _make_env_for
    for name in ROLLOUTS:
        g = load_golden(f"rollout_{name}.npz")
        env, cfg = _make_env_for(qs, g)
        env.reset()
        ref = _oracle_ticks_for(g, cfg)
        if "rsi" in name:
            env.reset_to_state(cuda(np.stack([g["init_state"]] * 2)))
        if "springs" in g.files:
            env._views["spring"][:] = cuda(g["springs"])[:, None]
        if "masses" in g.files:
            m = g["masses"]
            env.robot.set_masses(leg_masses=m[:3], base_mass=m[3], offset_mass=m[4], offset_position=m[5:8])
            env._views["mu"][:] = float(g["mu"])
        tr = env.set_substep_trace([0, 1])
        for t in range(len(g["reward"])):
            env.set_state(cuda(np.stack([g["pre_state"][t]] * 2)))   # also clears contact bits and impulses
            env.step(cuda(g["actions"][t]).expand(2, -1))
            got = tr[:, :, 0].double().cpu().numpy()
            general = _counters(env)[0] > 0
            assert torch.equal(tr[:, :, 0], tr[:, :, 1])
            ref.world.set_state(g["pre_state"][t])
            rec = ref.step(g["actions"][t])
            cmp.add(got, rec, general)
    cmp.check()


@pytest.mark.gpu
def test_tick_rows_match_oracle_on_general_solver_states(qs):
    """joints at their limits and robots lying on the ground: steps run by k_step_slow, tick by tick against the oracle"""
    from test_gpu_parity import _general_states
    n = 128
    rng = np.random.default_rng(17)
    S = _general_states(n, rng)
    mu = rng.uniform(0.5, 1.0, size=n).astype(np.float32).astype(np.float64)
    act = rng.uniform(-1, 1, size=(n, 6)).astype(np.float32).astype(np.float64)
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, enable_noise=False, auto_reset=False, **JIP)
    env.reset()
    env.set_state(cuda(S))
    env._views["mu"][:] = cuda(mu)
    tr = env.set_substep_trace(torch.arange(n))
    env.step(cuda(act))
    assert _counters(env)[0] > n // 4
    got = tr.double().cpu().numpy()
    ref = OracleTicks(**JIP)
    cmp = _TickCompare()
    for i in range(n):
        ref.world.set_params(mu_ground=mu[i])
        ref.world.set_state(S[i])
        rec = ref.step(act[i])
        cmp.add(got[:, :, i], rec, True)
    cmp.check()


@pytest.mark.gpu
def test_trace_subset_clear_and_set_after_capture(qs):
    n = 64
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, auto_reset=False, enable_noise=False, seed=3, **CFG3)
    env.reset()
    rng = np.random.default_rng(0)
    act = lambda: cuda(rng.uniform(-1, 1, (n, env.action_dim)))
    for _ in range(3):                 # the step's graph is captured without a trace
        env.step(act())
    tr = env.set_substep_trace([7, 3, n - 1])
    assert tr.shape == (10, 66, 3)
    env.step(act())
    assert torch.equal(tr[-1, :37], env._views["state"][:, [7, 3, n - 1]])
    assert torch.equal(tr[-1, 37:49], env._views["tau_motor"][:, [7, 3, n - 1]])
    assert torch.isfinite(tr).all()
    env.set_substep_trace(None)
    old = tr.clone()
    for _ in range(3):
        env.step(act())
    torch.cuda.synchronize()
    assert torch.equal(tr, old)        # nothing writes the cleared buffer
    tr2 = env.set_substep_trace(np.array([n - 1]))
    env.step(act())
    assert torch.equal(tr2[-1, :37, 0], env._views["state"][:, n - 1])
    assert torch.equal(tr, old)


@pytest.mark.gpu
def test_trace_rejects_bad_ids(qs):
    env = qs.BatchedQuadrupedGymEnv(num_envs=16, auto_reset=False, **JIP)
    for bad in ([1, 2, 1], [0, 16], [-1], [], [0.0, 1.0], torch.tensor([[0, 1]])):
        with pytest.raises(ValueError):
            env.set_substep_trace(bad)
    assert env._trace is None


@pytest.mark.gpu
def test_trace_of_cpg_steps(qs):
    """qs_cpg_steps (action_repeat = 1): one tick row per step, equal to the state after the step"""
    n = 256
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, isRLGymInterface=False, action_repeat=1, motor_control_mode="TORQUE",
                                    enable_springs=True, auto_reset=False, seed=4)
    env.reset()
    cpg = qs.HopfNetwork(num_envs=n, gait="TROT", omega_swing=16 * np.pi, omega_stance=4 * np.pi, time_step=0.001, seed=1)
    tr = env.set_substep_trace(torch.arange(n))
    assert tr.shape == (1, 66, n)
    for _ in range(20):
        tr.fill_(float("nan"))
        cpg.drive(env, 1)
        assert torch.equal(tr[0, :37], env._views["state"])
        assert torch.equal(tr[0, 37:49], env._views["tau_motor"])
        # (the epilogue adds the step's self contacts to the env's invalid count: the foot bits are the tick's)
        assert torch.equal(tr[0, 65].int() & 15, env._views["contact"] & 15)
