"""External push on the trunk (Quadruped.apply_external_force, quadruped.py:338-343): the oracle-side push
(tools/oracle_push.c) against the laws of momentum, the pushed tick templates on the host against the oracle, and on the
GPU the step kernels' push
(qs_set_external_force / env.robot.apply_external_force) against the oracle tick by tick, its countdown, its clearing
on resets and episode ends, and its invisibility to every env it does not push."""
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
JIP = dict(enable_springs=True, task_env="JUMPING_IN_PLACE", observation_space_mode="ARS_BASIC")
CFG3 = dict(enable_springs=True, task_env="JUMPING_FORWARD", motor_control_mode="CARTESIAN_PD",
            action_space_mode="SYMMETRIC", observation_space_mode="ARS_BASIC")   # bench.py configuration 3
SL = (slice(0, 3), slice(3, 7), slice(7, 10), slice(10, 13), slice(13, 25), slice(25, 37))
TRUNK_HALF = np.array([0.1881, 0.04675, 0.057])   # half extents of the trunk box: points inside it


def _R(quat):
    x, y, z, w = np.asarray(quat, float) / np.linalg.norm(quat)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


_PUSH_LIB = None


def _oracle_push():
    """tools/oracle_push.c (Bullet's applyExternalForce on the base for the oracle's World), built once into a
    temporary directory"""
    global _PUSH_LIB
    if _PUSH_LIB is None:
        import ctypes as C
        import tempfile
        so = os.path.join(tempfile.mkdtemp(prefix="oracle_push_"), "liboracle_push.so")
        cc = shutil.which("gcc") or shutil.which("cc") or "gcc"
        res = subprocess.run([cc, "-O2", "-fPIC", "-std=c11", "-D_GNU_SOURCE", "-shared", "-o", so,
                              os.path.join(ROOT, "tools", "oracle_push.c"), "-lm"], capture_output=True, text=True)
        assert res.returncode == 0, res.stderr[-2000:]
        L = C.CDLL(so)
        dp = C.POINTER(C.c_double)
        L.qsp_push_before_step.restype = None
        L.qsp_push_before_step.argtypes = [C.c_void_p, dp, dp]
        _PUSH_LIB = (L, dp)
    return _PUSH_LIB


def _push_at(w, force, x):
    """push the base of the oracle World `w` in its next step with `force` at the world point `x`; the step's joint
    torques must already be added (World.add_torque)"""
    L, dp = _oracle_push()
    f = np.ascontiguousarray(force, dtype=np.float64)
    p = np.ascontiguousarray(x, dtype=np.float64)
    assert f.shape == (3,) and p.shape == (3,)
    L.qsp_push_before_step(w.h, f.ctypes.data_as(dp), p.ctypes.data_as(dp))


def _pushed_step(w, tau, force, point):
    """one oracle World tick with joint torques `tau`, pushed with `force` at the point `point` of the base frame (from
    the base position), placed with the tick's own pose"""
    s = w.get_state()
    w.add_torque(np.asarray(tau, float))
    _push_at(w, force, s[0:3] + _R(s[3:7]) @ np.asarray(point, float))
    w.step()


def _flight_state(rng):
    s = np.zeros(37)
    q = rng.normal(size=4)
    s[3:7] = q / np.linalg.norm(q)
    s[2] = 5.0
    s[7:13] = rng.normal(size=6)
    s[13:25] = np.array([0, np.pi / 4, -np.pi / 2] * 4) + rng.normal(size=12) * 0.2
    s[25:37] = rng.normal(size=12) * 2
    return s


# ------------------------------------------------------------------ CPU: the oracle
def test_oracle_push_changes_momentum_by_the_impulse():
    """free flight, zero joint torque, one tick from the same state with and without a force F at the world point x.
    Read in the configuration the tick's velocities were solved in (its starting pose, with the new velocities), the
    linear momentum differs by F dt and the angular momentum about the world origin by x x F dt, to fp64 rounding; in
    the new pose, to O(dt^2).  Pins the sign and the frame of the push."""
    from oracle import oracle as O
    rng = np.random.default_rng(0)
    w = O.World()
    dt = w.params().dt
    vel = np.r_[7:13, 25:37]

    def momenta(s0, s1, F=None, x=None):
        w.set_state(s0)
        w.add_torque(np.zeros(12))
        if F is not None:
            _push_at(w, F, x)
        w.step()
        after = w.get_state()
        mixed = s0.copy()
        mixed[vel] = after[vel]
        w.set_state(mixed)
        _, P, L = w.energy()
        w.set_state(after)
        _, P1, L1 = w.energy()
        return P, L, P1, L1

    for _ in range(12):
        s = _flight_state(rng)
        F = rng.normal(size=3) * 200.0
        x = s[0:3] + _R(s[3:7]) @ (rng.uniform(-1, 1, 3) * TRUNK_HALF)
        P0, L0, P0n, L0n = momenta(s, s)
        P1, L1, P1n, L1n = momenta(s, s, F, x)
        np.testing.assert_allclose(P1 - P0, F * dt, rtol=0, atol=1e-11 * (1 + np.abs(F).max()))
        np.testing.assert_allclose(L1 - L0, np.cross(x, F) * dt, rtol=0, atol=1e-11 * (1 + np.abs(F).max()))
        scale = np.abs(F).max() * dt
        np.testing.assert_allclose(P1n - P0n, F * dt, rtol=0, atol=scale * 3e-2)   # O(dt^2): |F| dt^2 x 30 /s
        np.testing.assert_allclose(L1n - L0n, np.cross(x, F) * dt, rtol=0, atol=scale * 3e-2)   # O(dt^2): |F| dt^2 x 30 /s


def test_oracle_push_zero_is_no_push_and_calls_add_up():
    from oracle import oracle as O
    rng = np.random.default_rng(1)
    s = _random_contact_state(rng)
    tau = rng.normal(size=12) * 5
    F, x = np.array([30.0, -10.0, 5.0]), s[0:3] + np.array([0.05, 0.02, 0.0])
    ref, a = O.World(), O.World()
    for w in (ref, a):
        w.set_state(s)
    # a zero force is no push at all, bit for bit, contacts and warm start included
    for _ in range(3):
        ref.step(tau)
        a.add_torque(tau)
        _push_at(a, np.zeros(3), x)
        a.step()
    assert np.array_equal(ref.get_state(), a.get_state())
    # two pushes before one step act as one push with the summed force
    b, c = O.World(), O.World()
    b.set_state(s), c.set_state(s)
    b.add_torque(tau), c.add_torque(tau)
    _push_at(b, F, x)
    _push_at(b, F, x)
    _push_at(c, 2 * F, x)
    b.step(), c.step()
    np.testing.assert_allclose(b.get_state(), c.get_state(), rtol=0, atol=1e-12)
    assert not np.allclose(b.get_state(), ref.get_state())


def _random_contact_state(rng):
    from test_gpu_parity import _random_states
    return _random_states(1, rng, True)[0]


# ------------------------------------------------------------------ CPU: the kernel templates on the host
def _host_cases(rng):
    """(n_ticks, mu, state, tau, force, point): airborne, feet touching and general-solver states"""
    from test_gpu_parity import _general_states, _random_states
    out = []
    for kind, S in (("air", _random_states(16, rng, False)), ("touch", _random_states(24, rng, True)),
                    ("general", _general_states(16, rng))):
        for s in S:
            n_ticks = 1 if kind == "general" else 5
            out.append((kind, n_ticks, float(rng.uniform(0.5, 1.0)), s, rng.normal(size=12) * 5,
                        rng.normal(size=3) * 150.0, rng.uniform(-1, 1, 3) * TRUNK_HALF))
    return out


def _host_run(tmp, tag, flags, cases):
    exe = os.path.join(tmp, f"push_host_check_{tag}")
    res = subprocess.run([NVCC, "-std=c++17", "-w", *flags, "-o", exe, os.path.join(ROOT, "tools", "push_host_check.cu")],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    inp, out = os.path.join(tmp, f"{tag}_in.txt"), os.path.join(tmp, f"{tag}_out.txt")
    with open(inp, "w") as f:
        for _, n_ticks, mu, s, tau, F, p in cases:
            f.write(" ".join([str(n_ticks), repr(mu)] + [repr(float(v)) for v in (*s, *tau, *F, *p)]) + "\n")
    res = subprocess.run([exe, inp, out], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    rows = {}
    for line in open(out):
        t = line.split()
        rows.setdefault(t[0], {}).setdefault(int(t[1]), []).append(t[4:])
    return rows


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not found")
@pytest.mark.parametrize("pack", [1, 0])
def test_pushed_tick_templates_match_oracle_on_host(tmp_path, pack):
    """physics_tick / physics_tick_general<double> with kExt (pairs of legs, and one leg at a time) on airborne, touching
    and general-solver states, pushed on every tick: each tick against the oracle World given the same force, at the
    fp64 GPU tolerances; and the kExt instantiation with no push is the default one bit for bit"""
    from oracle import oracle as O
    from test_gpu_parity import TOL_F64
    rng = np.random.default_rng(40)
    cases = _host_cases(rng)
    rows = _host_run(str(tmp_path), f"p{pack}", [] if pack else ["-DQS_PACK_LEGS=0"], cases)
    w = O.World()
    worst = {"P": 0.0, "D": 0.0}
    for c, (kind, n_ticks, mu, s, tau, F, p) in enumerate(cases):
        assert rows["Z"][c] == rows["D"][c], (kind, c)                 # no push: the default arithmetic, bit for bit
        for run in ("P", "D"):
            w.set_params(mu_ground=mu)
            w.set_state(s)
            got = np.array(rows[run][c], float)
            for t in range(n_ticks):
                if run == "P":
                    _pushed_step(w, tau, F, p)
                else:
                    w.step(tau)
                ref = w.get_state()
                for sl, tol in zip(SL, TOL_F64):
                    err = float(np.abs(got[t][sl] - ref[sl]).max())
                    worst[run] = max(worst[run], err / tol)
                    assert err < tol, (kind, c, run, t, sl, err)
        assert not np.array_equal(rows["P"][c], rows["D"][c])
    print(f"worst error / TOL_F64: pushed {worst['P']:.3g}, unpushed {worst['D']:.3g}")


# ------------------------------------------------------------------ GPU
def cuda(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32, device="cuda")


@pytest.fixture(scope="module")
def qs():
    import quadruped_springs_b200 as m
    assert torch.cuda.is_available()
    return m


def _outputs_equal(a, b):
    for key in ("state", "tau_motor", "tau_spring", "foot_force", "contact"):
        assert torch.equal(a._views[key], b._views[key]), key


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["graph", "host"])
def test_idle_push_buffer_is_invisible(qs, path):
    """4096 envs of configuration 3 (noise, auto_reset) for 300 steps: with the push buffers attached and every count 0,
    every output is bit-identical to a twin without buffers (obs, reward, done, truncated, terminal obs, state)"""
    n, steps = 4096, 300
    kw = dict(num_envs=n, seed=21, auto_reset=True, enable_noise=True, **CFG3)
    a, b = qs.BatchedQuadrupedGymEnv(**kw), qs.BatchedQuadrupedGymEnv(**kw)
    a.reset(), b.reset()
    term_a, term_b = (torch.zeros(n, a.obs_dim, device="cuda") for _ in range(2))
    a.set_terminal_obs_buffer(term_a), b.set_terminal_obs_buffer(term_b)
    a.robot.apply_external_force([100.0, 0, 0], n_ticks=0)      # attaches the buffers, pushes nobody
    assert a.robot.get_external_force() is not None and b.robot.get_external_force() is None
    rng = np.random.default_rng(2)
    dones = 0
    for step in range(steps):
        act = rng.uniform(-1, 1, (n, a.action_dim)).astype(np.float32)
        if path == "graph":
            oa, ra, da, ia = a.step(cuda(act))
            ob, rb, db, ib = b.step(cuda(act))
            assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
            assert torch.equal(ia["TimeLimit.truncated"], ib["TimeLimit.truncated"])
            dones += int(da.sum())
        else:
            oa, ra, da, ta = a.step_host(act)
            ob, rb, db, tb = b.step_host(act)
            assert np.array_equal(oa, ob) and np.array_equal(ra, rb) and np.array_equal(da, db) and np.array_equal(ta, tb)
            dones += int(da.sum())
        _outputs_equal(a, b)
        assert torch.equal(term_a, term_b)
    assert int(a.robot.get_external_force()[2].abs().sum()) == 0
    assert dones > 0


def _debug_vs_oracle(qs, S, use_f64, n_ticks, rng, masses=None):
    """debug_ticks with random pushes on every tick vs the oracle World; returns (got, ref) states"""
    from oracle import oracle as O
    n = len(S)
    tau = (rng.normal(size=(n, 12)) * 5).astype(np.float32).astype(np.float64)
    mu = rng.uniform(0.5, 1.0, size=n).astype(np.float32).astype(np.float64)
    F = (rng.normal(size=(n, 3)) * 150.0).astype(np.float32).astype(np.float64)
    p = (rng.uniform(-1, 1, (n, 3)) * TRUNK_HALF).astype(np.float32).astype(np.float64)
    kw = dict(env_randomizer_mode="MASS_RANDOMIZER", seed=3) if masses is not None else {}
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, enable_noise=False, auto_reset=False, **JIP, **kw)
    if masses is not None:
        env.reset()
        env.robot.set_masses(**masses)
    env.set_state(cuda(S))
    env._views["mu"][:] = cuda(mu)
    env.robot.apply_external_force(F, p, n_ticks=n_ticks + 3)
    env.debug_ticks(cuda(tau), n_ticks, use_f64)
    got = env.get_state().cpu().numpy().astype(np.float64)
    assert torch.equal(env.robot.get_external_force()[2].cpu(), torch.full((n,), 3, dtype=torch.int32))
    md = env._views["mass_draw"].cpu().numpy().astype(np.float64) if masses is not None else None
    w = O.World()
    ref = np.zeros_like(S)
    for i in range(n):
        if md is not None:
            w = O.World()
            for leg in range(4):
                for j in range(3):
                    w.set_mass(2 + 4 * leg + j, md[j, i])
            w.set_mass(0, md[3, i])
            w.set_payload(md[4, i], md[5:8, i])
        w.set_params(mu_ground=mu[i])
        w.set_state(S[i])
        for _ in range(n_ticks):
            _pushed_step(w, tau[i], F[i], p[i])
        ref[i] = w.get_state()
    return got, ref


@pytest.mark.gpu
@pytest.mark.parametrize("use_f64", [1, 0])
@pytest.mark.parametrize("contact", [False, True])
def test_pushed_tick_matches_oracle(qs, use_f64, contact):
    from test_gpu_parity import TOL_F32, TOL_F64, _random_states
    rng = np.random.default_rng(31 + contact)
    S = _random_states(192, rng, contact)
    got, ref = _debug_vs_oracle(qs, S, use_f64, 1, rng)
    tol = TOL_F64 if use_f64 else TOL_F32
    # (a foot exactly at the contact threshold may flip in fp32: compare the rows whose result is close in position)
    ok = np.abs(got[:, 13:25] - ref[:, 13:25]).max(1) < 10 * tol[4]
    assert ok.mean() > 0.98
    for s, t in zip(SL, tol):
        err = np.abs(got[ok][:, s] - ref[ok][:, s]).max()
        assert err < t, (s, err)


@pytest.mark.gpu
@pytest.mark.parametrize("use_f64", [1, 0])
def test_pushed_general_solver_matches_oracle(qs, use_f64):
    from test_gpu_parity import _general_states
    rng = np.random.default_rng(78)
    S = _general_states(128, rng)
    got, ref = _debug_vs_oracle(qs, S, use_f64, 1, rng)
    err = np.abs(got - ref)
    ok = err[:, :7].max(1) < 1e-2        # (an invalid-contact flag may flip: test_general_solver_matches_oracle)
    assert ok.mean() > 0.97
    err = err[ok]
    if use_f64:
        assert err[:, :7].max() < 2e-6 and err[:, 13:25].max() < 5e-6 and err[:, 7:13].max() < 2e-4 and err[:, 25:].max() < 2e-3
    else:
        assert err[:, :7].max() < 2e-4 and err[:, 13:25].max() < 1e-3
        assert np.quantile(err[:, 25:], 0.99) < 5e-2 and np.quantile(err[:, 7:13], 0.99) < 5e-3


@pytest.mark.gpu
def test_pushed_tick_with_mass_randomizer_matches_oracle(qs):
    from test_gpu_parity import TOL_F64
    rng = np.random.default_rng(9)
    S = np.stack([_flight_state(rng) for _ in range(32)]).astype(np.float32).astype(np.float64)
    masses = dict(leg_masses=[0.75, 1.3, 0.2], base_mass=6.5, offset_mass=1.5, offset_position=[0.05, -0.02, 0.01])
    got, ref = _debug_vs_oracle(qs, S, 1, 1, rng, masses=masses)
    for s, t in zip(SL, TOL_F64):       # 3x: the mass properties are stored in fp32
        assert np.abs(got[:, s] - ref[:, s]).max() < 3 * t, s


class _PushedWorld:
    """an oracle World that pushes its base before each of its first `n` steps"""

    def __init__(self, world, force, point, n):
        self.w, self.F, self.p, self.n, self.k = world, force, point, n, 0

    def step(self, tau):
        if self.k < self.n:
            _pushed_step(self.w, tau, self.F, self.p)
        else:
            self.w.step(tau)
        self.k += 1

    def __getattr__(self, name):
        return getattr(self.w, name)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_push_countdown_tick_by_tick(qs, graph, monkeypatch):
    """a count of 25 at action_repeat 10: ticks 0-24 pushed, every tick row of the substep trace against the oracle's;
    ticks_left reads 15, 5, 0, 0 after the steps"""
    from test_substep_trace import OracleTicks, _TickCompare
    if not graph:
        monkeypatch.setenv("QS_GRAPH", "0")
    n = 64
    rng = np.random.default_rng(12)
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, enable_noise=False, auto_reset=False, seed=5, **JIP)
    env.reset()
    env.set_state(env.get_state())      # a cold contact history, as the oracle's set_state leaves it
    S0 = env.get_state().cpu().numpy().astype(np.float64)
    mu = env._views["mu"].cpu().numpy().astype(np.float64)
    F = np.array([[60.0, -40.0, 20.0]] * n) * rng.uniform(0.5, 1.5, (n, 1))
    p = rng.uniform(-1, 1, (n, 3)) * TRUNK_HALF
    F, p = F.astype(np.float32).astype(np.float64), p.astype(np.float32).astype(np.float64)
    ids = [0, 5, 17, 63]
    env.robot.apply_external_force(F[ids], p[ids], n_ticks=25, env_ids=ids)
    tr = env.set_substep_trace(ids)
    acts = rng.uniform(-1, 1, (4, n, env.action_dim)).astype(np.float32).astype(np.float64)
    oracles = []
    for i in ids:
        ot = OracleTicks(mu=float(mu[i]), **JIP)
        ot.world.set_state(S0[i])
        ot.world = _PushedWorld(ot.world, F[i], p[i], 25)
        oracles.append(ot)
    cmp = _TickCompare()
    left = []
    for step in range(4):
        env.step(cuda(acts[step]))
        left.append(env.robot.get_external_force()[2].cpu().numpy().copy())
        got = tr.double().cpu().numpy()
        for j, i in enumerate(ids):
            cmp.add(got[:, :, j], oracles[j].step(acts[step, i]), False)
    cmp.check()
    assert [int(x[ids[0]]) for x in left] == [15, 5, 0, 0]
    for x in left:
        assert np.array_equal(x[ids], np.full(len(ids), x[ids[0]])) and int(np.delete(x, ids).sum()) == 0


@pytest.mark.gpu
def test_resets_clear_the_push(qs):
    """a masked reset, reset_to_state and an episode end (auto_reset) leave n = 0, and the next episode is bit-identical
    to a never-pushed twin"""
    n = 32
    kw = dict(num_envs=n, seed=8, auto_reset=True, enable_noise=False, **JIP)
    a, b = qs.BatchedQuadrupedGymEnv(**kw), qs.BatchedQuadrupedGymEnv(**kw)
    a.reset(), b.reset()
    zero = lambda e: cuda(np.zeros((n, e.action_dim)))
    left = lambda: a.robot.get_external_force()[2].cpu().numpy()
    # masked reset: envs 0-7 pushed for a long time, then reset with a mask covering 0-3
    a.robot.apply_external_force([0.0, 0.0, 30.0], n_ticks=10**6, env_ids=list(range(8)))
    mask = torch.zeros(n, dtype=torch.bool, device="cuda")
    mask[:4] = True
    a.reset(mask=mask)
    b.reset(mask=mask)
    assert (left()[:4] == 0).all() and (left()[4:8] == 10**6).all()
    # reset_to_state of 4-7 from the twin's state
    st = b.get_state()
    mask2 = torch.zeros(n, dtype=torch.bool, device="cuda")
    mask2[4:8] = True
    a.reset_to_state(st, mask=mask2)
    b.reset_to_state(st, mask=mask2)
    assert (left() == 0).all()
    # envs 0-7 were reset identically in both: from here they match bit for bit
    for _ in range(5):
        a.step(zero(a)), b.step(zero(b))
    assert torch.equal(a._views["state"][:, :8], b._views["state"][:, :8])
    # an episode end: a huge push that spins env 9 off the ground ends its episode, and clears the count.  The twin
    # ends env 9's episode in the same step through the NaN / Inf guard; both then start the same next episode.
    a.robot.apply_external_force([0.0, 0.0, 3000.0], [0.0, 0.04, 0.0], n_ticks=10**6, env_ids=[9])
    ended = False
    for _ in range(300):
        _, _, d, _ = a.step(zero(a))
        if bool(d[9]):
            sb = b.get_state()
            sb[9] = float("nan")
            b.set_state(sb)
            _, _, db, _ = b.step(zero(b))
            assert bool(db[9])
            ended = True
            break
        b.step(zero(b))
    assert ended
    assert left()[9] == 0
    for _ in range(20):
        oa, _, _, _ = a.step(zero(a))
        ob, _, _, _ = b.step(zero(b))
        assert torch.equal(a._views["state"][:, 9], b._views["state"][:, 9]) and torch.equal(oa[9], ob[9])
    assert left()[9] == 0


@pytest.mark.gpu
def test_pushing_a_subset_leaves_the_others_alone(qs):
    n = 2048
    kw = dict(num_envs=n, seed=13, auto_reset=True, enable_noise=True, **CFG3)
    a, b = qs.BatchedQuadrupedGymEnv(**kw), qs.BatchedQuadrupedGymEnv(**kw)
    a.reset(), b.reset()
    rng = np.random.default_rng(3)
    mask = rng.random(n) < 0.25
    for step in range(40):
        if step % 7 == 0:
            k = int(mask.sum())
            a.robot.apply_external_force(rng.normal(size=(k, 3)) * 80, rng.uniform(-1, 1, (k, 3)) * TRUNK_HALF,
                                         n_ticks=rng.integers(0, 30, k), env_ids=torch.as_tensor(mask))
        act = cuda(rng.uniform(-1, 1, (n, a.action_dim)))
        oa, ra, da, _ = a.step(act)
        ob, rb, db, _ = b.step(act)
        keep = torch.as_tensor(~mask, device="cuda")
        assert torch.equal(oa[keep], ob[keep]) and torch.equal(ra[keep], rb[keep]) and torch.equal(da[keep], db[keep])
        assert torch.equal(a._views["state"][:, keep], b._views["state"][:, keep])
    assert not torch.equal(a._views["state"], b._views["state"])


@pytest.mark.gpu
def test_push_momentum_at_full_size(qs):
    """65536 airborne robots, zero torque, a horizontal push at the base origin for 20 ticks: the whole robot's momentum
    changes by the impulse plus gravity's"""
    from oracle import oracle as O
    n, ticks = 65536, 20
    rng = np.random.default_rng(5)
    S = np.zeros((n, 37), dtype=np.float32)
    quat = rng.normal(size=(n, 4)); S[:, 3:7] = quat / np.linalg.norm(quat, axis=1, keepdims=True)
    S[:, 2] = 50.0
    S[:, 7:13] = rng.normal(size=(n, 6))
    S[:, 13:25] = np.array([0, np.pi / 4, -np.pi / 2] * 4) + rng.normal(size=(n, 12)) * 0.2
    S[:, 25:37] = rng.normal(size=(n, 12)) * 2
    F = np.zeros((n, 3), dtype=np.float32)
    F[:, :2] = rng.normal(size=(n, 2)) * 100
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, enable_noise=False, auto_reset=False)
    env.set_state(cuda(S))
    env.robot.apply_external_force(F, n_ticks=ticks)
    env.debug_ticks(torch.zeros(n, 12, device="cuda"), ticks, 0)
    S1 = env.get_state().cpu().numpy()
    assert np.isfinite(S1).all() and int(env.robot.get_external_force()[2].abs().sum()) == 0
    w = O.World()
    m = 12.01301
    dt = ticks * 1e-3
    for i in rng.choice(n, 48, replace=False):
        w.set_state(S[i].astype(np.float64)); _, P0, _ = w.energy()
        w.set_state(S1[i].astype(np.float64)); _, P1, _ = w.energy()
        expect = F[i].astype(np.float64) * dt + np.array([0, 0, -9.8 * m * dt])
        np.testing.assert_allclose(P1 - P0, expect, atol=2e-2)


@pytest.mark.gpu
def test_cpg_steps_push_one_tick(qs):
    """qs_cpg_steps (action_repeat = 1) honours a push: one pushed tick against the oracle from the same torques"""
    from oracle import oracle as O
    from test_gpu_parity import TOL_F32
    n = 128
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, isRLGymInterface=False, action_repeat=1, motor_control_mode="TORQUE",
                                    enable_springs=True, auto_reset=False, seed=4)
    env.reset()
    cpg = qs.HopfNetwork(num_envs=n, gait="TROT", omega_swing=16 * np.pi, omega_stance=4 * np.pi, time_step=0.001, seed=1)
    for _ in range(5):
        cpg.drive(env, 1)
    rng = np.random.default_rng(6)
    F = (rng.normal(size=(n, 3)) * 100).astype(np.float32).astype(np.float64)
    p = (rng.uniform(-1, 1, (n, 3)) * TRUNK_HALF).astype(np.float32).astype(np.float64)
    S0 = env.get_state().cpu().numpy().astype(np.float64)
    mu = env._views["mu"].cpu().numpy().astype(np.float64)
    env.robot.apply_external_force(F, p, n_ticks=1)
    cpg.drive(env, 1)
    got = env.get_state().cpu().numpy().astype(np.float64)
    tm = env._views["tau_motor"].cpu().numpy().T.astype(np.float64)
    ts = env._views["tau_spring"].cpu().numpy().T.astype(np.float64)
    assert int(env.robot.get_external_force()[2].abs().sum()) == 0
    w = O.World()
    err = np.zeros((n, 37))
    for i in range(n):
        w.set_params(mu_ground=mu[i])
        w.set_state(S0[i])
        _pushed_step(w, tm[i] + ts[i], F[i], p[i])
        err[i] = np.abs(got[i] - w.get_state())
    ok = err[:, 13:25].max(1) < 1e-3
    assert ok.mean() > 0.95
    for s, t in zip(SL, TOL_F32):
        assert err[ok][:, s].max() < 3 * t, (s, err[ok][:, s].max())


@pytest.mark.gpu
def test_push_api_errors_and_clear(qs):
    n = 16
    kw = dict(num_envs=n, auto_reset=False, enable_noise=False, seed=2, **JIP)
    a, b = qs.BatchedQuadrupedGymEnv(**kw), qs.BatchedQuadrupedGymEnv(**kw)
    a.reset(), b.reset()
    r = a.robot
    for bad in (dict(force=[1.0, 2.0]), dict(force=np.zeros((3, 3))), dict(force=[0, 0, float("nan")]),
                dict(force=[0, 0, 1.0], position=[0.0, 0.0]), dict(force=[0, 0, 1.0], n_ticks=-1),
                dict(force=[0, 0, 1.0], n_ticks=1.5), dict(force=[0, 0, 1.0], env_ids=[0, 16]),
                dict(force=[0, 0, 1.0], env_ids=[-1]), dict(force=[0, 0, 1.0], env_ids=[2, 2]),
                dict(force=[0, 0, 1.0], env_ids=np.ones(n - 1, bool)), dict(force=[0, 0, 1.0], n_ticks=[1, 2])):
        with pytest.raises(ValueError):
            r.apply_external_force(**bad)
    assert r.get_external_force() is None
    with pytest.raises(ValueError):            # exactly one buffer: QS_ERR_ARG
        from quadruped_springs_b200 import _lib
        t = torch.zeros(n, dtype=torch.int32, device="cuda")
        _lib.check(a._L.qs_set_external_force(a._h, None, t.data_ptr()))
    zero = cuda(np.zeros((n, a.action_dim)))
    r.apply_external_force([0.0, 80.0, 0.0], n_ticks=100)
    for _ in range(3):
        a.step(zero), b.step(zero)
    assert not torch.equal(a._views["state"], b._views["state"])
    # clear: back to the default kernels; a state copied over from the twin then runs bit for bit like it
    r.clear_external_force()
    assert r.get_external_force() is None
    a.set_state(b.get_state())
    b.set_state(b.get_state())
    for _ in range(5):
        a.step(zero), b.step(zero)
    assert torch.equal(a._views["state"], b._views["state"])
