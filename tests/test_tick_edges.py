"""The physics tick at its edges, against the fp64 oracle.

The other parity tests draw their states from `_random_states` and `_general_states` (test_gpu_parity.py), which never
reach the places where a fixed-size, hand-unrolled tick breaks.  This file builds one labelled corpus that does, and lets
the oracle decide what each group covers:

- capacity: every one of the 18 collision shapes (trunk, imu_link, and a hip, thigh, calf and foot per leg) inside its
  contact threshold at once, upright and upside down, with 0, 6 or 12 joints past a limit (up to 12 limit rows + 18
  contacts = 66 rows of the general solver); and 17-shape states, one shape short of that.  physics_tick_general keeps
  its candidates and rows in fixed arrays of QS_MAX_CONTACTS entries, which must hold all 18.
- feet: each of the 15 non-empty foot masks, the chosen feet just inside their threshold and the others well up, no joint
  at a limit and no body shape near the ground: the packed fast tick (two legs at a time) runs them, and its per-foot
  selects, warm start and impulse application see every subset.  Some swing their raised feet down during the run.
- sliding: feet states with a tangential base velocity of 1-3 m/s on low friction: the friction cone binds.
- clamp: joints at |qd| around the +-30.1 rad/s clamp with torques pushing them further, airborne and touching.

Over the runs the contact history changes: feet lift off with a warm-start history and touch down without one.

CPU: tools/push_host_check.cu (fp64 tick templates on the host, zero push) built with AddressSanitizer and UBSan runs the
corpus, and its default-instantiation rows are held to the oracle tick by tick.  GPU: qs_debug_ticks in fp64 and fp32,
both sides carrying the contact history from tick to tick, and the step (k_step / k_step_contact / k_step_slow) through
the substep trace, under the dispatch switches QS_SLOW_SPREAD 1 and 32 as well."""
import json
import os
import subprocess
from collections import namedtuple

import numpy as np
import pytest
import torch

from test_external_force import NVCC, SL, _host_run
from test_gpu_parity import TOL_F32, TOL_F64
from test_substep_trace import FOOT_LINKS, JIP, OracleTicks, _counters, _TickCompare

LO = np.array([-1.0471975512, -0.663225115758, -2.72271363311] * 4)   # go1.urdf joint limits
HI = np.array([1.0471975512, 2.96705972839, -0.837758040957] * 4)
STAND = np.array([0, np.pi / 4, -np.pi / 2] * 4)
FOOT_BODIES = (6, 10, 14, 18)      # the oracle's link indices of the four feet (World.link_pose)
FOOT_R = 0.02
N_SHAPES = 18
MCV = 30.1                          # max_coord_vel of the oracle's World
# The kernels take the solver's parameters in fp32 (SolverConst: 30.1f, 0.08f, ...).  Robots sunk up to 0.37 m drive
# the 18 contacts' targets to the velocity clamp, where 30.1f - 30.1 = 3.8e-7, and the coupled rows spread that: the fp64
# tick of a capacity state is within 2.1 x TOL_F64 of the oracle, the other groups within 0.7 x.
CAP_F64 = 3.0


# ------------------------------------------------------------------ the corpus
def _f32(s):
    return np.asarray(s, np.float64).astype(np.float32).astype(np.float64)


class _Probe:
    """what the oracle sees in a pose: its contacts (one World.step, whose collision phase runs on the pose at the start
    of the tick) and the lowest points of the feet"""

    def __init__(self):
        from oracle import oracle as O
        self.w = O.World()

    def contacts(self, s):
        self.w.set_state(s)
        self.w.step(np.zeros(12))
        return self.w.contacts(), self.w.last_rows

    def count(self, s):
        return len(self.contacts(s)[0])

    def feet(self, s):
        """heights of the lowest points of the four foot spheres"""
        self.w.set_state(s)
        return np.array([self.w.link_pose(b)[1][2] - FOOT_R for b in FOOT_BODIES])

    def z_for(self, s, n_min, lo=-1.5, hi=1.5):
        """the largest base height (to 1e-5 m) at which at least n_min shapes are inside their thresholds; every shape's
        gap grows with the base height, so the count falls as it rises"""
        s = s.copy()
        for _ in range(20):
            s[2] = 0.5 * (lo + hi)
            if self.count(s) >= n_min:
                lo = s[2]
            else:
                hi = s[2]
        return lo


def _random_quat(rng, upside_down, spread):
    base = np.array([1.0, 0, 0, 0]) if upside_down else np.array([0, 0, 0, 1.0])   # (x, y, z, w): pi about x, identity
    q = base + rng.normal(size=4) * spread
    return q / np.linalg.norm(q)


def _capacity(rng, P):
    """(kind, state) of the capacity group: all 18 shapes at least 2 mm inside their thresholds (the count is
    still 18 with the base 2 mm higher), with 0, 6 or 12 joints 0.005-0.03 rad past a limit; and states with exactly 17
    shapes inside, 2 mm clear of both neighbouring counts"""
    out = []
    for i in range(48):
        upside_down = i % 2 == 1
        n_lim = (0, 6, 12)[(i // 2) % 3]
        s = np.zeros(37)
        s[3:7] = _random_quat(rng, upside_down, 0.08)
        q = np.clip(STAND + rng.normal(size=12) * 0.3, LO + 0.05, HI - 0.05)
        past = rng.permutation(12)[:n_lim]
        side = rng.random(n_lim) < 0.5
        q[past] = np.where(side, HI[past] + rng.uniform(0.005, 0.03, n_lim), LO[past] - rng.uniform(0.005, 0.03, n_lim))
        s[13:25] = q
        s[7:13] = rng.normal(size=6) * 0.5
        s[25:37] = rng.normal(size=12) * 3
        if i < 36:
            s[2] = P.z_for(s, N_SHAPES) - 0.002 - rng.uniform(0, 0.004)
            out.append(("cap18", s))
        else:   # one shape short of all
            z18, z17 = P.z_for(s, N_SHAPES), P.z_for(s, N_SHAPES - 1)
            if z17 - z18 < 0.006:
                continue
            s[2] = rng.uniform(z18 + 0.002, z17 - 0.002)   # float32 storage moves it by < 1e-7
            out.append(("cap17", s))
    return out


def _foot_state(rng, P, mask, landing=False, tries=40):
    """the feet of `mask` with gaps in [-2, -0.2] mm, the other feet at least 2 cm up; no joint within 0.15 rad of a
    limit.  landing: the raised feet swing down, so that they touch down within the run.  None if it fails."""
    for _ in range(tries):
        s = np.zeros(37)
        s[3:7] = _random_quat(rng, False, 0.04)
        s[13:25] = np.clip(STAND + rng.normal(size=12) * 0.12, LO + 0.2, HI - 0.2)
        s[2] = 1.0
        down = [k for k in range(4) if mask >> k & 1]
        s[2] -= P.feet(s)[down].min() + 0.001
        # each foot onto its own height, the chosen ones just inside their threshold, the others 2-3.5 cm up: the calf
        # moves the foot mostly along the leg (secant steps)
        target = np.where([mask >> k & 1 for k in range(4)], -rng.uniform(0.0002, 0.002, 4), rng.uniform(0.0205, 0.035, 4))
        for k in range(4):
            j = 13 + 3 * k + 2
            for _ in range(8):
                h0 = P.feet(s)[k] - target[k]
                if abs(h0) < 2e-5:
                    break
                s[j] += 1e-3
                h1 = P.feet(s)[k] - target[k]
                s[j] -= 1e-3
                if abs(h1 - h0) < 1e-9:
                    break
                s[j] -= h0 * 1e-3 / (h1 - h0)
        s[7:13] = rng.normal(size=6) * np.array([0.2, 0.2, 0.2, 0.5, 0.5, 0.5])
        s[25:37] = rng.normal(size=12) * 1.5
        if landing:       # swing each raised foot down at 3.5-5 m/s (least-norm joint rates along the foot's height)
            for k in range(4):
                if not mask >> k & 1:
                    h0, J = P.feet(s)[k], np.zeros(3)
                    for j in range(3):
                        s[13 + 3 * k + j] += 1e-6
                        J[j] = (P.feet(s)[k] - h0) / 1e-6
                        s[13 + 3 * k + j] -= 1e-6
                    s[25 + 3 * k:28 + 3 * k] = -rng.uniform(3.5, 5.0) * J / (J @ J)
        s = _f32(s)
        g = P.feet(s)
        if not ((s[13:25] > LO + 0.15).all() and (s[13:25] < HI - 0.15).all()):
            continue
        if not all(-0.002 <= g[k] <= -0.0002 if mask >> k & 1 else g[k] >= 0.02 for k in range(4)):
            continue
        cts, rows = P.contacts(s)
        if sorted(c[0] for c in cts) != [FOOT_LINKS[k] for k in down] or rows[0] != 0:
            continue
        low = s.copy()
        low[2] -= 0.01                       # no body shape within 1 cm of its threshold
        if any(c[0] not in FOOT_LINKS for c in P.contacts(low)[0]):
            continue
        return s
    return None


Case = namedtuple("Case", "group kind n_ticks mu s tau mask")   # mask: the feet the state was built to touch with (-1: any)


def corpus(seed=0):
    """[Case], in float32-representable values"""
    rng = np.random.default_rng(seed)
    P = _Probe()
    out = []
    for kind, s in _capacity(rng, P):
        s = _f32(s)
        mu, tau = rng.uniform(0.3, 1.0), rng.normal(size=12) * 5
        for n_ticks in (1, 3):
            out.append(("capacity", kind, n_ticks, mu, s, tau, -1))
    for mask in range(1, 16):
        for i in range(10):
            s = _foot_state(rng, P, mask, landing=i >= 7)
            assert s is not None, mask
            out.append(("feet", "landing" if i >= 7 else "mask", 10, rng.uniform(0.5, 1.0), s, rng.normal(size=12) * 5, mask))
    for i in range(45):
        mask = int(rng.integers(1, 16))
        s = _foot_state(rng, P, mask)
        a = rng.uniform(0, 2 * np.pi)
        s[7:9] = rng.uniform(1.0, 3.0) * np.array([np.cos(a), np.sin(a)])
        out.append(("sliding", "slide", 10, rng.uniform(0.1, 0.3), s, rng.normal(size=12) * 5, mask))
    from oracle import oracle as O
    w, n_clamp, i = O.World(), 0, 0
    while n_clamp < 40:
        i += 1
        touching = i % 2 == 1
        mask = int(rng.integers(1, 16)) if touching else 0
        if touching:
            s = _foot_state(rng, P, mask)
        else:
            s = np.zeros(37)
            s[3:7] = _random_quat(rng, False, 0.3)
            s[2] = 1.5
            s[13:25] = STAND + rng.normal(size=12) * 0.15
            s[7:13] = rng.normal(size=6) * 0.5
            s[25:37] = rng.normal(size=12) * 1.5
        tau = rng.normal(size=12) * 3
        fast = rng.permutation(12)[:rng.integers(2, 5)]
        sign = np.where(rng.random(len(fast)) < 0.5, -1.0, 1.0)
        s[25 + fast] = sign * rng.uniform(29.5, 31.0, len(fast))
        tau[fast] = sign * rng.uniform(10.0, 30.0, len(fast))
        mu = rng.uniform(0.5, 1.0)
        if (np.abs(OracleRun(w, mu, _f32(s), _f32(tau), 10).state[:, 25:37]) == MCV).any():   # the clamp binds
            out.append(("clamp", "touch" if touching else "air", 10, mu, s, tau, mask))
            n_clamp += 1
    return [Case(g, k, n, float(np.float32(mu)), _f32(s), _f32(tau), m) for g, k, n, mu, s, tau, m in out]


class OracleRun:
    """the oracle World tick by tick on a corpus entry: states [n_ticks, 37], foot masks, invalid counts, rows"""

    def __init__(self, w, mu, s, tau, n_ticks):
        w.set_params(mu_ground=mu)
        w.set_state(s)
        self.state = np.zeros((n_ticks, 37))
        self.mask = np.zeros(n_ticks, int)
        self.invalid = np.zeros(n_ticks, int)
        self.rows = []
        for t in range(n_ticks):
            w.step(tau)
            self.state[t] = w.get_state()
            for link, nf, dist, pos in w.contacts():
                if link in FOOT_LINKS:
                    self.mask[t] |= 1 << FOOT_LINKS.index(link)
                else:
                    self.invalid[t] += 1
            self.rows.append(w.last_rows)


_CORPUS = {}


def _labelled(seed=0):
    """the corpus with its oracle runs, and what the oracle says it covers"""
    if seed not in _CORPUS:
        from oracle import oracle as O
        cases = corpus(seed)
        w = O.World()
        runs = [OracleRun(w, c.mu, c.s, c.tau, c.n_ticks) for c in cases]
        _CORPUS[seed] = (cases, runs, _coverage(cases, runs))
    return _CORPUS[seed]


def _coverage(cases, runs):
    masks = np.zeros(16, int)
    lift = touch = clamp_hits = cap18 = cap17 = most = 0
    for (g, kind, n, mu, s, tau, m), r in zip(cases, runs):
        if g == "feet":
            masks[r.mask[0]] += 1
        if g == "capacity":
            cap18 += r.rows[0][1] == N_SHAPES
            cap17 += r.rows[0][1] == N_SHAPES - 1
            most = max(most, r.rows[0][0] + 3 * r.rows[0][1])
        if g == "clamp":
            clamp_hits += bool((np.abs(r.state[:, 25:37]) == MCV).any())
        if n > 1 and g != "capacity":
            prev, now = r.mask[:-1], r.mask[1:]
            lift += sum(bin(x).count("1") for x in (prev & ~now))        # a foot with a history lets go
            touch += sum(bin(x).count("1") for x in (now & ~prev))       # a foot without one comes down
    return dict(masks_seen=int((masks[1:] > 0).sum()), min_per_mask=int(masks[1:].min()), lift_offs=int(lift),
                touch_downs=int(touch), clamp_hits=int(clamp_hits), states_at_18=int(cap18), states_at_17=int(cap17),
                most_rows=int(most))


def test_corpus_covers_the_edges():
    """what each group reaches, as the oracle sees it"""
    cases, runs, cov = _labelled()
    groups = [c.group for c in cases]
    for c, r in zip(cases, runs):
        if c.kind == "cap18":
            assert r.rows[0][1] == N_SHAPES, r.rows[0]
        if c.kind == "cap17":
            assert r.rows[0][1] == N_SHAPES - 1, r.rows[0]
        if c.mask >= 0:   # the oracle's first-tick contact set is the mask the state was built for, and only feet touch
            assert r.mask[0] == c.mask and r.invalid[0] == 0 and r.rows[0] == (0, bin(c.mask).count("1")), (c.kind, r.rows[0])
        if c.group == "clamp":
            assert (np.abs(r.state[:, 25:37]) == MCV).any(), c.kind          # the clamp binds on some tick
    seen = np.bincount([c.mask for c in cases if c.group == "feet"], minlength=16)
    assert seen[0] == 0 and (seen[1:] >= 8).all(), seen
    assert cov["most_rows"] == 12 + 3 * N_SHAPES
    assert cov["states_at_18"] >= 60 and cov["states_at_17"] >= 4
    assert cov["lift_offs"] >= 50 and cov["touch_downs"] >= 50, cov
    assert cov["clamp_hits"] == groups.count("clamp")
    assert groups.count("sliding") >= 40
    print(json.dumps(dict(test="corpus", states=len(cases), **cov)))


# ------------------------------------------------------------------ CPU: the tick templates on the host, sanitized
SAN = ["-g", "-Xcompiler", "-fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer", "-lasan", "-lubsan"]


def _sanitizers_link(tmp):
    src, exe = os.path.join(tmp, "trivial.cu"), os.path.join(tmp, "trivial")
    with open(src, "w") as f:
        f.write("int main() { return 0; }\n")
    res = subprocess.run([NVCC, "-std=c++17", "-w", *SAN, "-o", exe, src], capture_output=True, text=True)
    return res.returncode == 0 and subprocess.run([exe], capture_output=True).returncode == 0


def _host_rc(tmp, tag):
    """the fast tick's return code of every D row (0: it ran the tick; 1: it handed it to the general solver)"""
    rc = {}
    for line in open(os.path.join(tmp, f"{tag}_out.txt")):
        t = line.split()
        if t[0] == "D":
            rc.setdefault(int(t[1]), []).append(int(t[3]))
    return rc


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not found")
@pytest.mark.parametrize("pack", [1, 0])
def test_tick_edges_on_host_sanitized(tmp_path, monkeypatch, pack):
    """tools/push_host_check.cu (no push) under AddressSanitizer and UBSan over the whole corpus: no error report, and
    every tick of the default instantiation (fast tick, general solver when it asks) within TOL_F64 of the oracle.
    The 18-shape states overflowed the general solver's contact arrays while they held 17."""
    tmp = str(tmp_path)
    if not _sanitizers_link(tmp):
        pytest.skip("the AddressSanitizer / UBSan runtimes do not link here")
    log = os.path.join(tmp, "san")
    monkeypatch.setenv("ASAN_OPTIONS", f"detect_leaks=0:log_path={log}")
    monkeypatch.setenv("UBSAN_OPTIONS", f"print_stacktrace=1:log_path={log}")
    cases, runs, cov = _labelled()
    z3 = np.zeros(3)
    tag = f"san{pack}"
    reports = lambda: "".join(open(os.path.join(tmp, f)).read() for f in os.listdir(tmp) if f.startswith("san."))
    try:
        rows = _host_run(tmp, tag, SAN + ([] if pack else ["-DQS_PACK_LEGS=0"]),
                         [(c.kind, c.n_ticks, c.mu, c.s, c.tau, z3, z3) for c in cases])
    except AssertionError:   # a sanitizer error ends the run: show its report
        raise AssertionError(reports()[-4000:])
    assert "AddressSanitizer" not in reports() and "runtime error" not in reports(), reports()[-4000:]
    rc = _host_rc(tmp, tag)
    worst = 0.0
    for i, (c, r) in enumerate(zip(cases, runs)):
        assert rows["Z"][i] == rows["D"][i], (c.group, c.kind, i)        # the kExt instantiation with no push
        got = np.array(rows["D"][i], float)
        assert got.shape == (c.n_ticks, 37)
        if c.group in ("feet", "sliding") and c.kind != "landing":
            assert rc[i] == [0] * c.n_ticks, (c.kind, i, rc[i])              # the fast tick ran every tick
        if c.group == "capacity":
            assert rc[i][0] == 1
        scale = CAP_F64 if c.group == "capacity" else 1.0
        for t in range(c.n_ticks):
            for sl, tol in zip(SL, TOL_F64):
                err = float(np.abs(got[t][sl] - r.state[t][sl]).max())
                worst = max(worst, err / (tol * scale))
                assert err < tol * scale, (c.group, c.kind, i, t, sl, err)
    print(json.dumps(dict(test="host", pack=pack, worst_over_tol=worst, **cov)))


# ------------------------------------------------------------------ GPU
def cuda(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32, device="cuda")


@pytest.fixture(scope="module")
def qs():
    import quadruped_springs_b200 as m
    assert torch.cuda.is_available()
    return m


def _gpu_cases():
    """the corpus without the 1-tick copies of the capacity states (their first tick is the 3-tick run's)"""
    cases, runs, cov = _labelled()
    keep = [i for i, c in enumerate(cases) if not (c.group == "capacity" and c.n_ticks == 1)]
    return [cases[i] for i in keep], [runs[i] for i in keep], cov


@pytest.mark.gpu
@pytest.mark.parametrize("use_f64", [1, 0])
def test_debug_ticks_at_the_edges_match_oracle(qs, use_f64):
    """qs_debug_ticks against the oracle World tick by tick, both sides carrying the contact history (mask, impulses)
    from the same cold start.  fp32: one tick per call, so that the history also goes through the env's stored contact
    word and foot forces between ticks as it does between steps; TOL_F32 on the fast groups (widened with the tick like
    the trace comparison) and the bounds of test_general_solver_matches_oracle on the capacity states.  fp64: tick t is
    the state after one call of t + 1 ticks from the start, so that nothing is rounded to fp32 between ticks (a one-tick
    call stores the state and impulses in fp32, and the contact rows amplify that rounding past TOL_F64); TOL_F64, and
    CAP_F64 x TOL_F64 on the capacity states.  Capacity states must agree on the foot bits and the invalid count
    exactly; elsewhere the foot bits must agree on 98 % of the states, and a state is compared while they do."""
    cases, runs, cov = _gpu_cases()
    n, T = len(cases), max(c.n_ticks for c in cases)
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, enable_noise=False, auto_reset=False, **JIP)
    S = cuda([c.s for c in cases])
    env.set_state(S)
    env._views["mu"][:] = cuda([c.mu for c in cases])
    tau = cuda([c.tau for c in cases])
    alive = np.ones(n, bool)
    cap = np.array([c.group == "capacity" for c in cases])
    cap_err, worst = [], {}
    for t in range(T):
        if use_f64:
            env.set_state(S)                 # also clears the contact history, as the oracle's set_state does
            env.debug_ticks(tau, t + 1, 1)
        else:
            env.debug_ticks(tau, 1, 0)
        got = env.get_state().cpu().numpy().astype(np.float64)
        word = env._views["contact"].cpu().numpy()
        for i, (c, r) in enumerate(zip(cases, runs)):
            if t >= c.n_ticks or not alive[i]:
                continue
            if c.group == "capacity":
                assert (word[i] & 15, word[i] >> 8) == (r.mask[t], r.invalid[t]), (c.kind, i, t, word[i])
            elif word[i] & 15 != r.mask[t]:
                alive[i] = False
                continue
            if c.group == "capacity" and not use_f64:
                cap_err.append(np.abs(got[i] - r.state[t]))
                continue
            scale = CAP_F64 if c.group == "capacity" else 1.0 + 2.0 * t / 9.0
            for q, (sl, tol) in enumerate(zip(SL, TOL_F64 if use_f64 else TOL_F32)):
                err = float(np.abs(got[i][sl] - r.state[t][sl]).max())
                worst[q] = max(worst.get(q, 0.0), err / (tol * scale))
                assert err < tol * scale, (c.group, c.kind, i, t, sl, err)
    assert alive[~cap].mean() >= 0.98, alive[~cap].mean()
    if cap_err:   # fp32 on the general solver: stiff impacts, the bounds of test_general_solver_matches_oracle
        err = np.array(cap_err)
        assert err[:, :7].max() < 2e-4 and err[:, 13:25].max() < 1e-3, (err[:, :7].max(), err[:, 13:25].max())
        assert np.quantile(err[:, 25:], 0.99) < 5e-2 and np.quantile(err[:, 7:13], 0.99) < 5e-3
        worst["cap_pos"] = float(err[:, :7].max() / 2e-4)
    print(json.dumps(dict(test="debug_ticks", use_f64=use_f64, states=n, bits_agree=float(alive[~cap].mean()),
                          worst_over_tol={str(k): v for k, v in worst.items()}, **cov)))


def _step_run(qs, monkeypatch, cases, act, env_vars=None):
    """set_state, one traced step of every env; the trace [10, 66, n], the done flags and the general-solver count"""
    for k, v in (env_vars or {}).items():
        monkeypatch.setenv(k, str(v))
    try:
        env = qs.BatchedQuadrupedGymEnv(num_envs=len(cases), enable_noise=False, auto_reset=False, **JIP)
    finally:
        for k in env_vars or {}:
            monkeypatch.delenv(k)
    env.reset()
    env.set_state(cuda([c.s for c in cases]))
    env._views["mu"][:] = cuda([c.mu for c in cases])
    tr = env.set_substep_trace(torch.arange(len(cases)))
    _, _, done, _ = env.step(cuda(act))
    torch.cuda.synchronize()
    return tr.clone(), done.cpu().numpy().astype(bool), _counters(env)[0], {k: env._views[k].clone() for k in
                                                                        ("state", "contact", "foot_force")}


@pytest.mark.gpu
def test_step_at_the_edges_matches_oracle(qs, monkeypatch):
    """set_state, then one step of every corpus state with every env traced: each tick row against OracleTicks through
    _TickCompare.  Every capacity env runs in k_step_slow and ends its episode (an invalid contact).  The dispatch
    switches QS_SLOW_SPREAD=1 and 32 give the same bits."""
    cases, _, cov = _gpu_cases()
    n = len(cases)
    rng = np.random.default_rng(5)
    act = rng.uniform(-1, 1, size=(n, 6)).astype(np.float32).astype(np.float64)
    tr, done, general, views = _step_run(qs, monkeypatch, cases, act)
    cap = np.array([c.group == "capacity" for c in cases])
    got = tr.double().cpu().numpy()
    assert (got[0, 65][cap].astype(int) >> 8 > 0).all()                 # an invalid contact on the first tick
    assert general >= cap.sum() and done[cap].all(), (general, cap.sum(), done[cap].mean())
    ref = OracleTicks(**JIP)
    cmp = _TickCompare()
    for i, c in enumerate(cases):
        ref.world.set_params(mu_ground=c.mu)
        ref.world.set_state(c.s)
        rec = ref.step(act[i])
        hard = c.group == "capacity" or (got[:, 65, i].astype(int) >> 8 > 0).any() or (rec[:, 65].astype(int) >> 8 > 0).any() \
            or any((rec[t, 13:25] <= LO).any() or (rec[t, 13:25] >= HI).any() for t in range(10)) \
            or (c.s[13:25] <= LO).any() or (c.s[13:25] >= HI).any()
        cmp.add(got[:, :, i], rec, hard)
    cmp.check()
    for spread in (1, 32):
        tr2, done2, general2, views2 = _step_run(qs, monkeypatch, cases, act, {"QS_SLOW_SPREAD": spread})
        assert torch.equal(tr2.view(torch.int32), tr.view(torch.int32)), spread
        assert np.array_equal(done2, done) and general2 == general, spread
        for k in views:
            assert torch.equal(views2[k], views[k]), (spread, k)
    print(json.dumps(dict(test="step", states=n, general=int(general), capacity=int(cap.sum()),
                          same_bits=cmp.same / cmp.ticks, compared=cmp.compared,
                          worst_over_tol={f"{'general' if k[0] else 'fast'}_{k[1]}": v for k, v in cmp.worst.items()},
                          **cov)))
