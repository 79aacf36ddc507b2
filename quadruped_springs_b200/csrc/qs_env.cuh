// qs_env.cuh -- per-env control-step logic around the physics tick: motor +
// PEA torques per substep, jumping-task bookkeeping, rewards, terminations and
// observation assembly (fp32).  Restates, per env and in registers, what the
// reference does in Python after its ten stepSimulation calls
// (quadruped_gym_env.py:239-256).
#pragma once
#include "qs_physics.cuh"

namespace qs {

// ---------------------------------------------------------------- Philox4x32-10
QS_DEVONLY void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
QS_DEVONLY float u01(uint32_t x) { return (float(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }  // (0,1)
// four N(0,1) samples for (stream, step, block)
QS_DEVONLY void normal4(uint64_t seed, uint64_t gid, uint32_t epoch, uint32_t step, uint32_t blk, float* n) {
  uint32_t r[4];
  philox4x32(uint32_t(gid), uint32_t(gid >> 32) ^ (blk << 16), step, epoch, uint32_t(seed), uint32_t(seed >> 32), r);
  float s, c;
  float m = sqrtf(-2.0f * __logf(u01(r[0])));
  sincospif(2.0f * u01(r[1]), &s, &c);
  n[0] = m * c; n[1] = m * s;
  m = sqrtf(-2.0f * __logf(u01(r[2])));
  sincospif(2.0f * u01(r[3]), &s, &c);
  n[2] = m * c; n[3] = m * s;
}
QS_DEVONLY float uniform1(uint64_t seed, uint64_t gid, uint32_t epoch, uint32_t blk) {
  uint32_t r[4];
  philox4x32(uint32_t(gid), uint32_t(gid >> 32) ^ (blk << 16), 0xFFFFFFFFu, epoch, uint32_t(seed), uint32_t(seed >> 32), r);
  return float(r[0] >> 8) * (1.0f / 16777216.0f);  // [0,1) like np.random.random
}

// ---------------------------------------------------------------- substeps
struct EnvCfg {
  int enable_springs, control_mode, action_mode, task, obs_mode, action_repeat, is_rl, enable_filter;
  int enable_noise, obs_dim, action_dim, settling_steps, ground_randomizer, auto_reset, landing_mode, spring_randomizer, rest_mode, mass_randomizer;
  float max_episode_time, mu_ground, leg_mass_err, payload_max, payload_pos[3], spring_err;
  const float* demo;  // [demo_len][action_dim] demonstration actions of the *_DEMO tasks (device)
  int demo_len;
  uint64_t seed;
  int64_t gid0;
};

// PD + PEA torque of one tick (quadruped.py:288-320, quadruped_motor.py:45-104)
__device__ __forceinline__ void tick_torques(const EnvState<float>& st, const float* cmd, bool torque_mode, int env,
                                             const DeviceView& D, const EnvCfg& C, const RobotConst& RC, const float* sk,
                                             const float* sb, const float* sr, float* tau, float* tau_m, float* tau_s,
                                             bool custom_gains) {
  const int n = D.n;
  if (custom_gains) {  // gains swapped at run time for this env (landing wrappers, landing_wrapper.py:21-33)
#pragma unroll
    for (int i = 0; i < 12; i++) {
      const float kp = D.kp[i * n + env], kd = D.kd[i * n + env];
      tau_m[i] = pd_torque1(kp, kd, RC.tau_max[i], cmd[i], st.q[i], st.qd[i], torque_mode);
    }
  } else {             // config gains straight from the constant bank: no global loads on the per-tick path
#pragma unroll
    for (int i = 0; i < 12; i++) tau_m[i] = pd_torque1(RC.kp[i], RC.kd[i], RC.tau_max[i], cmd[i], st.q[i], st.qd[i], torque_mode);
  }
#pragma unroll
  for (int i = 0; i < 12; i++) tau[i] = tau_m[i];
  if (C.enable_springs) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      spring_torque_leg(k, sk, sb, sr, st.q + 3 * k, st.qd + 3 * k, tau_s + 3 * k);
#pragma unroll
      for (int j = 0; j < 3; j++) tau[3 * k + j] += tau_s[3 * k + j];
    }
  } else {
#pragma unroll
    for (int i = 0; i < 12; i++) tau_s[i] = 0.f;
  }
}

QS_DEVONLY void load_springs(const DeviceView& D, int env, float* sk, float* sb, float* sr) {
  const int n = D.n;
#pragma unroll
  for (int j = 0; j < 3; j++) {
    sk[j] = D.spring[(0 + j) * n + env];
    sb[j] = D.spring[(3 + j) * n + env];
    sr[j] = D.spring[(6 + j) * n + env];
  }
}

// ---------------------------------------------------------------- per-substep trace (qs_set_substep_trace)
// buf[t][QS_TRACE_DIM][n_traced]: row t = the values after tick t of the step -- state (store_state's 37 words), the
// motor and spring torques applied in that tick, foot normal forces (0 off contact), contact word.  A tick handed over
// to another kernel (TICK_NEEDS_*) is run again by that kernel from the same state, which then owns its row.
struct SubstepTrace {
  float* buf;          // nullptr: no trace
  int32_t* col;        // [N]: the env's column, -1 when it is not traced
  int n_traced;
};
// one env's column of the trace: p = &buf[0][0][col], or nullptr when the env is not traced (or the thread has no env)
struct TraceColumn {
  float* p;
  int w;   // n_traced: distance between two rows
  QS_DEVONLY float* row(int t, int r) const { return p + (size_t(t) * QS_TRACE_DIM + r) * size_t(w); }
  QS_DEVONLY void torques(int t, const float* tm, const float* ts) const {
    if (!p) return;
#pragma unroll
    for (int i = 0; i < 12; i++) { *row(t, QS_TR_TAU_MOTOR + i) = tm[i]; *row(t, QS_TR_TAU_SPRING + i) = ts[i]; }
  }
  QS_DEVONLY void state(int t, const EnvState<float>& st, const ContactState<float>& cs, float dt) const {
    if (!p) return;
#pragma unroll
    for (int i = 0; i < 3; i++) *row(t, QS_TR_STATE + i) = st.pos[i];
#pragma unroll
    for (int i = 0; i < 4; i++) *row(t, QS_TR_STATE + 3 + i) = st.quat[i];
#pragma unroll
    for (int i = 0; i < 3; i++) { *row(t, QS_TR_STATE + 7 + i) = st.vlin[i]; *row(t, QS_TR_STATE + 10 + i) = st.vang[i]; }
#pragma unroll
    for (int i = 0; i < 12; i++) { *row(t, QS_TR_STATE + 13 + i) = st.q[i]; *row(t, QS_TR_STATE + 25 + i) = st.qd[i]; }
#pragma unroll
    for (int k = 0; k < 4; k++) *row(t, QS_TR_FOOT_FORCE + k) = (cs.mask >> k) & 1 ? cs.lam_n[k] / dt : 0.f;
    *row(t, QS_TR_CONTACT) = float((cs.mask & 15) | (cs.invalid << 8));
  }
};
QS_DEVONLY TraceColumn trace_column(const SubstepTrace& tr, int env, bool live) {
  const int c = live ? tr.col[env] : -1;
  return TraceColumn{c >= 0 ? tr.buf + c : nullptr, tr.n_traced};
}

// ---------------------------------------------------------------- external push on the base (qs_set_external_force)
// Caller-owned: wrench[QS_EXT_DIM][N] (force xyz, world frame, N; point xyz, base frame from the base position, m) and
// ticks[N], the ticks the push still lasts.  Every kernel that runs ticks of a step reads the count as of the start of
// the step (k_ext_countdown consumes it once the step is over), so a tick handed over to another kernel is pushed once.
struct ExtForce {
  const float* wrench;   // nullptr: no push buffer
  int32_t* ticks;
};
// one env's push for the ticks of this step: tick t is pushed iff t < n
struct ExtPush {
  ExtWrench<float> w;
  int n;
  QS_DEVONLY const ExtWrench<float>* at(int t) const { return t < n ? &w : nullptr; }
};
QS_DEVONLY ExtPush ext_push(const ExtForce& ef, int env, int n_envs) {
  ExtPush e;
  e.n = ef.ticks[env];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    e.w.f[i] = e.n > 0 ? ef.wrench[size_t(i) * n_envs + env] : 0.f;
    e.w.p[i] = e.n > 0 ? ef.wrench[size_t(3 + i) * n_envs + env] : 0.f;
  }
  return e;
}
// (the variadic tail of run_ticks_general: the trace column first, the push last)
template <typename A, typename... R> QS_DEVONLY A first_of(A a, R...) { return a; }
template <typename A> QS_DEVONLY A last_of(A a) { return a; }
template <typename A, typename B, typename... R> QS_DEVONLY auto last_of(A, B b, R... r) { return last_of(b, r...); }

// ApplyAction + stepSimulation for ticks [t0, n_ticks) (quadruped_gym_env.py:207-219).
// cmd = desired joint angles (PD) or torques (TORQUE).  Returns n_ticks when all ticks ran,
// or the index of the tick that needs another solver (state untouched by that tick; *why =
// TICK_NEEDS_GENERAL / TICK_NEEDS_CONTACT).  kContacts = false is the flight variant: it
// hands the env over as soon as a foot comes within its contact threshold.
// block size of the step / reset / settle kernels: a compile-time constant so that the per-leg scratch is addressed
// with immediate offsets (qs_physics.cuh Scratch)
constexpr int QS_BLOCK = 128;
using StepScratch = Scratch<float, QS_BLOCK>;

// kTrace: each tick this thread completes goes to its trace column `tc`.  kExt: `push` acts on the ticks it covers.
template <bool kContacts, bool kEM, bool kTrace = false, bool kExt = false>
__device__ __forceinline__ int run_ticks(EnvState<float>& st, ContactState<float>& cs, const float* cmd,
                                         bool torque_mode, int t0, int n_ticks, int env, const DeviceView& D,
                                         const EnvCfg& C, const RobotConst& RC, const ModelConstT<float>& M,
                                         const ModelLegPairsT<float>& M2, const SolverConst& SC, float* tau_m /*12 out*/,
                                         float* tau_s /*12 out*/, bool detect_invalid_last, const StepScratch& scr, int* why,
                                         TraceColumn tc = TraceColumn{nullptr, 0}, bool skip = false,
                                         const ExtPush& push = ExtPush{}) {
  const float mu = D.mu[env];
  const bool custom = D.custom_gains[env] != 0;
  {  // the motor command and the springs are the same for every tick: parked in the scratch, read back by each tick
     // (volatile, so that they do not sit in 21 registers across the loop)
    float sk[3], sb[3], sr[3];
    load_springs(D, env, sk, sb, sr);
#pragma unroll
    for (int i = 0; i < 12; i++) scr.park(i) = cmd[i];
#pragma unroll
    for (int j = 0; j < 3; j++) { scr.park(12 + j) = sk[j]; scr.park(15 + j) = sb[j]; scr.park(18 + j) = sr[j]; }
  }
  // skip: this thread only keeps the block's barriers matched (its env is handed over at t0)
  int bail = skip ? t0 : n_ticks;
  *why = skip ? TICK_NEEDS_CONTACT : TICK_DONE;
  // tau_m / tau_s = the torques of the LAST tick (what the step stores): parked in local memory when that tick comes
  // (volatile: a store, not 24 registers that stay allocated over the whole loop)
  volatile float keep[24];
  bool kept = false;
  for (int t = t0; t < n_ticks; t++) {
    // keep the warps of the block in lockstep: the tick is several times larger than the
    // instruction cache, so warps that run it together share every fetched line
    if (!__syncthreads_or(bail == n_ticks)) break;  // every env of the block was handed over
    if (bail == n_ticks) {
      float tau[12], tm[12], ts[12], c12[12], sk[3], sb[3], sr[3];
#pragma unroll
      for (int i = 0; i < 12; i++) c12[i] = *static_cast<const volatile float*>(&scr.park(i));
#pragma unroll
      for (int j = 0; j < 3; j++) {
        sk[j] = *static_cast<const volatile float*>(&scr.park(12 + j));
        sb[j] = *static_cast<const volatile float*>(&scr.park(15 + j));
        sr[j] = *static_cast<const volatile float*>(&scr.park(18 + j));
      }
      tick_torques(st, c12, torque_mode, env, D, C, RC, sk, sb, sr, tau, tm, ts, custom);
      if constexpr (kTrace) tc.torques(t, tm, ts);   // (rewritten by the next kernel if this tick is handed over)
      if (t == n_ticks - 1) {
        kept = true;
#pragma unroll
        for (int i = 0; i < 12; i++) { keep[i] = tm[i]; keep[12 + i] = ts[i]; }
      }
      const int r = physics_tick<float, kContacts, QS_BLOCK, kEM, kExt>(st, tau, mu, cs, M, SC, detect_invalid_last && (t == n_ticks - 1),
                                                                   scr, EnvModelRef{D.model, D.n, env}, &M2,
                                                                   kExt ? push.at(t) : nullptr);
      if (r != TICK_DONE) { bail = t; *why = r; }
      else if constexpr (kTrace) tc.state(t, st, cs, SC.dt);
    }
  }
  if (kept) {
#pragma unroll
    for (int i = 0; i < 12; i++) { tau_m[i] = keep[i]; tau_s[i] = keep[12 + i]; }
  }
  return bail;
}

// same loop on the general solver (joint limits, every collision shape); rare path.  The traced variant takes the env's
// trace column as one more argument, the pushed variant the env's ExtPush after it (`x`, a pack so that the default
// variant keeps its calling sequence).
template <bool kEM, bool kTrace = false, bool kExt = false, typename... Extra>
__device__ __noinline__ void run_ticks_general(EnvState<float>& st, ContactState<float>& cs, const float* cmd,
                                               bool torque_mode, int t0, int n_ticks, int env, const DeviceView& D,
                                               const EnvCfg& C, const RobotConst& RC, const ModelConstT<float>& M,
                                               const SolverConst& SC, float* tau_m, float* tau_s, float* dl, int dl_stride,
                                               Extra... x) {
  static_assert(sizeof...(Extra) == int(kTrace) + int(kExt), "one TraceColumn when traced, then one ExtPush when pushed");
  const float mu = D.mu[env];
  const bool custom = D.custom_gains[env] != 0;
  float sk[3], sb[3], sr[3];
  load_springs(D, env, sk, sb, sr);
  for (int t = t0; t < n_ticks; t++) {
    float tau[12];
    tick_torques(st, cmd, torque_mode, env, D, C, RC, sk, sb, sr, tau, tau_m, tau_s, custom);
    if constexpr (kExt)
      physics_tick_general<float, kEM, true>(st, tau, mu, cs, M, SC, EnvModelRef{D.model, D.n, env}, dl, dl_stride,
                                             last_of(x...).at(t));
    else
      physics_tick_general<float, kEM>(st, tau, mu, cs, M, SC, EnvModelRef{D.model, D.n, env}, dl, dl_stride);
    if constexpr (kTrace) {
      const TraceColumn c0 = first_of(x...);
      c0.torques(t, tau_m, tau_s);
      c0.state(t, st, cs, SC.dt);
    }
  }
}

// ---------------------------------------------------------------- self collision (detection only)
// quadruped.py:530-543 loads the robot with URDF_USE_SELF_COLLISION and GetContactInfo counts a self contact as
// invalid when a calf is involved (:236-241); every task ends the episode on an invalid contact (task_base.py:146-147),
// so no contact RESPONSE is modelled for these pairs.  A pure function of the twelve joint angles (everything in the
// base frame).  Pairs per calf: trunk, imu_link, the four hips (Bullet's default filter drops parent-child pairs only:
// calf-thigh and calf-foot of the same leg), thighs, calves and feet of the other legs; in contact while the distance is
// below the smaller of the two shapes' breaking thresholds.  Same geometry as the oracle (oracle/qso_physics.c
// collide_self): calf / thigh boxes as capsules (axis inset by the radius; radii 0.008 / 0.0146), feet and imu_link
// spheres, exact hip cylinder and trunk box, segment-to-shape distance by a 21-step ternary search.  Bounding spheres
// cull the pairs first (conservative: the result is that of the full enumeration).
QS_DEVONLY float sc_seg_seg(const float* p0, const float* p1, const float* q0, const float* q1) {
  float d1[3], d2[3], r[3];
#pragma unroll
  for (int k = 0; k < 3; k++) { d1[k] = p1[k] - p0[k]; d2[k] = q1[k] - q0[k]; r[k] = p0[k] - q0[k]; }
  const float a = dot3(d1, d1), e = dot3(d2, d2), f = dot3(d2, r), c = dot3(d1, r), b = dot3(d1, d2);
  const float den = a * e - b * b;
  float sN = den > 1e-12f ? (b * f - c * e) / den : 0.f;
  sN = clampt(sN, 0.f, 1.f);
  float tN = (b * sN + f) / e;
  if (tN < 0.f) { tN = 0.f; sN = clampt(-c / a, 0.f, 1.f); }
  else if (tN > 1.f) { tN = 1.f; sN = clampt((b - c) / a, 0.f, 1.f); }
  float d[3];
#pragma unroll
  for (int k = 0; k < 3; k++) d[k] = r[k] + sN * d1[k] - tN * d2[k];
  return sqrtf(dot3(d, d));
}
QS_DEVONLY float sc_pt_seg(const float* c, const float* p0, const float* p1) {
  float d[3], r[3];
#pragma unroll
  for (int k = 0; k < 3; k++) { d[k] = p1[k] - p0[k]; r[k] = c[k] - p0[k]; }
  const float t = clampt(dot3(r, d) / dot3(d, d), 0.f, 1.f);
#pragma unroll
  for (int k = 0; k < 3; k++) r[k] -= t * d[k];
  return sqrtf(dot3(r, r));
}
QS_DEVONLY float sc_pt_box(const float* p, const float* h) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 3; k++) { const float e = fabsf(p[k]) - h[k]; if (e > 0.f) s += e * e; }
  return sqrtf(s);
}
QS_DEVONLY float sc_pt_cyl(const float* p, const float* c, const float* a, float r, float hl) {
  const float v[3] = {p[0] - c[0], p[1] - c[1], p[2] - c[2]};
  const float ax = dot3(v, a);
  const float rho2 = dot3(v, v) - ax * ax;
  const float er = sqrtf(fmaxf(rho2, 0.f)) - r, ea = fabsf(ax) - hl;
  return sqrtf((er > 0.f ? er * er : 0.f) + (ea > 0.f ? ea * ea : 0.f));
}
// Per-leg points live in `sm` (this thread's column of a [QS_SELF_SCRATCH][stride] shared-memory area, dead tick scratch in
// the step kernels): they are indexed by leg at run time, and as a local-memory array they cost more than the whole test
// (the step kernels leave ~20 KB of L1 per SM next to their shared memory: measured +0.18 ms per step).
constexpr int QS_SELF_SCRATCH = 7 * 12;
static_assert(QS_SELF_SCRATCH <= QS_TICK_SCRATCH, "the self-collision points reuse the tick scratch");
struct ScPts {
  float* p; int stride;
  QS_DEVONLY float& operator()(int arr, int leg, int a) const { return p[(arr * 12 + leg * 3 + a) * stride]; }
  QS_DEVONLY void get(int arr, int leg, float* o) const { o[0] = (*this)(arr, leg, 0); o[1] = (*this)(arr, leg, 1); o[2] = (*this)(arr, leg, 2); }
};
enum { SC_C0 = 0, SC_C1, SC_T0, SC_T1, SC_R1, SC_R4, SC_AX };
__device__ __forceinline__ int self_collision_count(const float* q12, const ModelConstT<float>& M, float* __restrict__ sm, int stride) {
  constexpr float RC = 0.008f, RT = 0.0146f;
  const ScPts P{sm, stride};
#pragma unroll 1
  for (int k = 0; k < 4; k++) {
    LegKin<float> K;
    leg_kin(k, q12 + 3 * k, M, K);
    const float fc = RC / M.link_len, ft = RT / M.link_len;
    for (int a = 0; a < 3; a++) {
      P(SC_C0, k, a) = K.r3[a] + fc * (K.r4[a] - K.r3[a]);
      P(SC_C1, k, a) = K.r3[a] + (1.f - fc) * (K.r4[a] - K.r3[a]);
      P(SC_T0, k, a) = K.r2[a] + ft * (K.r3[a] - K.r2[a]);
      P(SC_T1, k, a) = K.r2[a] + (1.f - ft) * (K.r3[a] - K.r2[a]);
      P(SC_R1, k, a) = K.r1[a]; P(SC_R4, k, a) = K.r4[a]; P(SC_AX, k, a) = K.a2[a];
    }
  }
  // Culling (conservative, so the count is that of the full enumeration): a calf capsule lies within half_c of the middle
  // of its axis.  The calf of a leg never reaches that leg's own hip: its axis stays in the plane at 0.08 m from the hip
  // centre along the hip axis, i.e. at least 0.08 - 0.02 - 0.008 = 0.052 m from the cylinder.
  const float half_c = 0.5f * M.link_len, thc = M.calf_thresh;
  const float reach = half_c + thc + 1e-4f;
  int count = 0;
#pragma unroll 1
  for (int i = 0; i < 4; i++) {
    float mid[3], ci0[3], ci1[3];
    P.get(SC_C0, i, ci0); P.get(SC_C1, i, ci1);
    for (int a = 0; a < 3; a++) mid[a] = 0.5f * (ci0[a] + ci1[a]);
    // trunk box (s = 0) and the hip cylinders of the other legs (s = 1..4)
#pragma unroll 1
    for (int s = 0; s < 5; s++) {
      const int j = s - 1;
      if (j == i) continue;
      float hj[3], aj[3];
      if (s > 0) { P.get(SC_R1, j, hj); P.get(SC_AX, j, aj); }
      // three samples of the (1-Lipschitz) distance along the axis: every point of the axis is within a quarter of its
      // length of one of them
      const float slack = 0.25f * M.link_len + RC + thc + 1e-4f;
      if (s == 0) {
        if (fminf(sc_pt_box(mid, M.trunk_half), fminf(sc_pt_box(ci0, M.trunk_half), sc_pt_box(ci1, M.trunk_half))) > slack) continue;
      } else {
        float d2 = 1e30f;
        for (int e = 0; e < 3; e++) {
          const float* p = e == 0 ? ci0 : (e == 1 ? mid : ci1);
          const float v[3] = {p[0] - hj[0], p[1] - hj[1], p[2] - hj[2]};
          d2 = fminf(d2, dot3(v, v));
        }
        const float ro = slack + 0.0502f;  // the hip cylinder lies within sqrt(0.046^2 + 0.02^2) of its centre
        if (d2 > ro * ro) continue;
      }
      const float thr = fminf(thc, s == 0 ? M.trunk_thresh : M.hip_thresh);
      float lo = 0.f, hi = 1.f, best = 1e30f;
      for (int it = 0; it <= 20; it++) {
        const float ta = lo + (hi - lo) / 3.f, tb = hi - (hi - lo) / 3.f;
        float pa[3], pb[3];
        for (int a = 0; a < 3; a++) { pa[a] = ci0[a] + ta * (ci1[a] - ci0[a]); pb[a] = ci0[a] + tb * (ci1[a] - ci0[a]); }
        const float da = s == 0 ? sc_pt_box(pa, M.trunk_half) : sc_pt_cyl(pa, hj, aj, M.hip_r, M.hip_hl);
        const float db = s == 0 ? sc_pt_box(pb, M.trunk_half) : sc_pt_cyl(pb, hj, aj, M.hip_r, M.hip_hl);
        best = fminf(best, fminf(da, db));
        if (da <= db) hi = tb; else lo = ta;
      }
      count += (best - RC) < thr;
    }
    {
      const float v[3] = {mid[0] - M.imu_pos[0], mid[1] - M.imu_pos[1], mid[2] - M.imu_pos[2]};
      if (dot3(v, v) <= (reach + 0.001f) * (reach + 0.001f))
        count += (sc_pt_seg(M.imu_pos, ci0, ci1) - RC - M.imu_half) < fminf(thc, M.imu_thresh);
    }
#pragma unroll 1
    for (int j = 0; j < 4; j++) {
      if (j == i) continue;
      float v[3], a0[3], a1[3];
      // capsule pairs: culled by the separation along the line between the two axis middles (each axis reaches
      // |half axis . n| along a unit direction n)
      const float hi_[3] = {0.5f * (ci1[0] - ci0[0]), 0.5f * (ci1[1] - ci0[1]), 0.5f * (ci1[2] - ci0[2])};
#pragma unroll 1
      for (int kind = 0; kind < 2; kind++) {   // 0: thigh of leg j, 1: calf of leg j (each pair of calves once)
        if (kind == 1 && j < i) continue;
        P.get(kind ? SC_C0 : SC_T0, j, a0); P.get(kind ? SC_C1 : SC_T1, j, a1);
        float hj_[3];
        for (int a = 0; a < 3; a++) { v[a] = mid[a] - 0.5f * (a0[a] + a1[a]); hj_[a] = 0.5f * (a1[a] - a0[a]); }
        const float rr = RC + (kind ? RC : RT), thr = kind ? thc : fminf(thc, M.thigh_thresh);
        const float dm = sqrtf(dot3(v, v));
        if (dm * dm - fabsf(dot3(hi_, v)) - fabsf(dot3(hj_, v)) > (rr + thr + 1e-4f) * dm) continue;
        count += (sc_seg_seg(ci0, ci1, a0, a1) - rr) < thr;
      }
      P.get(SC_R4, j, a0);
      for (int a = 0; a < 3; a++) v[a] = mid[a] - a0[a];
      if (dot3(v, v) <= (reach + M.foot_radius) * (reach + M.foot_radius))
        count += (sc_pt_seg(a0, ci0, ci1) - RC - M.foot_radius) < fminf(thc, M.foot_thresh);
    }
  }
  return count;
}

// ---------------------------------------------------------------- task logic
QS_DEV bool is_jump_task(int task) { return task != QS_TASK_NO_TASK; }
// 0 = TaskJumping, 1 = TaskContinuousJumping, 2 = TaskContinuousJumping2 (task_base.py:222,280)
QS_DEV int task_family(int task) {
  if (task == QS_TASK_CONTINUOUS_JUMPING_FORWARD || task == QS_TASK_CONTINUOUS_JUMPING_FORWARD2) return 1;
  if (task == QS_TASK_CONTINUOUS_JUMPING_FORWARD3 || task == QS_TASK_CONTINUOUS_JUMPING_FORWARD_PPO ||
      task == QS_TASK_CONTINUOUS_JUMPING_FORWARD_DEMO) return 2;   // TaskJumpingDemo2(TaskContinuousJumping2), task_base.py:402
  return 0;
}
// rows of DeviceView::task this task reads and writes
QS_DEV bool is_demo_task(int task) { return task >= QS_TASK_JUMPING_IN_PLACE_DEMO && task <= QS_TASK_CONTINUOUS_JUMPING_FORWARD_DEMO; }
// row of the imitation tasks' position in the demonstration (the rows left at reset follow it)
QS_DEV int demo_slot(int task) { return task == QS_TASK_CONTINUOUS_JUMPING_FORWARD_DEMO ? int(TS_DEMO2_COUNTER) : int(TS_DEMO_COUNTER); }
QS_DEV int task_slots(int task) {
  if (task == QS_TASK_CONTINUOUS_JUMPING_FORWARD_DEMO) return int(TS_END_ALL);
  return task_family(task) ? int(TS_END) : (is_demo_task(task) ? int(TS_END_DEMO) : int(TS_END_BASIC));
}

QS_DEVONLY float jumping_distance(const float* ts, const float* pos) {  // task_base.py:109-116
  float s, c;
  sincosf(ts[TS_TAKEOFF_YAW], &s, &c);
  const float dx = pos[0] - ts[TS_TAKEOFF_X], dy = pos[1] - ts[TS_TAKEOFF_Y];
  return fmaxf(c * dx - s * dy, 0.f);
}

// TaskJumping._on_step (task_base.py:61-107) + subclass overrides
QS_DEVONLY void task_on_step(float* ts, const EnvState<float>& st, const ContactState<float>& cs, const float* tau_m,
                         const float* rpy, const float* Rb, float sim_time, int task) {
  if (!is_jump_task(task)) return;
  const bool flying = (cs.mask & 15) == 0;
  if (ts[TS_SWITCHED] == 0.f && flying && st.vlin[2] / 9.81f > 0.06f) ts[TS_SWITCHED] = 1.f;  // :152-160
  const float z = st.pos[2];
  ts[TS_REL_MAX_H] = fmaxf(ts[TS_REL_MAX_H], fmaxf(z - ts[TS_INIT_HEIGHT], 0.f));
  ts[TS_MAX_H] = fmaxf(ts[TS_MAX_H], fabsf(z));
  ts[TS_MAX_DX] = fmaxf(ts[TS_MAX_DX], fabsf(st.pos[0]));
  ts[TS_MAX_PITCH] = fmaxf(ts[TS_MAX_PITCH], fabsf(rpy[1]));
  const int fam = task_family(task);
  if (fam == 0) {
    if (flying) {
      if (ts[TS_IN_AIR] == 0.f) {
        ts[TS_IN_AIR] = 1.f;
        ts[TS_T_TAKEOFF] = sim_time;
        ts[TS_TAKEOFF_X] = st.pos[0]; ts[TS_TAKEOFF_Y] = st.pos[1]; ts[TS_TAKEOFF_Z] = st.pos[2];
        ts[TS_TAKEOFF_YAW] = rpy[2];
      } else {
        ts[TS_MAX_FWD] = fmaxf(ts[TS_MAX_FWD], jumping_distance(ts, st.pos));
      }
    } else {
      if (ts[TS_IN_AIR] != 0.f) {
        ts[TS_MAX_FLIGHT] = fmaxf(ts[TS_MAX_FLIGHT], sim_time - ts[TS_T_TAKEOFF]);
        ts[TS_MAX_FWD] = fmaxf(ts[TS_MAX_FWD], jumping_distance(ts, st.pos));
        ts[TS_IN_AIR] = 0.f;
      } else {
        ts[TS_MAX_FWD] = 0.f;  // task_base.py:106-107
      }
    }
  } else {
    // TaskContinuousJumping(2)._compute_jumping_info (task_base.py:243-262, 319-338)
    const bool cj2 = fam == 2;
    ts[TS_END_JUMP] = 0.f;
    if (flying) {
      if (ts[TS_IN_AIR] == 0.f) {
        ts[TS_IN_AIR] = 1.f;
        ts[TS_T_TAKEOFF] = sim_time;
        ts[TS_TAKEOFF_X] = st.pos[0]; ts[TS_TAKEOFF_Y] = st.pos[1]; ts[TS_TAKEOFF_Z] = st.pos[2];
        ts[TS_TAKEOFF_YAW] = rpy[2];
        ts[TS_IS_JUMPING] = st.vlin[2] / 9.81f > 0.06f ? 1.f : 0.f;  // detect_jumping, :236-241
        ts[TS_MAX_JUMP_H] = 0.f;  // set to z, then zeroed by restart_jump_performance_variables (:326-330)
      } else if (cj2) {
        ts[TS_MAX_JUMP_H] = fmaxf(ts[TS_MAX_JUMP_H], st.pos[2]);
      }
    } else if (ts[TS_IN_AIR] != 0.f) {
      ts[TS_MAX_FLIGHT] = fmaxf(ts[TS_MAX_FLIGHT], sim_time - ts[TS_T_TAKEOFF]);
      const float d = jumping_distance(ts, st.pos);
      if (!cj2) {  // update_end_jump :264-266
        const float time_limit = task == QS_TASK_CONTINUOUS_JUMPING_FORWARD ? 0.15f : 0.35f;  // robot_tasks.py:105-106,139-140
        ts[TS_MAX_FWD] = fmaxf(ts[TS_MAX_FWD], d);
        ts[TS_CUM_FWD] += fminf(ts[TS_MAX_FWD], 0.5f);
        ts[TS_CUM_FLIGHT] += fminf(ts[TS_MAX_FLIGHT], time_limit);
      } else if (ts[TS_FIRST_JUMP] == 0.f) {  // update_end_jump :340-353
        const bool t3 = task == QS_TASK_CONTINUOUS_JUMPING_FORWARD3;  // robot_tasks.py:172-177 / 553-561
        const float jump_limit = 0.6f, height_limit = t3 ? 0.45f : 0.5f, bound = t3 ? 0.7f : 0.85f;
        const float fwd = fminf(d, jump_limit);
        const float perf = 0.7f * fwd / jump_limit + 0.3f * fminf(ts[TS_MAX_JUMP_H], height_limit) / height_limit;
        ts[TS_JUMP_COUNT] += 1.f;
        if (perf >= bound) ts[TS_GOOD_JUMPS] += 1.f;
        ts[TS_SUM_FWD] += fwd;
        ts[TS_SUM_FLOG] += fwd > 0.f ? fwd * log2f(fwd) : 0.f;
        ts[TS_SUM_PERF] += perf;
        ts[TS_MAX_PERF] = ts[TS_JUMP_COUNT] == 1.f ? perf : fmaxf(ts[TS_MAX_PERF], perf);
        ts[TS_LAST_PERF] = perf;
        ts[TS_END_JUMP] = 1.f;
      } else {
        ts[TS_FIRST_JUMP] = 0.f;
      }
      ts[TS_IN_AIR] = 0.f;
      ts[TS_IS_JUMPING] = 0.f;
    }
  }
  if (task == QS_TASK_BACKFLIP)  // robot_tasks.py:527-530
    ts[TS_MAX_PITCH_BF] = fmaxf(ts[TS_MAX_PITCH_BF], backflip_pitch(Rb, ts[TS_SWITCHED] != 0.f));
  if (task == QS_TASK_BACKFLIP_PPO)  // robot_tasks.py:745-747
    ts[TS_MAX_PITCH] = fmaxf(ts[TS_MAX_PITCH], backflip_pitch(Rb, ts[TS_SWITCHED] != 0.f));
  if (task == QS_TASK_JUMPING_FORWARD_PPO || task == QS_TASK_JUMPING_FORWARD_PPO_HP) {  // :420-426
    ts[TS_OLD_FWD] = ts[TS_ACTUAL_FWD];
    ts[TS_ACTUAL_FWD] = ts[TS_MAX_FWD];
  }
}

QS_DEVONLY bool task_terminated(const float* ts, const EnvState<float>& st, const ContactState<float>& cs,
                            const float* Rb, float fallen_height, int task) {
  if (!is_jump_task(task)) return false;
  const bool fallen_ground = st.pos[2] < fallen_height;  // task_base.py:123-124
  const bool fallen_orient = Rb[8] < 0.85f;              // task_base.py:126-130
  if (task == QS_TASK_BACKFLIP || task == QS_TASK_BACKFLIP_DEMO) return fallen_ground || cs.invalid > 0;  // robot_tasks.py:532-533,239-241
  return (fallen_orient && fallen_ground) || cs.invalid > 0;            // task_base.py:146-147
}

// per-step reward (robot_tasks.py:334-344, 461-471, 783-800); 0 for the sparse tasks.
// old_tau = torque of the previous control step, tau_m = of this one.
QS_DEVONLY float task_reward(const float* ts, const EnvState<float>& st, const float* foot_force, const float* old_tau,
                         const float* tau_m, const float* rpy, const float* Rb, int task) {
  float max_h_task, k_h;
  switch (task) {
    case QS_TASK_JUMPING_IN_PLACE_PPO: max_h_task = 1.0f; k_h = 0.023f; break;
    case QS_TASK_JUMPING_IN_PLACE_PPO_HP: max_h_task = 1.25f; k_h = 0.023f; break;
    case QS_TASK_JUMPING_FORWARD_PPO: max_h_task = 0.9f; k_h = 0.026f; break;
    case QS_TASK_JUMPING_FORWARD_PPO_HP: max_h_task = 1.1f; k_h = 0.026f; break;
    case QS_TASK_BACKFLIP_PPO: max_h_task = 0.7f; k_h = 0.026f; break;
    default: return 0.f;
  }
  const float z = st.pos[2];
  const float h_clip = (z < 0.29f || z > max_h_task) ? 0.f : z;
  const float F = foot_force[0] + foot_force[1] + foot_force[2] + foot_force[3];
  const float over = F > 800.f ? F : 0.f;
  float dn = 0.f;
#pragma unroll
  for (int i = 0; i < 12; i++) { const float d = old_tau[i] - tau_m[i]; dn += d * d; }
  const float rew_h = k_h * h_clip;
  const float rew_smooth = 0.015f * expf(-0.1f * sqrtf(dn));
  const float rew_contact = -3e-4f * over;
  const float rew_pitch = 0.014f * expf(-26.f * fabsf(rpy[1]));
  if (task == QS_TASK_JUMPING_IN_PLACE_PPO || task == QS_TASK_JUMPING_IN_PLACE_PPO_HP) {
    const float rew_pos = 0.013f * expf(-40.f * fabsf(st.pos[0]));
    return 0.05f * rew_pos + 0.5f * rew_contact + 0.2f * rew_smooth + 0.45f * rew_h + 0.3f * rew_pitch;
  }
  if (task == QS_TASK_JUMPING_FORWARD_PPO || task == QS_TASK_JUMPING_FORWARD_PPO_HP) {
    const float max_fwd = task == QS_TASK_JUMPING_FORWARD_PPO ? 1.3f : 1.4f;
    const float fwd = (ts[TS_ACTUAL_FWD] > max_fwd || ts[TS_ACTUAL_FWD] == ts[TS_OLD_FWD]) ? 0.f : ts[TS_ACTUAL_FWD];
    return 0.4f * rew_contact + 0.2f * rew_smooth + 0.25f * rew_h + 0.3f * rew_pitch + 0.4f * (0.038f * fwd);
  }
  const float pbf = z > 0.5f ? backflip_pitch(Rb, ts[TS_SWITCHED] != 0.f) : 0.f;
  return 0.4f * rew_contact + 0.2f * rew_smooth + 0.25f * rew_h + 0.3f * (0.014f * pbf);
}

// end-of-episode bonus / malus (robot_tasks.py:31-57, 70-99, 535-550, 349-358, 476-485, 802-809)
QS_DEVONLY float task_reward_end(const float* ts, bool term, int task, float sim_time, float max_ep_time) {
  float r = 0.f;
  switch (task) {
    case QS_TASK_JUMPING_IN_PLACE: {
      const float h = ts[TS_REL_MAX_H] > 0.9f ? 1.f : ts[TS_REL_MAX_H] / 0.9f;
      r += 0.7f * h;
      r += h * 0.3f * expf(-ts[TS_MAX_PITCH] * ts[TS_MAX_PITCH] / (0.15f * 0.15f));
      r += h * 0.05f * expf(-ts[TS_MAX_DX] * ts[TS_MAX_DX] / 0.05f);
      if (!term) r += 0.1f * h; else r -= 0.08f * (1.f + 0.8f * h);
      return r;
    }
    case QS_TASK_JUMPING_FORWARD: {
      const float h = ts[TS_REL_MAX_H] > 0.3f ? 1.f : ts[TS_REL_MAX_H] / 0.3f;
      const float d = ts[TS_MAX_FWD] > 1.3f ? 1.f : ts[TS_MAX_FWD] / 1.3f;
      const float bm = (h + d) / 2.f;
      r += 0.25f * h;
      r += 0.5f * d * h;
      r += h * 0.25f * expf(-ts[TS_MAX_PITCH] * ts[TS_MAX_PITCH] / (0.15f * 0.15f));
      if (!term) r += 0.1f * bm; else r -= 0.08f * (1.f + 1.2f * bm);
      return r;
    }
    case QS_TASK_BACKFLIP: {
      const float h = fminf(fmaxf(ts[TS_MAX_H] - 0.3f, 0.f), 0.4f) / 0.4f;
      const float p = ts[TS_MAX_PITCH_BF] / float(2 * QS_PI);
      r += p * 0.4f; r += h * 0.4f; r += h * p;
      if (ts[TS_SWITCHED] != 0.f && !term) r += 0.2f;
      return r;
    }
    case QS_TASK_JUMPING_IN_PLACE_PPO:
    case QS_TASK_JUMPING_IN_PLACE_PPO_HP: return term ? -0.25f * ts[TS_MAX_H] : 0.f;
    case QS_TASK_JUMPING_FORWARD_PPO:
    case QS_TASK_JUMPING_FORWARD_PPO_HP: return term ? 0.f : 0.05f * (ts[TS_MAX_FWD] + ts[TS_MAX_H]) / 2.f;
    case QS_TASK_BACKFLIP_PPO: return term ? 0.f : 0.2f * (0.7f * ts[TS_MAX_PITCH] / 5.f + 0.3f * ts[TS_MAX_H]) / 2.f;
    case QS_TASK_CONTINUOUS_JUMPING_FORWARD: {  // robot_tasks.py:112-131
      const float a = ts[TS_CUM_FLIGHT] / 0.15f, b = ts[TS_CUM_FWD] / 0.5f;
      r += 0.25f * a; r += 0.5f * b;
      r += a * 0.25f * expf(-ts[TS_MAX_PITCH] * ts[TS_MAX_PITCH] / (0.15f * 0.15f));
      if (!term) r += 0.1f * (a + b) / 2.f;
      return r;
    }
    case QS_TASK_CONTINUOUS_JUMPING_FORWARD2: {  // robot_tasks.py:146-166
      const float a = fminf(ts[TS_MAX_FLIGHT], 0.35f) / 0.35f, b = fminf(ts[TS_MAX_FWD], 0.5f) / 0.5f, bm = (a + b) / 2.f;
      r += 0.25f * a; r += 0.5f * b;
      r += b * 0.15f * expf(-(ts[TS_MAX_PITCH] * ts[TS_MAX_PITCH] / (0.15f * 0.15f)));
      r += 0.4f * (sim_time / max_ep_time) * bm;
      if (!term) r += 0.2f * bm;
      return r;
    }
    case QS_TASK_CONTINUOUS_JUMPING_FORWARD3:      // robot_tasks.py:183-212
    case QS_TASK_CONTINUOUS_JUMPING_FORWARD_PPO: {  // robot_tasks.py:687-698
      const float n = ts[TS_JUMP_COUNT], size = fmaxf(n, 3.f);  // arrays are zero-padded to >= 3 entries
      const float avg = ts[TS_SUM_PERF] / size;
      float entropy = 0.f;  // get_entropy_fwd, task_base.py:376-383: -sum p log2 p / log2(size), p = f / S
      if (n > 0.f && ts[TS_SUM_FWD] >= 0.05f)
        entropy = (log2f(ts[TS_SUM_FWD]) - ts[TS_SUM_FLOG] / ts[TS_SUM_FWD]) / log2f(size);
      const float rew_entropy = expf((entropy - 1.f) / 0.3f);
      if (task == QS_TASK_CONTINUOUS_JUMPING_FORWARD_PPO) return avg * rew_entropy - (term ? 1.f : 0.f);
      const float mx = n < 3.f ? fmaxf(n > 0.f ? ts[TS_MAX_PERF] : 0.f, 0.f) : ts[TS_MAX_PERF];
      float rew_avg = avg * 0.15f * expf(-ts[TS_MAX_PITCH] * ts[TS_MAX_PITCH] / (0.15f * 0.15f));
      rew_avg += avg * 0.4f * (sim_time / max_ep_time);
      rew_avg += avg * rew_entropy * 0.2f;
      rew_avg += avg * 0.25f;
      r = 0.8f * rew_avg + 0.2f * mx;
      r += 0.1f * ts[TS_GOOD_JUMPS];
      if (!term) r += 0.2f * avg;
      return r;
    }
    default: return 0.f;
  }
}

// TaskJumping._reset (task_base.py:40-59): reset_params + one _on_step
QS_DEVONLY void task_reset(float* ts, const EnvState<float>& st, const ContactState<float>& cs, const float* tau_m,
                       const float* rpy, const float* Rb, float sim_time, int task) {
  if (!is_jump_task(task)) return;
  const float keep_bf = ts[TS_MAX_PITCH_BF];  // BackFlip.max_pitch lives in __init__ only (robot_tasks.py:524)
#pragma unroll
  for (int i = 0; i < TS_END; i++) ts[i] = 0.f;
  ts[TS_MAX_PITCH_BF] = keep_bf;
  ts[TS_FIRST_JUMP] = 1.f;
  ts[TS_T_TAKEOFF] = sim_time;
  ts[TS_TAKEOFF_X] = st.pos[0]; ts[TS_TAKEOFF_Y] = st.pos[1]; ts[TS_TAKEOFF_Z] = st.pos[2];
  ts[TS_INIT_HEIGHT] = st.pos[2];
  ts[TS_TAKEOFF_YAW] = rpy[2];
#pragma unroll
  for (int i = 0; i < 12; i++) ts[TS_OLD_TAU0 + i] = tau_m[i];
  task_on_step(ts, st, cs, tau_m, rpy, Rb, sim_time, task);
}

// ---------------------------------------------------------------- sensors
// SensorList.get_obs / get_noisy_obs (sensor.py:101-111) for the modes of
// sensor_collection.py:18-105; obs is written row-major [N, O].
QS_DEVONLY void observe(const EnvState<float>& st, const ContactState<float>& cs, const float* ts, const float* rpy,
                    const float* Rb, int obs_mode, int task, float* o /*QS_MAX_OBS regs*/) {
  const float* q = st.q;
  const float* qd = st.qd;
  float wl[3];
  m3t_v(Rb, st.vang, wl);  // quadruped.py:141-170
  const float landing = ts[TS_SWITCHED];
  const float jumping = task_family(task) ? ts[TS_IS_JUMPING] : 0.f;  // the attribute exists on those tasks only
  int n = 0;
#define PUT(x) o[n++] = (x)
#define PUT12(p) _Pragma("unroll") for (int _i = 0; _i < 12; _i++) o[n++] = (p)[_i]
  switch (obs_mode) {
    case QS_OBS_ENCODER: PUT12(q); PUT12(qd); break;
    case QS_OBS_ENCODER_2:
      PUT(st.vlin[0]); PUT(st.vlin[1]); PUT(st.vlin[2]); PUT(st.vang[0]); PUT(st.vang[1]); PUT(st.vang[2]);
      PUT12(q); PUT12(qd); break;
    case QS_OBS_CARTESIAN_NO_IMU: {
      float fp[12], fv[12];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        float J[9];
        fk_jacobian(q + 3 * k, k, fp + 3 * k, J);
#pragma unroll
        for (int a = 0; a < 3; a++)
          fv[3 * k + a] = J[3 * a] * qd[3 * k] + J[3 * a + 1] * qd[3 * k + 1] + J[3 * a + 2] * qd[3 * k + 2];
      }
      PUT12(fp); PUT12(fv);
      break;
    }
    case QS_OBS_ARS_BASIC: PUT12(q); PUT12(qd); PUT(rpy[1]); PUT(st.pos[2]); PUT(st.vlin[2]); break;
    case QS_OBS_ARS_SENSOR: PUT12(q); PUT12(qd); PUT(rpy[1]); PUT(wl[1]); PUT(st.pos[2]); PUT(st.vlin[2]); break;
    case QS_OBS_LANDING_SENSOR:
      PUT12(q); PUT12(qd); PUT(rpy[1]); PUT(wl[1]); PUT(st.pos[2]); PUT(st.vlin[2]); PUT(landing); break;
    case QS_OBS_PPO_BASIC: PUT12(q); PUT12(qd); PUT(rpy[1]); PUT(st.pos[2]); PUT(st.vlin[2]); PUT(landing); break;
    case QS_OBS_PPO_BASIC_X:
      PUT12(q); PUT12(qd); PUT(rpy[1]); PUT(st.pos[2]); PUT(st.vlin[2]); PUT(st.vlin[0]); PUT(landing); break;
    case QS_OBS_PPO_BASIC_CONTACT:
      PUT12(q); PUT12(qd); PUT(rpy[1]); PUT(st.pos[2]); PUT(st.vlin[2]); PUT(landing);
#pragma unroll
      for (int k = 0; k < 4; k++) PUT((cs.mask >> k) & 1 ? 1.f : 0.f);
      break;
    case QS_OBS_ARS_BACKFLIP:
      PUT12(q); PUT12(qd); PUT(st.pos[2]); PUT(st.vlin[2]); PUT(backflip_pitch(Rb, landing != 0.f)); break;
    case QS_OBS_PPO_BACKFLIP:
      PUT12(q); PUT12(qd); PUT(st.pos[2]); PUT(st.vlin[2]); PUT(backflip_pitch(Rb, landing != 0.f)); PUT(landing); break;
    default:  // QS_OBS_PPO_CONTINUOUS_JUMPING_FORWARD: is_jumping only exists on the continuous tasks
      PUT12(q); PUT12(qd); PUT(st.pos[2]); PUT(st.vlin[2]); PUT(rpy[1]); PUT(landing); PUT(jumping); break;
  }
#undef PUT
#undef PUT12
}

// add N(0, sigma) per element (sensor.py:25-32,46-52) and store the row
QS_DEVONLY void store_obs(float* obs_row, float* o, const EnvCfg& C, const RobotConst& RC, uint64_t gid, uint32_t epoch,
                      uint32_t step, bool with_noise) {
  if (with_noise) {
#pragma unroll
    for (int b = 0; b < QS_MAX_OBS / 4; b++) {
      if (4 * b < C.obs_dim) {
        float nz[4];
        normal4(C.seed, gid, epoch, step, b, nz);
#pragma unroll
        for (int j = 0; j < 4; j++) o[4 * b + j] += RC.obs_noise[4 * b + j] * nz[j];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < QS_MAX_OBS; i++)
    if (i < C.obs_dim) obs_row[i] = o[i];
}

// ---------------------------------------------------------------- SoA load/store
QS_DEVONLY void load_state(const DeviceView& D, int env, EnvState<float>& st, ContactState<float>& cs, float dt) {
  const int n = D.n;
  const float* s = D.state + env;
#pragma unroll
  for (int i = 0; i < 3; i++) st.pos[i] = s[i * n];
#pragma unroll
  for (int i = 0; i < 4; i++) st.quat[i] = s[(3 + i) * n];
#pragma unroll
  for (int i = 0; i < 3; i++) st.vlin[i] = s[(7 + i) * n];
#pragma unroll
  for (int i = 0; i < 3; i++) st.vang[i] = s[(10 + i) * n];
#pragma unroll
  for (int i = 0; i < 12; i++) st.q[i] = s[(13 + i) * n];
#pragma unroll
  for (int i = 0; i < 12; i++) st.qd[i] = s[(25 + i) * n];
  const int c = D.contact[env];
  cs.mask = c & 15;
  cs.invalid = c >> 8;
  cs.work_contacts = 0;
  cs.work_row_iters = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) cs.lam_n[k] = D.foot_force[k * n + env] * dt;
}
QS_DEVONLY void store_state(const DeviceView& D, int env, const EnvState<float>& st, const ContactState<float>& cs, float dt) {
  const int n = D.n;
  float* s = D.state + env;
#pragma unroll
  for (int i = 0; i < 3; i++) s[i * n] = st.pos[i];
#pragma unroll
  for (int i = 0; i < 4; i++) s[(3 + i) * n] = st.quat[i];
#pragma unroll
  for (int i = 0; i < 3; i++) s[(7 + i) * n] = st.vlin[i];
#pragma unroll
  for (int i = 0; i < 3; i++) s[(10 + i) * n] = st.vang[i];
#pragma unroll
  for (int i = 0; i < 12; i++) s[(13 + i) * n] = st.q[i];
#pragma unroll
  for (int i = 0; i < 12; i++) s[(25 + i) * n] = st.qd[i];
  D.contact[env] = (cs.mask & 15) | (cs.invalid << 8);
#pragma unroll
  for (int k = 0; k < 4; k++) D.foot_force[k * n + env] = cs.lam_n[k] / dt;
}

}  // namespace qs
