// qs_step_kernels.cuh -- the step / reset kernel family (K1, K2).
//
//   k_step       one thread per env: action map, action_repeat fast ticks, epilogue.
//                An env whose tick needs the general solver (joint at its limit, body
//                shape on the ground) is parked untouched on the slow list.
//   k_step_slow  resumes parked envs with the general tick and runs the same epilogue
//                (a handful of envs per step: launched for N, exits on `count`).
//   k_reset      in-place reset + 2500-tick settle (exact QuadrupedGymEnv.reset), for a
//                mask / list / all envs.
//   k_settle_slice / k_conveyor_ctl   the settle conveyor: episodes settled ahead of time.
//   k_settle_urgent                   an episode nobody settled in time (rare).
//
// Auto-reset without stalls: the state an env starts its next episode from is a pure
// function of (seed, global env id, episode number): mu ~ U[0.5,1) from Philox, then the
// reference's 2500 settle ticks.  Each env owns a ring of QS_SLOTS slots holding its next
// episodes' settled states; a finished env copies its slot inside k_step and queues the
// slot's next tenant on the conveyor.  Every control step the conveyor advances all its
// entries by a slice of ticks (k_settle_slice, on a second stream, next to the latency-bound
// blocks of k_step_contact and k_step_slow), saving the unfinished ones bit-exactly in between,
// so the settles run as dense waves and their cost hides behind the step's serial chain.
// If a slot is not ready in time the episode is settled start to end at the end of the step
// (k_settle_urgent) -- same numbers either way, so results never depend on scheduling,
// slicing or sharding.
#pragma once

// settling / reset-time command: _convert_reference_to_command(get_init_pose())
// (interface_base.py:68-72,182-200); also returns the settling action.
__device__ __forceinline__ void settle_command(const EnvCfg& C, const RobotConst& RC, float* cmd, float* act12) {
  if (C.is_rl) {
    const bool cart = C.control_mode == QS_CTRL_CARTESIAN_PD;
    const int sidx = cart ? 1 : 0;
    float a12[12];
#pragma unroll
    for (int i = 0; i < 12; i++)
      a12[i] = cart ? command_to_action1(RC.nominal_foot[i], RC.cart_lo[i], RC.cart_hi[i])
                    : command_to_action1(RC.init_angles[i], RC.ang_lo[i], RC.ang_hi[i]);
    // _convert_to_actual_action_space (action_interface.py:17-18,41-44,67-74)
#pragma unroll
    for (int i = 0; i < 12; i++) act12[i] = 0.f;
    if (C.action_mode == QS_ACT_DEFAULT) {
#pragma unroll
      for (int i = 0; i < 12; i++) act12[i] = a12[i];
    } else if (C.action_mode == QS_ACT_SYMMETRIC) {
#pragma unroll
      for (int j = 0; j < 3; j++) { act12[j] = a12[j]; act12[3 + j] = a12[6 + j]; }
    } else {
      if (sidx == 0) { act12[0] = a12[1]; act12[1] = a12[2]; act12[2] = a12[7]; act12[3] = a12[8]; }
      else { act12[0] = a12[0]; act12[1] = a12[2]; act12[2] = a12[6]; act12[3] = a12[8]; }
    }
    float b12[12];
    expand_action(C.action_mode, sidx, act12, b12);
    action12_to_command(RC, C.control_mode, b12, cmd);
    // settling_action = _transform_motor_command_to_action(settling_command)
    // (interface_base.py:196-200).  In CARTESIAN_PD mode the command holds JOINT
    // ANGLES (it went through IK) yet is scaled with the CARTESIAN limits, so the
    // reference stores (0, 1, -1) per leg as _last_action: reproduced as is.
#pragma unroll
    for (int i = 0; i < 12; i++)
      a12[i] = cart ? command_to_action1(cmd[i], RC.cart_lo[i], RC.cart_hi[i])
                    : command_to_action1(cmd[i], RC.ang_lo[i], RC.ang_hi[i]);
#pragma unroll
    for (int i = 0; i < 12; i++) act12[i] = 0.f;
    if (C.action_mode == QS_ACT_DEFAULT) {
#pragma unroll
      for (int i = 0; i < 12; i++) act12[i] = a12[i];
    } else if (C.action_mode == QS_ACT_SYMMETRIC) {
#pragma unroll
      for (int j = 0; j < 3; j++) { act12[j] = a12[j]; act12[3 + j] = a12[6 + j]; }
    } else {
      if (sidx == 0) { act12[0] = a12[1]; act12[1] = a12[2]; act12[2] = a12[7]; act12[3] = a12[8]; }
      else { act12[0] = a12[0]; act12[1] = a12[2]; act12[2] = a12[6]; act12[3] = a12[8]; }
    }
  } else {
    // settle_robot_by_pd (control_interface/utils.py:22-30): PD limits, DEFAULT space
#pragma unroll
    for (int i = 0; i < 12; i++) {
      const float a = command_to_action1(RC.init_angles[i], RC.ang_lo[i], RC.ang_hi[i]);
      cmd[i] = clampt(RC.ang_lo[i] + 0.5f * (a + 1.f) * (RC.ang_hi[i] - RC.ang_lo[i]), RC.ang_lo[i], RC.ang_hi[i]);
      act12[i] = 0.f;
    }
  }
}

// settle_command() once, on the device (its inverse kinematics must be the device's own arithmetic), for
// RobotConst::settle_cmd: run by qs_create with one thread
__global__ void k_settle_cmd(const __grid_constant__ KernelArgs A, float* __restrict__ out) {
  float cmd[12], act12[12];
  settle_command(A.C, A.RC, cmd, act12);
  for (int i = 0; i < 12; i++) out[i] = cmd[i];
}

__device__ __forceinline__ void finish_episode_stats(const DeviceView& D, int env, const float* ts, float ep_return,
                                                     int ep_len, bool terminated, int task, bool nonfinite = false) {
  const int n = D.n;
  float* s = D.stats + env;
  if (nonfinite) {  // an episode cut short by the NaN / Inf guard: counted, its (meaningless) maxima are not
    s[0 * n] += 1.f;
    s[9 * n] += float(ep_len);
    s[11 * n] += 1.f;
    return;
  }
  s[0 * n] += 1.f;
  s[1 * n] += ts[TS_MAX_H];
  s[2 * n] = fmaxf(s[2 * n], ts[TS_MAX_H]);
  s[3 * n] += ts[TS_REL_MAX_H];
  s[4 * n] += ts[TS_MAX_FWD];
  s[5 * n] = fmaxf(s[5 * n], ts[TS_MAX_FWD]);
  s[6 * n] += ts[TS_MAX_FLIGHT];
  const float flip = (task == QS_TASK_BACKFLIP ? ts[TS_MAX_PITCH_BF] : ts[TS_MAX_PITCH]) / float(2 * QS_PI);
  s[7 * n] += flip;
  s[8 * n] += ep_return;
  s[9 * n] += float(ep_len);
  s[10 * n] += terminated ? 1.f : 0.f;
}

enum { LAND_POLICY = 0, LAND_HOLD = 1, LAND_LANDING = 2, LAND_SPENT = 3, LAND_TAKEOFF_BF = 4 };
constexpr int QS_SLOTS = 4;  // settled episodes kept ahead per env (ring indexed by episode number)

// ---- settle conveyor: the queue of (env, episode) pairs whose settled start state is computed
// ahead of time, a slice of ticks per control step, on a second stream next to k_step_slow.
//   fifo[2 * (i & cap_mask)] = {env, episode} of entry i; entries are pushed at `head` and retire at `tail`
//   tick[i & cap_mask]       = settle ticks already done for entry i (CV_DONE: finished or dropped)
//   wip[row][i % width]      = state of entry i between slices (raw floats: slicing is bit-invisible)
// The first `active` entries after `tail` run `slice` ticks in k_settle_slice; k_conveyor_ctl picks both.
enum {
  CV_HEAD = 0, CV_TAIL, CV_ACTIVE, CV_SLICE, CV_URGENT, CV_URGENT_LAST, CV_PREV_HEAD, CV_DEMAND,
  // ring pressure: slots consumed this step, and how many of those envs found their next slot missing
  CV_TAKEN, CV_LOW2, CV_EMA_TAKEN, CV_EMA_LOW2, CV_PRESS,
  // the early slice (next to k_step_contact): entries, ticks; ticks per entry wanted from this step in total
  CV_ACTIVE_EARLY, CV_SLICE_EARLY, CV_WANT, CV_CTL_WORDS = 16
};
constexpr int CV_DONE = -1;
constexpr int WIP_ROWS = 37 + 4;  // state | normal impulses (warm start); + contact mask (int row)
struct Conveyor {
  int* fifo;
  int* tick;
  float* wip;
  int* wip_contact;
  float* model;      // [EM_ROWS][width] mass properties of the episodes in flight (mass randomizer)
  uint32_t* ctl;
  int* urgent_list;  // (env, episode) pairs that must be settled and started NOW; count in ctl[CV_URGENT]
  unsigned long long* work;  // settle ticks, foot-contact ticks, contact x PGS-sweep count done by the slices
  uint32_t cap_mask;
  int width;
};

struct StepIO {
  const float* actions;
  float* obs;
  float* reward;
  uint8_t* done;
  uint8_t* truncated;
  float* term_obs;   // optional [N][O]: last observation of the episodes that finished in this step (qs_set_terminal_obs)
  int* slow_list;    // envs parked for the general solver, slow_list[n] = count
  int* contact_list; // envs with a foot on the ground (k_pre) or reaching it (flight kernel), contact_list[n] = count
  int* flight_list;  // the others: k_step's work, flight_list[n] = count
  Conveyor cv;
  unsigned long long* stamps;  // this step's {late slice start, end, general solver start, end} in globaltimer ns
  int flight_cap;    // envs the flight kernel takes at most (one wave of its blocks); the rest ride with the contact kernel
};

// device-side duration of a kernel that runs concurrently with another one in the same stream (programmatic dependent
// launch: no event can be recorded between the two without serialising them)
__device__ __forceinline__ unsigned long long qs_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void stamp_begin(unsigned long long* st) { if (st) atomicMin(st, qs_globaltimer()); }
__device__ __forceinline__ void stamp_end(unsigned long long* st) { if (st) atomicMax(st + 1, qs_globaltimer()); }

__device__ __forceinline__ uint32_t ld_acquire(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ void conveyor_push(const Conveyor& cv, int env, uint32_t epoch) {
  const uint32_t i = atomicAdd(cv.ctl + CV_HEAD, 1u);
  const uint32_t tail = *reinterpret_cast<volatile uint32_t*>(cv.ctl + CV_TAIL);
  // a full queue only loses a prefetch: the position keeps its retired entry and the env takes the urgent path
  if (i - tail > cv.cap_mask) return;
  const uint32_t pos = i & cv.cap_mask;
  cv.fifo[2 * pos] = env;
  cv.fifo[2 * pos + 1] = int(epoch);
  cv.tick[pos] = 0;
}
__device__ __forceinline__ void urgent_push(const Conveyor& cv, int env, uint32_t epoch) {
  const uint32_t i = atomicAdd(cv.ctl + CV_URGENT, 1u);
  cv.urgent_list[2 * i] = env;  // at most one per env and step
  cv.urgent_list[2 * i + 1] = int(epoch);
}

// ---- spare slot of an env: the settled state its next episode starts from
// rows: state 37 | tau_motor 12 | tau_spring 12 | foot_force 4 | mu 1   (floats), contact, epoch (ints)
constexpr int SLOT_ROWS = 37 + 12 + 12 + 4 + 1;

__device__ __forceinline__ bool slot_ready(const DeviceView& D, int env, uint32_t epoch) {
  return ld_acquire(D.slot_epoch + int(epoch % QS_SLOTS) * D.n + env) == epoch;
}

__device__ __forceinline__ void slot_store(const DeviceView& D, int env, const EnvState<float>& st,
                                           const ContactState<float>& cs, const float* tau_m, const float* tau_s,
                                           float mu, uint32_t epoch, float dt) {
  const int n = D.n;
  const int sl = int(epoch % QS_SLOTS);
  float* s = D.slot + size_t(sl) * SLOT_ROWS * n + env;
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
#pragma unroll
  for (int i = 0; i < 12; i++) { s[(37 + i) * n] = tau_m[i]; s[(49 + i) * n] = tau_s[i]; }
#pragma unroll
  for (int k = 0; k < 4; k++) s[(61 + k) * n] = cs.lam_n[k] / dt;
  s[65 * n] = mu;
  D.slot_contact[sl * n + env] = (cs.mask & 15) | (cs.invalid << 8);
  st_release(D.slot_epoch + sl * n + env, epoch);  // readers on the other stream see the rows before the tag
}

// state of a settle between two slices (bit-exact round trip)
__device__ __forceinline__ void wip_store(const Conveyor& cv, int col, const EnvState<float>& st, const ContactState<float>& cs) {
  const int w = cv.width;
  float* s = cv.wip + col;
#pragma unroll
  for (int i = 0; i < 3; i++) s[i * w] = st.pos[i];
#pragma unroll
  for (int i = 0; i < 4; i++) s[(3 + i) * w] = st.quat[i];
#pragma unroll
  for (int i = 0; i < 3; i++) s[(7 + i) * w] = st.vlin[i];
#pragma unroll
  for (int i = 0; i < 3; i++) s[(10 + i) * w] = st.vang[i];
#pragma unroll
  for (int i = 0; i < 12; i++) s[(13 + i) * w] = st.q[i];
#pragma unroll
  for (int i = 0; i < 12; i++) s[(25 + i) * w] = st.qd[i];
#pragma unroll
  for (int k = 0; k < 4; k++) s[(37 + k) * w] = cs.lam_n[k];
  cv.wip_contact[col] = (cs.mask & 15) | (cs.invalid << 8);
}
__device__ __forceinline__ void wip_load(const Conveyor& cv, int col, EnvState<float>& st, ContactState<float>& cs) {
  const int w = cv.width;
  const float* s = cv.wip + col;
#pragma unroll
  for (int i = 0; i < 3; i++) st.pos[i] = s[i * w];
#pragma unroll
  for (int i = 0; i < 4; i++) st.quat[i] = s[(3 + i) * w];
#pragma unroll
  for (int i = 0; i < 3; i++) st.vlin[i] = s[(7 + i) * w];
#pragma unroll
  for (int i = 0; i < 3; i++) st.vang[i] = s[(10 + i) * w];
#pragma unroll
  for (int i = 0; i < 12; i++) st.q[i] = s[(13 + i) * w];
#pragma unroll
  for (int i = 0; i < 12; i++) st.qd[i] = s[(25 + i) * w];
#pragma unroll
  for (int k = 0; k < 4; k++) cs.lam_n[k] = s[(37 + k) * w];
  const int c = cv.wip_contact[col];
  cs.mask = c & 15;
  cs.invalid = c >> 8;
  cs.work_contacts = 0;
  cs.work_row_iters = 0;
}

__device__ __forceinline__ void slot_load(const DeviceView& D, int env, uint32_t epoch, EnvState<float>& st,
                                          ContactState<float>& cs, float* tau_m, float* tau_s, float* mu, float dt) {
  const int n = D.n;
  const int sl = int(epoch % QS_SLOTS);
  const float* s = D.slot + size_t(sl) * SLOT_ROWS * n + env;
#pragma unroll
  for (int i = 0; i < 3; i++) st.pos[i] = __ldcg(s + i * n);
#pragma unroll
  for (int i = 0; i < 4; i++) st.quat[i] = __ldcg(s + (3 + i) * n);
#pragma unroll
  for (int i = 0; i < 3; i++) st.vlin[i] = __ldcg(s + (7 + i) * n);
#pragma unroll
  for (int i = 0; i < 3; i++) st.vang[i] = __ldcg(s + (10 + i) * n);
#pragma unroll
  for (int i = 0; i < 12; i++) st.q[i] = __ldcg(s + (13 + i) * n);
#pragma unroll
  for (int i = 0; i < 12; i++) st.qd[i] = __ldcg(s + (25 + i) * n);
#pragma unroll
  for (int i = 0; i < 12; i++) { tau_m[i] = __ldcg(s + (37 + i) * n); tau_s[i] = __ldcg(s + (49 + i) * n); }
#pragma unroll
  for (int k = 0; k < 4; k++) cs.lam_n[k] = __ldcg(s + (61 + k) * n) * dt;
  *mu = __ldcg(s + 65 * n);
  const int c = __ldcg(D.slot_contact + sl * n + env);
  cs.mask = c & 15;
  cs.invalid = c >> 8;
  cs.work_contacts = 0;
  cs.work_row_iters = 0;
}

// The robot as reset() spawns it (quadruped_gym_env.py:278-289, configs:23)
__device__ __forceinline__ void fresh_state(const KernelArgs& A, EnvState<float>& st, ContactState<float>& cs) {
  st.pos[0] = 0.f; st.pos[1] = 0.f; st.pos[2] = 0.32f;  // INIT_POSITION
  st.quat[0] = st.quat[1] = st.quat[2] = 0.f; st.quat[3] = 1.f;
#pragma unroll
  for (int i = 0; i < 3; i++) { st.vlin[i] = 0.f; st.vang[i] = 0.f; }
#pragma unroll
  for (int i = 0; i < 12; i++) { st.q[i] = A.RC.init_angles[i]; st.qd[i] = 0.f; }
  cs.mask = 0; cs.invalid = 0; cs.work_contacts = 0; cs.work_row_iters = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) cs.lam_n[k] = 0.f;
}
__device__ __forceinline__ float episode_mu(const EnvCfg& C, uint64_t gid, uint32_t epoch) {  // env_randomizer.py:287-289
  return C.ground_randomizer ? 0.5f + 0.5f * uniform1(C.seed, gid, epoch, 100) : C.mu_ground;
}
__device__ __forceinline__ int settle_length(const EnvCfg& C) { return C.is_rl ? C.settling_steps : 1500; }
// spring stiffness / damping / rest angle (hip, thigh, calf) of an episode: nominal, or EnvRandomizerSprings'
// U[(1 - 0.1) x, (1 + 0.1) x] draw (env_randomizer.py:101-122), taken before the settle like randomize_env()
__device__ __forceinline__ void episode_springs(const EnvCfg& C, const RobotConst& RC, uint64_t gid, uint32_t epoch,
                                                float* sk, float* sb, float* sr) {
#pragma unroll
  for (int j = 0; j < 3; j++) {
    sk[j] = RC.spring_k[j]; sb[j] = RC.spring_b[j]; sr[j] = RC.spring_rest[j];
    if (C.spring_randomizer) {
      sk[j] *= 1.f - C.spring_err + 2.f * C.spring_err * uniform1(C.seed, gid, epoch, 101 + j);
      sb[j] *= 1.f - C.spring_err + 2.f * C.spring_err * uniform1(C.seed, gid, epoch, 104 + j);
    }
  }
}

// EnvRandomizerMasses.randomize_env (env_randomizer.py:56-84) for episode `epoch` of global env `gid`:
// raw = hip, thigh, calf link mass | trunk mass | block mass | block position (base frame)
__device__ __forceinline__ void episode_masses(const EnvCfg& C, uint64_t gid, uint32_t epoch, float* raw) {
  const float nominal[3] = {0.591f, 0.92f, 0.131f};  // go1.urdf hip / thigh / calf
  float legs = 0.f;
#pragma unroll
  for (int j = 0; j < 3; j++) {  // _randomize_leg_masses :62-71: each leg in the same way
    raw[j] = nominal[j] * (1.f - C.leg_mass_err + 2.f * C.leg_mass_err * uniform1(C.seed, gid, epoch, 110 + j));
    legs += raw[j];
  }
  raw[4] = C.payload_max * uniform1(C.seed, gid, epoch, 113);  // _add_mass_offset :73-84
#pragma unroll
  for (int j = 0; j < 3; j++) raw[5 + j] = C.payload_pos[j] * (2.f * uniform1(C.seed, gid, epoch, 114 + j) - 1.f);
  // _change_base_mass :56-60: total (all 19 URDF links, 12.01301 kg) - block - leg links - feet
  raw[3] = 12.01301f - raw[4] - 4.f * legs - 4.f * 0.06f;
}
// The mass properties the tick reads (EnvModelRef rows) for those draws.  changeDynamics(mass=) leaves every link's
// inertia diagonal and inertial frame as loaded (collision-geometry inertias of the NOMINAL masses, SURVEY.md App. B.2),
// so only masses, first moments and parallel-axis terms move.  Same constants as qs_model_host.h build_model.
__device__ __noinline__ void model_from_masses(const float* raw, float* em) {
  em[EM_HIP_M] = raw[0];
  em[EM_THIGH_M] = raw[1];
  {  // calf + foot (fixed joint), in the calf frame
    const double mc = raw[2], mf = 0.06, m = mc + mf;
    const double cc[3] = {0.006286, 0.001307, -0.122269}, cf[3] = {0.0, 0.0, -0.213};
    const double Ic[3] = {0.131 / 12.0 * (0.016 * 0.016 + 0.213 * 0.213), 0.131 / 12.0 * (0.016 * 0.016 + 0.213 * 0.213),
                          0.131 / 12.0 * (0.016 * 0.016 + 0.016 * 0.016)};
    const double If = 0.4 * 0.06 * 0.02 * 0.02;
    double c[3], I[6] = {Ic[0] + If, 0, 0, Ic[1] + If, 0, Ic[2] + If};
    for (int i = 0; i < 3; i++) c[i] = (mc * cc[i] + mf * cf[i]) / m;
    for (int b = 0; b < 2; b++) {
      const double mm = b ? mf : mc;
      const double d[3] = {(b ? cf[0] : cc[0]) - c[0], (b ? cf[1] : cc[1]) - c[1], (b ? cf[2] : cc[2]) - c[2]};
      const double dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
      I[0] += mm * (dd - d[0] * d[0]); I[1] -= mm * d[0] * d[1]; I[2] -= mm * d[0] * d[2];
      I[3] += mm * (dd - d[1] * d[1]); I[4] -= mm * d[1] * d[2]; I[5] += mm * (dd - d[2] * d[2]);
    }
    em[EM_CALF_M] = float(m);
    for (int i = 0; i < 3; i++) em[EM_CALF_COM + i] = float(c[i]);
    for (int i = 0; i < 6; i++) em[EM_CALF_IC + i] = float(I[i]);
  }
  {  // body 0 about the base origin: base (1e-5 kg, no inertia) + trunk + imu_link + block (0.1 m cube)
    const double mt = raw[3], mp = raw[4];
    const double ct[3] = {0.0223, 0.0, -0.0005}, ci[3] = {-0.01592, -0.06659, -0.00617}, cp[3] = {raw[5], raw[6], raw[7]};
    const double It[3] = {5.204 / 12.0 * (0.0935 * 0.0935 + 0.114 * 0.114), 5.204 / 12.0 * (0.3762 * 0.3762 + 0.114 * 0.114),
                          5.204 / 12.0 * (0.3762 * 0.3762 + 0.0935 * 0.0935)};
    const double Ii = 0.001 / 12.0 * (2e-6), Ip = mp * 0.01 / 6.0;
    double I[6] = {It[0] + Ii + Ip, 0, 0, It[1] + Ii + Ip, 0, It[2] + Ii + Ip}, hh[3] = {0, 0, 0};
    const double ms[3] = {mt, 0.001, mp};
    for (int b = 0; b < 3; b++) {
      const double* c = b == 0 ? ct : (b == 1 ? ci : cp);
      const double mm = ms[b], dd = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
      for (int i = 0; i < 3; i++) hh[i] += mm * c[i];
      I[0] += mm * (dd - c[0] * c[0]); I[1] -= mm * c[0] * c[1]; I[2] -= mm * c[0] * c[2];
      I[3] += mm * (dd - c[1] * c[1]); I[4] -= mm * c[1] * c[2]; I[5] += mm * (dd - c[2] * c[2]);
    }
    em[EM_TRUNK_M] = float(0.00001 + mt + 0.001 + mp);
    for (int i = 0; i < 3; i++) em[EM_TRUNK_H + i] = float(hh[i]);
    for (int i = 0; i < 6; i++) em[EM_TRUNK_I + i] = float(I[i]);
  }
}
// draws of (gid, epoch) -> the rows of column idx
__device__ __forceinline__ void episode_model_store(const EnvCfg& C, uint64_t gid, uint32_t epoch, float* base, int stride, int idx,
                                                    float* draw_base /* [8][stride] or nullptr */) {
  float raw[8], em[EM_ROWS];
  episode_masses(C, gid, epoch, raw);
  model_from_masses(raw, em);
  for (int i = 0; i < EM_ROWS; i++) base[size_t(i) * stride + idx] = em[i];
  if (draw_base)
    for (int i = 0; i < 8; i++) draw_base[size_t(i) * stride + idx] = raw[i];
}

// Settle ticks [t0, t1) of the reset (control_interface/interface_base.py:182-200), at most `span` of them.
// Every thread of the block runs the same `span` iterations (one barrier each, see run_ticks);
// a thread works while t < t1.
template <bool kEM>
__device__ __forceinline__ void settle_ticks(const KernelArgs& A, uint64_t gid, uint32_t epoch, EnvState<float>& st,
                                             ContactState<float>& cs, float mu, int t0, int t1, int span, float* tau_m,
                                             float* tau_s, const StepScratch& scr, float* em_base, int em_stride, int em_idx) {
  const EnvCfg& C = A.C;
  // randomize_env() comes before the settle (quadruped_gym_env.py:286-289): the episode's masses, in the column
  // (em_base, em_stride, em_idx) -- the env's own rows, or the conveyor's for an episode settled ahead
  if (kEM && t1 > t0) episode_model_store(C, gid, epoch, em_base, em_stride, em_idx, nullptr);
  const EnvModelRef em{em_base, em_stride, em_idx};
  const float* cmd = A.RC.settle_cmd;   // = settle_command(), from the constant bank
  // a fresh Quadruped has the default gains / springs (quadruped_gym_env.py:299-319); the settle
  // runs on the fast tick only: the standing pose is far from every joint limit and body contact
  SolverConst SCs = A.SC;
  SCs.enable_limits = 0;
  SCs.body_response = 0;
  const int nsettle = settle_length(C);
  {  // the episode's springs: parked in the scratch, read back by each tick (not 9 registers across the loop)
    float sk[3], sb[3], sr[3];
    episode_springs(C, A.RC, gid, epoch, sk, sb, sr);
#pragma unroll
    for (int j = 0; j < 3; j++) { scr.park(12 + j) = sk[j]; scr.park(15 + j) = sb[j]; scr.park(18 + j) = sr[j]; }
  }
  // The callers want the motor / spring torques of the LAST settle tick only.  They are parked in local memory when that
  // tick comes (volatile: a store, not 24 registers that stay allocated over the whole loop).
  volatile float keep[24];
  bool kept = false;
  for (int i = 0; i < span; i++) {
    __syncthreads();  // lockstep across the block (see run_ticks)
    const int t = t0 + i;
    if (t >= t1) continue;
    float tau[12], tm[12], ts[12], sk[3], sb[3], sr[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
      sk[j] = *static_cast<const volatile float*>(&scr.park(12 + j));
      sb[j] = *static_cast<const volatile float*>(&scr.park(15 + j));
      sr[j] = *static_cast<const volatile float*>(&scr.park(18 + j));
    }
#pragma unroll
    for (int i2 = 0; i2 < 12; i2++) {
      tm[i2] = pd_torque1(A.RC.kp[i2], A.RC.kd[i2], A.RC.tau_max[i2], cmd[i2], st.q[i2], st.qd[i2], false);
      tau[i2] = tm[i2];
      ts[i2] = 0.f;
    }
    if (C.enable_springs) {
#pragma unroll
      for (int k = 0; k < 4; k++) {
        spring_torque_leg(k, sk, sb, sr, st.q + 3 * k, st.qd + 3 * k, ts + 3 * k);
#pragma unroll
        for (int j = 0; j < 3; j++) tau[3 * k + j] += ts[3 * k + j];
      }
    }
    if (t == nsettle - 1) {
      kept = true;
#pragma unroll
      for (int i2 = 0; i2 < 12; i2++) { keep[i2] = tm[i2]; keep[12 + i2] = ts[i2]; }
    }
    physics_tick<float, true, QS_BLOCK, kEM>(st, tau, mu, cs, A.M, SCs, t == nsettle - 1, scr, em, &A.M2);
  }
  if (kept) {
#pragma unroll
    for (int i2 = 0; i2 < 12; i2++) { tau_m[i2] = keep[i2]; tau_s[i2] = keep[12 + i2]; }
  }
}

// ActionWrapper._transform_motor_command_to_action (action_interface.py:17-18,41-44,67-74 after
// interface_base.py:92-100): a 12-vector scaled with the interface's limits, reduced to the action space.
__device__ __forceinline__ void command_to_action_space(const EnvCfg& C, const RobotConst& RC, const float* cmd12, float* act12) {
  const bool cart = C.control_mode == QS_CTRL_CARTESIAN_PD;
  float a12[12];
#pragma unroll
  for (int i = 0; i < 12; i++) {
    a12[i] = cart ? command_to_action1(cmd12[i], RC.cart_lo[i], RC.cart_hi[i]) : command_to_action1(cmd12[i], RC.ang_lo[i], RC.ang_hi[i]);
    act12[i] = 0.f;
  }
  if (C.action_mode == QS_ACT_DEFAULT) {
#pragma unroll
    for (int i = 0; i < 12; i++) act12[i] = a12[i];
  } else if (C.action_mode == QS_ACT_SYMMETRIC) {
#pragma unroll
    for (int j = 0; j < 3; j++) { act12[j] = a12[j]; act12[3 + j] = a12[6 + j]; }
  } else if (!cart) { act12[0] = a12[1]; act12[1] = a12[2]; act12[2] = a12[7]; act12[3] = a12[8]; }
  else { act12[0] = a12[0]; act12[1] = a12[2]; act12[2] = a12[6]; act12[3] = a12[8]; }
}

// A fresh robot settled for episode `epoch` of global env `gid`, start to end.
template <bool kEM>
__device__ __forceinline__ void settle_fresh(const KernelArgs& A, int env, uint64_t gid, uint32_t epoch,
                                             EnvState<float>& st, ContactState<float>& cs, float* tau_m, float* tau_s,
                                             float* mu_out, const StepScratch& scr, bool need) {
  // `need` = this thread really settles; the others only keep the block's barriers matched.
  // Must be called by every thread of the block.
  if (!__syncthreads_or(need)) return;
  const float mu = episode_mu(A.C, gid, epoch);
  if (need) *mu_out = mu;
  EnvState<float> st_keep = st;  // a thread that does not need the settle gets its state back untouched
  ContactState<float> cs_keep = cs;
  fresh_state(A, st, cs);
#pragma unroll
  for (int i = 0; i < 12; i++) { tau_m[i] = 0.f; tau_s[i] = 0.f; }
  const int nsettle = settle_length(A.C);
  settle_ticks<kEM>(A, gid, epoch, st, cs, mu, 0, need ? nsettle : 0, nsettle, tau_m, tau_s, scr, A.D.model, A.D.n, env);
  if (!need) { st = st_keep; cs = cs_keep; }
}

// Everything QuadrupedGymEnv.reset does after the settle (quadruped_gym_env.py:282-297),
// from a settled state: counters, task._reset, sensors, filter history; writes the env back.
template <bool kEM>
__device__ __forceinline__ void begin_episode(const KernelArgs& A, int env, uint32_t epoch, float mu,
                                              const EnvState<float>& st, const ContactState<float>& cs,
                                              const float* tau_m, const float* tau_s, float* obs, bool settled = true) {
  const DeviceView& D = A.D;
  const EnvCfg& C = A.C;
  const int n = D.n;
  const float dt = A.SC.dt;
  D.reset_count[env] = epoch;
  D.mu[env] = mu;
  D.custom_gains[env] = 0;
  D.land_mode[env] = 0;
  if (C.rest_mode) {  // GoToRestWrapper.reset: h_old = h_actual = z (go_to_rest_wrapper.py:83-87)
    D.rest_active[env] = 0;
    D.rest[env] = st.pos[2];
  }
#pragma unroll
  for (int i = 0; i < 12; i++) { D.kp[i * n + env] = A.RC.kp[i]; D.kd[i * n + env] = A.RC.kd[i]; }
  if (kEM) episode_model_store(C, uint64_t(C.gid0 + env), epoch, D.model, n, env, D.mass_draw);
  float sk[3], sb[3], sr[3];
  episode_springs(C, A.RC, uint64_t(C.gid0 + env), epoch, sk, sb, sr);
#pragma unroll
  for (int j = 0; j < 3; j++) {
    D.spring[(0 + j) * n + env] = sk[j];
    D.spring[(3 + j) * n + env] = sb[j];
    D.spring[(6 + j) * n + env] = sr[j];
  }
  float cmd[12], act12[12];
  settle_command(C, A.RC, cmd, act12);
  if (!settled) {  // robot_desired_state: no settle, _last_action stays zero (quadruped_gym_env.py:284,288-289)
#pragma unroll
    for (int i = 0; i < 12; i++) act12[i] = 0.f;
  }
  float Rb[9], rpy[3];
  quat_to_R(st.quat, Rb);
  rpy_from_quat(st.quat, rpy);
  float ts[QS_TASK_DIM];
#pragma unroll
  for (int i = 0; i < TS_END_ALL; i++) ts[i] = i < task_slots(C.task) ? D.task[i * n + env] : 0.f;
  const int ds = demo_slot(C.task);
  const float demo_at = ts[ds];
  task_reset(ts, st, cs, tau_m, rpy, Rb, 0.f, C.task);
  if (is_demo_task(C.task)) {  // TaskJumpingDemo._reset (task_base.py:178-183): the counter survives a desired-state reset
    ts[ds] = settled ? 0.f : demo_at;
    ts[ds + 1] = float(C.demo_len) - ts[ds];
  }
#pragma unroll
  for (int i = 0; i < TS_END_ALL; i++) if (i < task_slots(C.task)) D.task[i * n + env] = ts[i];
#pragma unroll
  for (int i = 0; i < 12; i++) {
    D.last_action[i * n + env] = act12[i];
    D.tau_motor[i * n + env] = tau_m[i];
    D.tau_spring[i * n + env] = tau_s[i];
    // action_filter.py:123-127 init_history(last_action)
    D.filt[(0 * 12 + i) * n + env] = act12[i]; D.filt[(1 * 12 + i) * n + env] = act12[i];
    D.filt[(2 * 12 + i) * n + env] = act12[i]; D.filt[(3 * 12 + i) * n + env] = act12[i];
  }
  D.sim_steps[env] = 0;
  D.env_steps[env] = 0;
  D.ep_return[env] = 0.f;
  store_state(D, env, st, cs, dt);
  if (obs) {
    float o[QS_MAX_OBS];
#pragma unroll
    for (int i = 0; i < QS_MAX_OBS; i++) o[i] = 0.f;
    observe(st, cs, ts, rpy, Rb, C.obs_mode, C.task, o);
    store_obs(obs + size_t(env) * C.obs_dim, o, C, A.RC, uint64_t(C.gid0 + env), epoch, 0u, C.enable_noise);
  }
}

// Epilogue of a control step (quadruped_gym_env.py:239-256) + write-back + auto-reset.
// kStored: the caller (k_finish) read state and torques from the env's rows, where the tick kernel left them: the plain
// write-back at the end does not store them again
template <bool kEM, bool kStored = false>
__device__ __forceinline__ void finish_step(const KernelArgs& A, const StepIO& io, int env, EnvState<float>& st,
                                            ContactState<float>& cs, const float* tau_m, const float* tau_s,
                                            float* sm /* this thread's column of >= QS_SELF_SCRATCH shared floats */, int sm_stride) {
  const DeviceView& D = A.D;
  const EnvCfg& C = A.C;
  const int n = D.n;
  const float dt = A.SC.dt;
  const int sim_steps = D.sim_steps[env] + C.action_repeat;
  const int env_steps = D.env_steps[env] + 1;
  float Rb[9], rpy[3];
  quat_to_R(st.quat, Rb);
  rpy_from_quat(st.quat, rpy);
  const float sim_time = float(double(sim_steps) * A.time_step_d);
  // NaN / Inf guard (SURVEY.md section 5): a state that stopped being finite (a poisoned set_state, a solver
  // blow-up) must not spread into rewards, statistics and the policy's batch.  The env is cut off: done = 1,
  // truncated = 0, reward 0, a zero observation, and -- with auto_reset -- a fresh episode like any other done.
  bool finite = true;
  {
    // exponent all ones <=> NaN or +-Inf; min over the 37 words of (0x7f800000 - exponent bits) hits 0 for those
    uint32_t room = 0x7f800000u;
    auto look = [&](float x) { room = min(room, 0x7f800000u - (__float_as_uint(x) & 0x7f800000u)); };
#pragma unroll
    for (int i = 0; i < 3; i++) { look(st.pos[i]); look(st.vlin[i]); look(st.vang[i]); }
#pragma unroll
    for (int i = 0; i < 4; i++) look(st.quat[i]);
#pragma unroll
    for (int i = 0; i < 12; i++) { look(st.q[i]); look(st.qd[i]); }
    finite = room != 0u;
  }
  if (!finite) {
    fresh_state(A, st, cs);  // something finite to read back (without auto_reset the caller has to reset the env)
    quat_to_R(st.quat, Rb);
    rpy_from_quat(st.quat, rpy);
  }
  if (A.SC.self_collision) {
    // Self contacts of the last tick's collision phase, i.e. on the poses at the START of that tick:
    // q_before = q - dt * qd (integrate_positions).  Calf-involved pairs are invalid contacts (quadruped.py:236-241).
    float qb[12];
#pragma unroll
    for (int i = 0; i < 12; i++) qb[i] = st.q[i] - dt * st.qd[i];
    cs.invalid += self_collision_count(qb, A.M, sm, sm_stride);
  }
  float ts[QS_TASK_DIM];
#pragma unroll
  for (int i = 0; i < TS_END_ALL; i++) ts[i] = i < task_slots(C.task) ? D.task[i * n + env] : 0.f;
  float foot_force[4];
#pragma unroll
  for (int k = 0; k < 4; k++) foot_force[k] = (cs.mask >> k) & 1 ? cs.lam_n[k] / dt : 0.f;
  task_on_step(ts, st, cs, tau_m, rpy, Rb, sim_time, C.task);
  float r = task_reward(ts, st, foot_force, ts + TS_OLD_TAU0, tau_m, rpy, Rb, C.task);
  bool term = task_terminated(ts, st, cs, Rb, A.RC.fallen_height, C.task);
  if (is_demo_task(C.task)) {
    // TaskJumpingDemo._reward / _terminated (task_base.py:194-212): distance of this step's action to the demonstration's
    const int ds = demo_slot(C.task);
    const int row = min(int(ts[ds]), C.demo_len - 1);
    float s = 0.f;
    for (int i = 0; i < C.action_dim; i++) {
      const float d = C.demo[row * C.action_dim + i] - D.last_action[i * n + env];
      s += d * d;
    }
    r = expf(-0.35f * sqrtf(s)) / ts[ds + 1];
    ts[ds] += 1.f;
    term = term || int(ts[ds]) == C.demo_len;
  }
  if (!finite) term = true;
  const bool dn = term || (double(sim_steps) * A.time_step_d > A.max_time_d);
  if (dn) r += task_reward_end(ts, term, C.task, sim_time, C.max_episode_time);
  if (!finite) r = 0.f;
#pragma unroll
  for (int i = 0; i < 12; i++) ts[TS_OLD_TAU0 + i] = finite ? tau_m[i] : 0.f;
  const float ep_ret = D.ep_return[env] + r;
  io.reward[env] = r;
  io.done[env] = dn;
  io.truncated[env] = dn && !term;
  D.work[0 * n + env] += uint32_t(C.action_repeat);
  const uint64_t gid = uint64_t(C.gid0 + env);
  int land_now = C.landing_mode ? D.land_mode[env] : LAND_POLICY;
  if (C.landing_mode && !dn) {
    const int mode = land_now, lm = C.landing_mode;
    const bool flying = (cs.mask & 15) == 0;
    // what starts the scripted phase: the take-off switch (landing_wrapper.py:58-66) or, continuous variant, a detected jump
    const bool trigger = lm == 3 ? ts[TS_IS_JUMPING] != 0.f : ts[TS_SWITCHED] != 0.f;
    if (mode == LAND_POLICY && trigger) {
      if (lm >= 4) {
        land_now = LAND_TAKEOFF_BF;  // landing_wrapper_backflip.py:54-60,72-73
      } else {                               // take_off_phase with the apex timer, start_jumping_timer :47-60
        land_now = LAND_HOLD;
        D.land_timer[env] = sim_time;
        D.land_timer[n + env] = sim_time + st.vlin[2] / 9.81f;  // task.compute_time_for_peak_heihgt, task_base.py:157-160
      }
    } else if (mode == LAND_TAKEOFF_BF) {
      // until PitchBackFlip._get_pitch >= 5 pi / 8 (landing_wrapper_backflip.py:22-23,57-60)
      if (backflip_pitch(Rb, ts[TS_SWITCHED] != 0.f) >= 5.f * float(QS_PI) / 8.f)
        land_now = (lm == 5 && !flying) ? LAND_SPENT : LAND_LANDING;  // backflip2: `while ... and is_flying` :50
    } else if (mode == LAND_LANDING) {
      if ((lm == 2 || lm == 5) && !flying) land_now = LAND_SPENT;             // landing_wrapper_2.py:39-46,71
      else if (lm == 3 && ts[TS_IS_JUMPING] == 0.f) land_now = LAND_POLICY;  // landing_wrapper_continuous.py:39-46
    }
    D.land_mode[env] = land_now;
  }
  if (C.rest_mode && !dn && (land_now == LAND_POLICY || land_now == LAND_SPENT) && D.rest_active[env] == 0) {
    // GoToRestWrapper.step (go_to_rest_wrapper.py:43-52) runs where the wrapper below it returns, i.e. after a
    // step that leaves the landing controller unscripted; rest_condition :89-95
    const float h_old = D.rest[env];
    D.rest[env] = st.pos[2];
    if (ts[TS_SWITCHED] != 0.f && (cs.mask & 15) == 15 && st.pos[2] - h_old > 0.f) {
      D.rest_active[env] = 1;
      D.rest[1 * n + env] = float(sim_steps);  // t_start as a tick count: exact
      float start[12];
      command_to_action_space(C, A.RC, st.q, start);  // get_start_action :54-56
#pragma unroll
      for (int i = 0; i < 12; i++) {
        D.rest[(2 + i) * n + env] = start[i];
        D.kp[i * n + env] = 60.f;  // temporary_switch_motor_control_gain :21-41, until the episode ends
        D.kd[i * n + env] = C.enable_springs ? 0.8f : 1.5f;
      }
      D.custom_gains[env] = 1;
    }
  }
  if (dn) finish_episode_stats(D, env, ts, ep_ret, env_steps, term, C.task, !finite);
  // ---- sensors (:253-254)
  float o[QS_MAX_OBS];
#pragma unroll
  for (int i = 0; i < QS_MAX_OBS; i++) o[i] = 0.f;
  observe(st, cs, ts, rpy, Rb, C.obs_mode, C.task, o);
  if (dn && C.auto_reset) {
    // SB3's VecEnv contract: infos["terminal_observation"] of an env that is reset inside step_wait
    if (io.term_obs)
      store_obs(io.term_obs + size_t(env) * C.obs_dim, o, C, A.RC, gid, D.reset_count[env], uint32_t(env_steps), C.enable_noise);
    // the finished env starts its next episode inside the same call; its obs row becomes the
    // first observation of that episode (SB3 VecEnv convention)
#pragma unroll
    for (int i = 0; i < TS_END_ALL; i++) if (i < task_slots(C.task)) D.task[i * n + env] = ts[i];  // BackFlip.max_pitch survives resets
    const uint32_t epoch = D.reset_count[env] + 1;
    if (slot_ready(D, env, epoch)) {
      float tm[12], tsp[12], mu;
      slot_load(D, env, epoch, st, cs, tm, tsp, &mu, dt);
      D.slot_epoch[int(epoch % QS_SLOTS) * n + env] = 0;
      conveyor_push(io.cv, env, epoch + QS_SLOTS);  // the freed slot's next tenant
      atomicAdd(io.cv.ctl + CV_TAKEN, 1u);           // feedback for the slice length (k_conveyor_ctl)
      if (!slot_ready(D, env, epoch + 1)) atomicAdd(io.cv.ctl + CV_LOW2, 1u);
      begin_episode<kEM>(A, env, epoch, mu, st, cs, tm, tsp, io.obs);
    } else {
      // no spare slot ready: an urgent entry makes k_settle_urgent (launched at the end of this step)
      // settle this episode now and start it; same numbers as the prefetched path
      store_state(D, env, st, cs, dt);
      urgent_push(io.cv, env, epoch);
    }
    return;
  }
  // ---- write-back
  store_obs(io.obs + size_t(env) * C.obs_dim, o, C, A.RC, gid, D.reset_count[env], uint32_t(env_steps), C.enable_noise);
  if (!kStored || !finite) {
    store_state(D, env, st, cs, dt);
#pragma unroll
    for (int i = 0; i < 12; i++) { D.tau_motor[i * n + env] = finite ? tau_m[i] : 0.f; D.tau_spring[i * n + env] = finite ? tau_s[i] : 0.f; }
  } else if (A.SC.self_collision) {
    D.contact[env] = (cs.mask & 15) | (cs.invalid << 8);   // the self-collision count joined cs.invalid after the store
  }
#pragma unroll
  for (int i = 0; i < TS_END_ALL; i++) if (i < task_slots(C.task)) D.task[i * n + env] = ts[i];
  D.sim_steps[env] = sim_steps;
  D.env_steps[env] = env_steps;
  D.ep_return[env] = ep_ret;
}

// All ticks of the control step are done: the state and the last tick's torques go back to the env's rows, and k_finish
// (one thread per env, a small kernel at full occupancy) runs the step's epilogue from there.  The tick kernels are
// pinned at 255 registers and 8 warps per SM: the epilogue's dependent chains (task logic, self collision, Philox noise)
// cost several times more inside them than in a kernel of their own (round 2: +0.07 ms per step for the self-collision
// test alone when it ran in the tick kernels' tails).
__device__ __forceinline__ void tick_done_store(const KernelArgs& A, int env, const EnvState<float>& st,
                                                const ContactState<float>& cs, const float* tau_m, const float* tau_s) {
  const DeviceView& D = A.D;
  const int n = D.n;
  store_state(D, env, st, cs, A.SC.dt);
#pragma unroll
  for (int i = 0; i < 12; i++) { D.tau_motor[i * n + env] = tau_m[i]; D.tau_spring[i * n + env] = tau_s[i]; }
  D.work[1 * n + env] += uint32_t(cs.work_contacts);
  D.work[2 * n + env] += uint32_t(cs.work_row_iters);
  D.resume_tick[env] = A.C.action_repeat;   // "ticks done, epilogue pending"
}

// hand an env over to another kernel of the step: state as of the start of tick `t`
__device__ __forceinline__ void park_env(const KernelArgs& A, const StepIO& io, int env, const EnvState<float>& st,
                                         const ContactState<float>& cs, const float* cmd, int t, int* list,
                                         bool store = true) {
  const DeviceView& D = A.D;
  const int n = D.n;
  if (store) {
    store_state(D, env, st, cs, A.SC.dt);
    D.work[1 * n + env] += uint32_t(cs.work_contacts);
    D.work[2 * n + env] += uint32_t(cs.work_row_iters);
  }
#pragma unroll
  for (int i = 0; i < 12; i++) D.cmd[i * n + env] = cmd[i];
  D.resume_tick[env] = t;
  list[atomicAdd(list + n, 1)] = env;
}

// -------------------------------------------------------------------- K0: action -> motor command, and who goes where
// The step's prologue for every env (quadruped_gym_env.py:229-234: scripted-controller overrides, _last_action, action
// filter, action -> motor command) and the classification the step kernels work from: an env with a foot on the ground
// goes straight to k_step_contact's list, the others to the flight kernel's, so that both run dense warps.
__global__ void __launch_bounds__(256)
k_pre(const __grid_constant__ KernelArgs A, const StepIO io) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const EnvCfg& C = A.C;
  const int n = D.n;
  const bool live = tid < n;
  const int env = live ? tid : n - 1;
  if (tid == 0 && io.stamps) { io.stamps[0] = ~0ull; io.stamps[1] = 0ull; io.stamps[2] = ~0ull; io.stamps[3] = 0ull; }
  // ---- action (quadruped_gym_env.py:229-234)
  float act[12];
#pragma unroll
  for (int i = 0; i < 12; i++) act[i] = i < C.action_dim ? io.actions[size_t(env) * C.action_dim + i] : 0.f;
  if (C.rest_mode && D.rest_active[env]) {
    // go_to_rest (go_to_rest_wrapper.py:58-81): ramp from the pose at activation to the init action
    // (generate_ramp, interface_base.py:112-119), then hold it; the policy's action is ignored
    float cmd0[12], init12[12];
    settle_command(C, A.RC, cmd0, init12);  // ac_interface.get_init_action(), interface_base.py:74-78
    const float T = C.enable_springs ? 1.0f : 0.3f;
    const float el = float(double(D.sim_steps[env] - int(D.rest[1 * n + env])) * A.time_step_d);
#pragma unroll
    for (int i = 0; i < 12; i++) {
      const float s0 = D.rest[(2 + i) * n + env];
      act[i] = el < 0.f ? s0 : (el > T ? init12[i] : s0 + (init12[i] - s0) * el / T);
    }
  }
  if (C.landing_mode) {
    // landing controllers (landing_wrapper.py:38-66, landing_wrapper_2.py:39-72) as a mode machine: the
    // wrappers' inner env.step loops, one control step per call; a scripted env ignores the policy's action
    int mode = D.land_mode[env];
    if (mode == LAND_HOLD) {  // take_off_phase: repeat the action until the timer is up (utils/timer.py:39-43)
      const float timer = D.land_timer[env];
      if (timer > D.land_timer[n + env]) {
        mode = LAND_LANDING;
        if (live) D.land_mode[env] = mode;
        if (C.landing_mode == 1 && live) {  // temporary_switch_motor_control_gain, landing_wrapper.py:18-36
#pragma unroll
          for (int i = 0; i < 12; i++) { D.kp[i * n + env] = 60.f; D.kd[i * n + env] = 1.5f; }
          D.custom_gains[env] = 1;
        }
      } else {
        if (live) D.land_timer[env] = timer + A.RC.env_dt;  // step_timer
#pragma unroll
        for (int i = 0; i < 12; i++) act[i] = D.last_action[i * n + env];
      }
    }
    if (mode == LAND_TAKEOFF_BF) {  // take_off_action (0, 1, -1) per leg pair, landing_wrapper_backflip.py:21
#pragma unroll
      for (int i = 0; i < 12; i++) act[i] = i >= 6 ? 0.f : (i % 3 == 0 ? 0.f : (i % 3 == 1 ? 1.f : -1.f));
    }
    if (mode == LAND_LANDING) {
#pragma unroll
      for (int i = 0; i < 12; i++) act[i] = A.RC.landing_action[i];
    }
  }
  if (live) {
#pragma unroll
    for (int i = 0; i < 12; i++) D.last_action[i * n + env] = act[i];
  }
  if (C.enable_filter) {  // utils/action_filter.py:110-121
#pragma unroll
    for (int i = 0; i < 12; i++) {
      if (i < C.action_dim) {
        float* f = D.filt + env;
        const float x0 = f[(0 * 12 + i) * n], x1 = f[(1 * 12 + i) * n];
        const float y0 = f[(2 * 12 + i) * n], y1 = f[(3 * 12 + i) * n];
        const float y = act[i] * A.RC.filt_b[0] + (x0 * A.RC.filt_b[1] + x1 * A.RC.filt_b[2]) -
                        (y0 * A.RC.filt_a[1] + y1 * A.RC.filt_a[2]);
        if (live) {
          f[(1 * 12 + i) * n] = x0; f[(0 * 12 + i) * n] = act[i];
          f[(3 * 12 + i) * n] = y0; f[(2 * 12 + i) * n] = y;
        }
        act[i] = y;
      }
    }
  }
  float cmd[12];
  bool torque_mode = false;
  if (C.is_rl) {
    // _interpolate_actions (:187-205) is a no-op in the reference: step() overwrites
    // _last_action with the current action before the substeps (:229-234).
    float a12[12];
    expand_action(C.action_mode, C.control_mode == QS_CTRL_CARTESIAN_PD ? 1 : 0, act, a12);
    action12_to_command(A.RC, C.control_mode, a12, cmd);
  } else {
#pragma unroll
    for (int i = 0; i < 12; i++) cmd[i] = act[i];
    torque_mode = C.control_mode == QS_CTRL_TORQUE;
  }

  bool grounded = false;
  if (live) {
#pragma unroll
    for (int i = 0; i < 12; i++) D.cmd[i * n + env] = cmd[i];
    D.resume_tick[env] = 0;
    grounded = (D.contact[env] & 15) != 0;  // standing / pushing
  }
  // one atomic per warp and list
  const unsigned lane = threadIdx.x & 31u;
  const unsigned mg = __ballot_sync(0xffffffffu, live && grounded), mf = __ballot_sync(0xffffffffu, live && !grounded);
  int bg = 0, bf = 0;
  if (lane == 0) {
    if (mg) bg = atomicAdd(io.contact_list + n, __popc(mg));
    if (mf) bf = atomicAdd(io.flight_list + n, __popc(mf));
  }
  bg = __shfl_sync(0xffffffffu, bg, 0);
  bf = __shfl_sync(0xffffffffu, bf, 0);
  const unsigned below = (1u << lane) - 1u;
  if (live && grounded) io.contact_list[bg + __popc(mg & below)] = env;
  // The flight kernel runs whole waves of blocks: a few blocks more than a wave cost a second round on a nearly idle
  // GPU (~1.2 waves under the benchmark's actions: 0.20 ms instead of 0.12).  Envs beyond one wave go to the contact
  // kernel instead, which has room (about half a wave) and runs the same tick with the contact code skipped while no foot
  // is near the ground.
  if (live && !grounded) {
    const int at = bf + __popc(mf & below);
    if (at < io.flight_cap) io.flight_list[at] = env;
    else io.contact_list[atomicAdd(io.contact_list + n, 1)] = env;
  }
  (void)torque_mode;
}

// -------------------------------------------------------------------- K1: step, flight part
// The envs with no foot on the ground (dense warps: thread i takes flight_list[i]): flight variant of the tick, no
// foot-contact code.  An env that reaches the ground goes on to k_step_contact as of the start of that tick.
// kTrace (all three tick kernels): the variant launched while a substep trace is set (qs_set_substep_trace); `tr` is
// read by that variant only.  kExt: likewise while a push buffer is attached (qs_set_external_force), `ef`.
template <bool kEM, bool kTrace, bool kExt>
__global__ void __launch_bounds__(256, 1)
k_step(const __grid_constant__ KernelArgs A, const StepIO io, const SubstepTrace tr, const ExtForce ef) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const EnvCfg& C = A.C;
  const int n = D.n;
  const int count = min(io.flight_list[n], io.flight_cap);
  if (blockIdx.x * blockDim.x >= count) return;  // uniform over the block
  // threads past the end shadow the last entry (block-wide barriers inside run_ticks need every
  // thread); they compute the same thing and write nothing
  const bool live = tid < count;
  const int env = io.flight_list[live ? tid : count - 1];
  EnvState<float> st;
  ContactState<float> cs;
  load_state(D, env, st, cs, A.SC.dt);
  float cmd[12];
#pragma unroll
  for (int i = 0; i < 12; i++) cmd[i] = D.cmd[i * n + env];
  const bool torque_mode = !C.is_rl && C.control_mode == QS_CTRL_TORQUE;

  // ---- action_repeat substeps (:236-237)
  float tau_m[12], tau_s[12];
  extern __shared__ __align__(16) float qs_smem[];
  const StepScratch scr{qs_smem, QS_BLOCK, int(threadIdx.x)};
  int why;
  const int t_done = run_ticks<false, kEM, kTrace, kExt>(st, cs, cmd, torque_mode, 0, C.action_repeat, env, D, C, A.RC, A.M, A.M2, A.SC,
                                                    tau_m, tau_s, true, scr, &why,
                                                    kTrace ? trace_column(tr, env, live) : TraceColumn{nullptr, 0}, false,
                                                    kExt ? ext_push(ef, env, n) : ExtPush{});
  if (!live) return;
  if (t_done < C.action_repeat) {
    park_env(A, io, env, st, cs, cmd, t_done, why == TICK_NEEDS_GENERAL ? io.slow_list : io.contact_list);
    return;
  }
  tick_done_store(A, env, st, cs, tau_m, tau_s);
}

// -------------------------------------------------------------------- K1a: envs with foot contacts
// Resumes the envs the flight kernel handed over (dense warps: thread i takes contact_list[i]) with
// the full fast tick; joint limits / body contacts still go on to k_step_slow.
template <bool kEM, bool kTrace, bool kExt>
__global__ void __launch_bounds__(256, 1)
k_step_contact(const __grid_constant__ KernelArgs A, const StepIO io, const SubstepTrace tr, const ExtForce ef) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const EnvCfg& C = A.C;
  const int n = D.n;
  const int count = io.contact_list[n];
  if (blockIdx.x * blockDim.x >= count) return;  // uniform over the block
  const bool live = tid < count;
  const int env = io.contact_list[live ? tid : count - 1];
  EnvState<float> st;
  ContactState<float> cs;
  load_state(D, env, st, cs, A.SC.dt);
  float cmd[12], tau_m[12], tau_s[12];
#pragma unroll
  for (int i = 0; i < 12; i++) cmd[i] = D.cmd[i * n + env];
  const bool torque_mode = !C.is_rl && C.control_mode == QS_CTRL_TORQUE;
  extern __shared__ __align__(16) float qs_smem[];
  const StepScratch scr{qs_smem, QS_BLOCK, int(threadIdx.x)};
  int why;
  const int t_done = run_ticks<true, kEM, kTrace, kExt>(st, cs, cmd, torque_mode, D.resume_tick[env], C.action_repeat, env, D, C, A.RC,
                                                   A.M, A.M2, A.SC, tau_m, tau_s, true, scr, &why,
                                                   kTrace ? trace_column(tr, env, live) : TraceColumn{nullptr, 0}, false,
                                                   kExt ? ext_push(ef, env, n) : ExtPush{});
  if (!live) return;
  if (t_done < C.action_repeat) {
    park_env(A, io, env, st, cs, cmd, t_done, io.slow_list);
    return;
  }
  tick_done_store(A, env, st, cs, tau_m, tau_s);
}

// -------------------------------------------------------------------- K1b: general-solver continuation
template <bool kEM, bool kTrace, bool kExt>
__global__ void __launch_bounds__(64)
k_step_slow(const __grid_constant__ KernelArgs A, const StepIO io, int spread, const SubstepTrace tr, const ExtForce ef) {
  // Programmatic dependent launch: the late settle slice follows in the same stream and may start as soon as every block
  // of this grid has been placed (has got here or exited), not when the grid is complete.  That ordering is the point: the
  // slice fills every SM, and when the hardware happened to place it first (two streams racing), the few latency-bound
  // blocks of this kernel waited for the whole slice: +1 ms on that step.
  asm volatile("griddepcontrol.launch_dependents;");
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const int n = D.n;
  // `spread` envs per warp: these envs take different paths through the general solver (which shapes touch, which
  // limits are active), so a full warp runs the union of 32 paths; the kernel is a few hundred envs, latency-bound,
  // on an otherwise idle part of the GPU, so fewer envs per warp shorten the step's serial chain.
  const int count = io.slow_list[n];
  const int warps = int(gridDim.x * blockDim.x) >> 5;
  int K = spread;
  while (K < 32 && (count + K - 1) / K > warps) K <<= 1;  // a list too long for the grid packs denser
  const int lane = tid & 31;
  if (lane >= K) return;
  const int idx = (tid >> 5) * K + lane;
  if (idx >= count) return;
  const int env = io.slow_list[idx];
  if (lane == 0) stamp_begin(io.stamps ? io.stamps + 2 : nullptr);
  EnvState<float> st;
  ContactState<float> cs;
  load_state(D, env, st, cs, A.SC.dt);
  float cmd[12], tau_m[12], tau_s[12];
#pragma unroll
  for (int i = 0; i < 12; i++) cmd[i] = D.cmd[i * n + env];
  const bool torque_mode = !A.C.is_rl && A.C.control_mode == QS_CTRL_TORQUE;
  __shared__ float dl_sm[12 * 64];   // the solver's per-leg vector delta (qs_physics.cuh GenRow), one column per thread
  if constexpr (kTrace && kExt)
    run_ticks_general<kEM, true, true>(st, cs, cmd, torque_mode, D.resume_tick[env], A.C.action_repeat, env, D, A.C, A.RC, A.M,
                                       A.SC, tau_m, tau_s, dl_sm + threadIdx.x, 64, trace_column(tr, env, true),
                                       ext_push(ef, env, n));
  else if constexpr (kTrace)
    run_ticks_general<kEM, true>(st, cs, cmd, torque_mode, D.resume_tick[env], A.C.action_repeat, env, D, A.C, A.RC, A.M, A.SC,
                                 tau_m, tau_s, dl_sm + threadIdx.x, 64, trace_column(tr, env, true));
  else if constexpr (kExt)
    run_ticks_general<kEM, false, true>(st, cs, cmd, torque_mode, D.resume_tick[env], A.C.action_repeat, env, D, A.C, A.RC, A.M,
                                        A.SC, tau_m, tau_s, dl_sm + threadIdx.x, 64, ext_push(ef, env, n));
  else
    run_ticks_general<kEM>(st, cs, cmd, torque_mode, D.resume_tick[env], A.C.action_repeat, env, D, A.C, A.RC, A.M, A.SC,
                      tau_m, tau_s, dl_sm + threadIdx.x, 64);
  // The epilogue of these envs runs here (not in k_finish): this kernel ends well before the late settle slice it runs
  // next to, while a kernel launched after it would have to wait for that slice.
  D.work[1 * n + env] += uint32_t(cs.work_contacts);
  D.work[2 * n + env] += uint32_t(cs.work_row_iters);
  D.resume_tick[env] = -1;
  float sc_pts[QS_SELF_SCRATCH];   // (local memory like the solver rows: more shared memory would keep this kernel's blocks off
                                   // the SMs the settle slice fills)
  finish_step<kEM>(A, io, env, st, cs, tau_m, tau_s, sc_pts, 1);
  stamp_end(io.stamps ? io.stamps + 2 : nullptr);
}

// -------------------------------------------------------------------- K1c: the step's epilogue
// One thread per env (list == nullptr) or per entry of `list` (list[n] = count): the envs whose ticks are done run
// finish_step -- task bookkeeping, reward, done, self-collision test, observation + noise, auto-reset.  Launched after
// k_step_contact for everybody and after k_step_slow for the general solver's envs.
constexpr int QS_FINISH_BLOCK = 128;
template <bool kEM>
__global__ void __launch_bounds__(QS_FINISH_BLOCK, 4)
k_finish(const __grid_constant__ KernelArgs A, const StepIO io, const int* __restrict__ list) {
  // (device-buffer steps launch this kernel behind k_step_slow and the late settle slice behind it, both as programmatic
  // dependents: the slice may be scheduled once every block of this grid has been placed -- none of them then waits
  // behind a slice block -- and fills the SMs as they drain.  A no-op under an ordinary launch.)
  asm volatile("griddepcontrol.launch_dependents;");
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const int n = D.n;
  const int count = list ? list[n] : n;
  if (tid >= count) return;
  const int env = list ? list[tid] : tid;
  if (D.resume_tick[env] != A.C.action_repeat) return;   // parked for the general solver, or already finished
  D.resume_tick[env] = -1;
  EnvState<float> st;
  ContactState<float> cs;
  load_state(D, env, st, cs, A.SC.dt);
  float tau_m[12];
#pragma unroll
  for (int i = 0; i < 12; i++) tau_m[i] = D.tau_motor[i * n + env];
  __shared__ float sc_pts[QS_SELF_SCRATCH * QS_FINISH_BLOCK];
  finish_step<kEM, true>(A, io, env, st, cs, tau_m, tau_m /* spring torques: only stored, and not by this caller */, sc_pts + threadIdx.x, QS_FINISH_BLOCK);
}

// -------------------------------------------------------------------- K2: reset + settle
// list == nullptr: thread i resets env i (all envs).  Otherwise thread i resets env list[i]
// for i < list[n] (dense warps whatever the done pattern).
template <bool kEM>
__global__ void __launch_bounds__(256, 1)
k_reset(const __grid_constant__ KernelArgs A, const int* __restrict__ list, const Conveyor cv,
        float* __restrict__ obs) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const int n = D.n;
  const int count = list ? list[n] : n;
  if (count == 0) return;                       // uniform over the grid
  if (blockIdx.x * blockDim.x >= count) return;  // uniform over the block
  const bool live = tid < count;                 // stragglers shadow the last entry and write nothing
  const int idx = live ? tid : count - 1;
  const int env = list ? list[idx] : idx;
  const uint64_t gid = uint64_t(A.C.gid0 + env);
  const uint32_t epoch = D.reset_count[env] + 1;
  EnvState<float> st;
  ContactState<float> cs;
  float tau_m[12], tau_s[12], mu;
  const bool have = slot_ready(D, env, epoch);
  extern __shared__ __align__(16) float qs_smem[];
  const StepScratch scr{qs_smem, QS_BLOCK, int(threadIdx.x)};
  float tm2[12], ts2[12];
  settle_fresh<kEM>(A, env, gid, epoch, st, cs, tm2, ts2, &mu, scr, !have);
  if (have) {
    slot_load(D, env, epoch, st, cs, tau_m, tau_s, &mu, A.SC.dt);
  } else {
#pragma unroll
    for (int i = 0; i < 12; i++) { tau_m[i] = tm2[i]; tau_s[i] = ts2[i]; }
  }
  if (!live) return;
  if (A.C.auto_reset) {
    if (have) D.slot_epoch[int(epoch % QS_SLOTS) * n + env] = 0;
    // every future episode within the ring must be present or queued (a duplicate of an entry already
    // on the conveyor settles twice and stores the same rows)
#pragma unroll
    for (int d = 1; d <= QS_SLOTS; d++)
      if (!slot_ready(D, env, epoch + d)) conveyor_push(cv, env, epoch + d);
  }
  begin_episode<kEM>(A, env, epoch, mu, st, cs, tau_m, tau_s, obs);
}

// QuadrupedGymEnv.reset with robot_desired_state set (quadruped_gym_env.py:288-289, quadruped.py:470-471,521-525;
// ReferenceStateInitializationWrapper): the robot is placed in the given state [N][37] and NOT settled.
template <bool kEM>
__global__ void __launch_bounds__(128)
k_reset_state(const __grid_constant__ KernelArgs A, const int* __restrict__ list, const float* __restrict__ states,
              const Conveyor cv, float* __restrict__ obs) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const int n = D.n;
  const int count = list ? list[n] : n;
  if (tid >= count) return;
  const int env = list ? list[tid] : tid;
  const uint32_t epoch = D.reset_count[env] + 1;
  EnvState<float> st;
  ContactState<float> cs;
  fresh_state(A, st, cs);  // no contact points until the first stepSimulation
  const float* s = states + size_t(env) * QS_STATE_DIM;
#pragma unroll
  for (int i = 0; i < 3; i++) { st.pos[i] = s[i]; st.vlin[i] = s[7 + i]; st.vang[i] = s[10 + i]; }
#pragma unroll
  for (int i = 0; i < 4; i++) st.quat[i] = s[3 + i];
#pragma unroll
  for (int i = 0; i < 12; i++) { st.q[i] = s[13 + i]; st.qd[i] = s[25 + i]; }
  float zero12[12];
#pragma unroll
  for (int i = 0; i < 12; i++) zero12[i] = 0.f;
  if (A.C.auto_reset) {
    // this episode's prefetched slot (if any) is skipped; the ring keeps the episodes after it
    if (slot_ready(D, env, epoch)) D.slot_epoch[int(epoch % QS_SLOTS) * n + env] = 0;
#pragma unroll
    for (int d = 1; d <= QS_SLOTS; d++)
      if (!slot_ready(D, env, epoch + d)) conveyor_push(cv, env, epoch + d);
  }
  begin_episode<kEM>(A, env, epoch, episode_mu(A.C, uint64_t(A.C.gid0 + env), epoch), st, cs, zero12, zero12, obs, false);
}

// Episodes of envs that finished without a ready slot: settled start to end and started, in stream
// order at the end of the step.  Exits at once when there is none (the usual case).
template <bool kEM>
__global__ void __launch_bounds__(256, 1)
k_settle_urgent(const __grid_constant__ KernelArgs A, const Conveyor cv, float* __restrict__ obs) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  const int count = int(cv.ctl[CV_URGENT]);
  if (blockIdx.x * blockDim.x >= count) return;  // uniform over the block
  const bool live = tid < count;
  const int i = live ? tid : count - 1;
  const int env = cv.urgent_list[2 * i];
  const uint32_t epoch = uint32_t(cv.urgent_list[2 * i + 1]);
  EnvState<float> st;
  ContactState<float> cs;
  float tau_m[12], tau_s[12], mu = 0.f;
  extern __shared__ __align__(16) float qs_smem[];
  const StepScratch scr{qs_smem, QS_BLOCK, int(threadIdx.x)};
  settle_fresh<kEM>(A, env, uint64_t(A.C.gid0 + env), epoch, st, cs, tau_m, tau_s, &mu, scr, live);
  if (!live) return;
  // its ring: the slot of this episode never became ready, the others may be missing too
#pragma unroll
  for (int d = 1; d <= QS_SLOTS; d++)
    if (!slot_ready(D, env, epoch + d)) conveyor_push(cv, env, epoch + d);
  begin_episode<kEM>(A, env, epoch, mu, st, cs, tau_m, tau_s, obs);
}
__global__ void k_urgent_clear(Conveyor cv) {
  cv.ctl[CV_URGENT_LAST] = cv.ctl[CV_URGENT];
  cv.ctl[CV_URGENT] = 0;
}

// Conveyor bookkeeping.  The slice length follows the demand (entries pushed per step, smoothed): with d
// episodes ending per step, nsettle * d / slice entries are in flight, and the slice is chosen so that they
// fill ~90 % of one wave -- the settles then run as a dense launch whatever the episode length.  With few
// envs that would deliver too late, so a settle is also kept shorter than half a mean episode, and the
// slice grows while envs find their ring nearly empty.  Entries beyond the window (start-up, bursts) or
// flush != 0 run the window to completion at once.
//
// A step runs two slices, each next to a latency-bound kernel that leaves SMs idle:
//   phase 0 (after k_step):         retire the finished entries at the tail, update demand and pressure, and give
//                                   the oldest entries that fit next to k_step_contact's blocks `early` ticks;
//   phase 1 (after k_step_contact): the entries that fit next to k_step_slow's blocks get the rest of the ticks.
__global__ void k_conveyor_ctl(Conveyor cv, int phase, const int* __restrict__ busy_count, int busy_block, int wave_blocks,
                               int block, int n_envs, int nsettle, int s_min, int s_max, int early, int flush) {
  __shared__ uint32_t first_live;
  const uint32_t head = cv.ctl[CV_HEAD];
  uint32_t tail = cv.ctl[CV_TAIL];
  if (phase == 0 || flush) {
    const uint32_t span = min(head - tail, uint32_t(cv.width));
    if (threadIdx.x == 0) first_live = span;
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < span; j += blockDim.x)
      if (cv.tick[(tail + j) & cv.cap_mask] != CV_DONE) { atomicMin(&first_live, j); break; }
    __syncthreads();
    tail += first_live;
  }
  if (threadIdx.x != 0) return;
  cv.ctl[CV_TAIL] = tail;
  const uint32_t pending = head - tail;
  if (flush) {
    cv.ctl[CV_ACTIVE] = min(pending, uint32_t(cv.width));
    cv.ctl[CV_SLICE] = uint32_t(nsettle);
    cv.ctl[CV_PREV_HEAD] = head;
    return;
  }
  // room next to the other kernel of this phase (busy_block = envs of it per block slot it takes from the slice)
  const int lanes = max(0, min(cv.width, (wave_blocks - (*busy_count + busy_block - 1) / busy_block) * block));
  const bool backlog = pending > uint32_t(cv.width);
  if (phase == 0) {
    float demand = __uint_as_float(cv.ctl[CV_DEMAND]);
    demand += (float(head - cv.ctl[CV_PREV_HEAD]) - demand) * 0.125f;
    cv.ctl[CV_DEMAND] = __float_as_uint(demand);
    cv.ctl[CV_PREV_HEAD] = head;
    // dense wave: nsettle * demand / slice entries in flight = target; ring safety: the settle must not take
    // longer than half a mean episode (n_envs / demand steps, Little's law)
    const float target = 0.9f * float(cv.width);
    float want = float(nsettle) * demand * fmaxf(1.f / target, 2.f / float(n_envs));
    if (float(pending) > 0.97f * float(cv.width)) want *= 1.5f;  // nearly full: catch up before a backlog forms
    // ring pressure (smoothed): more than 2 % of the finishing envs one episode from running dry
    float taken = __uint_as_float(cv.ctl[CV_EMA_TAKEN]), low2 = __uint_as_float(cv.ctl[CV_EMA_LOW2]);
    float press = fmaxf(__uint_as_float(cv.ctl[CV_PRESS]), 1.f);
    taken += (float(cv.ctl[CV_TAKEN]) - taken) * 0.125f;
    low2 += (float(cv.ctl[CV_LOW2]) - low2) * 0.125f;
    press = low2 > 0.02f * taken + 1e-3f ? fminf(8.f, press * 1.25f) : fmaxf(1.f, press * 0.95f);
    cv.ctl[CV_EMA_TAKEN] = __float_as_uint(taken);
    cv.ctl[CV_EMA_LOW2] = __float_as_uint(low2);
    cv.ctl[CV_PRESS] = __float_as_uint(press);
    cv.ctl[CV_TAKEN] = 0; cv.ctl[CV_LOW2] = 0;
    want = fmaxf(float(s_min), fminf(float(s_max), ceilf(want * press)));
    cv.ctl[CV_WANT] = __float_as_uint(want);
    const int s0 = backlog ? 0 : min(early, int(want) / 2);
    cv.ctl[CV_ACTIVE_EARLY] = s0 > 0 ? min(pending, uint32_t(lanes)) : 0u;
    cv.ctl[CV_SLICE_EARLY] = uint32_t(s0);
    return;
  }
  // phase 1: what is left of this step's ticks, spread over the entries that run now
  const uint32_t active = min(pending, uint32_t(max(lanes, block)));
  const float want = __uint_as_float(cv.ctl[CV_WANT]);
  const float done0 = float(cv.ctl[CV_ACTIVE_EARLY]) * float(cv.ctl[CV_SLICE_EARLY]);
  const float all = float(min(pending, uint32_t(cv.width)));  // the entries `want` was computed for
  int slice = int(ceilf((want * all - done0) / fmaxf(float(active), 1.f)));
  slice = max(s_min, min(s_max, slice));
  if (backlog) slice = nsettle;
  cv.ctl[CV_ACTIVE] = active;
  cv.ctl[CV_SLICE] = uint32_t(slice);
}

// One slice of the conveyor: entry tail + j advances by ctl[CV_SLICE] settle ticks; an entry that
// reaches the end of its settle stores the episode's slot and retires.
template <bool kEM>
__global__ void __launch_bounds__(256, 1)
k_settle_slice(const __grid_constant__ KernelArgs A, const Conveyor cv, int early, unsigned long long* stamps) {
  const DeviceView& D = A.D;
  const int n = D.n;
  const int active = int(cv.ctl[early ? CV_ACTIVE_EARLY : CV_ACTIVE]);
  if (blockIdx.x * blockDim.x >= active) return;  // uniform over the block
  if (threadIdx.x == 0) stamp_begin(stamps);
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = j < active;
  const uint32_t idx = cv.ctl[CV_TAIL] + uint32_t(live ? j : active - 1);
  const uint32_t pos = idx & cv.cap_mask;
  const int span = int(cv.ctl[early ? CV_SLICE_EARLY : CV_SLICE]);
  const int env = cv.fifo[2 * pos];
  const uint32_t epoch = uint32_t(cv.fifo[2 * pos + 1]);
  const int t0 = cv.tick[pos];
  bool need = live && t0 != CV_DONE;
  // stale (the env went past that episode on the urgent path) or already stored by a duplicate
  if (need && (epoch <= D.reset_count[env] || slot_ready(D, env, epoch))) {
    cv.tick[pos] = CV_DONE;
    need = false;
  }
  const int nsettle = settle_length(A.C);
  const int col = int(idx % uint32_t(cv.width));
  EnvState<float> st;
  ContactState<float> cs;
  float tau_m[12], tau_s[12];
#pragma unroll
  for (int i = 0; i < 12; i++) { tau_m[i] = 0.f; tau_s[i] = 0.f; }
  fresh_state(A, st, cs);
  if (need && t0 > 0) wip_load(cv, col, st, cs);
  const float mu = episode_mu(A.C, uint64_t(A.C.gid0 + env), epoch);
  const int t1 = need ? min(t0 + span, nsettle) : 0;
  extern __shared__ __align__(16) float qs_smem[];
  const StepScratch scr{qs_smem, QS_BLOCK, int(threadIdx.x)};
  settle_ticks<kEM>(A, uint64_t(A.C.gid0 + env), epoch, st, cs, mu, t0, t1, span, tau_m, tau_s, scr, cv.model, cv.width, col);
  if (threadIdx.x == 0) stamp_end(stamps);   // (the block's ticks are over: settle_ticks ends on a barrier-matched loop)
  if (!need) return;
  {  // work counters of the bench's flop model, one atomic per warp
    const unsigned m = __activemask();
    const unsigned a = __reduce_add_sync(m, unsigned(t1 - t0)), b = __reduce_add_sync(m, unsigned(cs.work_contacts));
    const unsigned c = __reduce_add_sync(m, unsigned(cs.work_row_iters));
    if ((threadIdx.x & 31) == __ffs(m) - 1) {
      atomicAdd(cv.work + 0, (unsigned long long)a);
      atomicAdd(cv.work + 1, (unsigned long long)b);
      atomicAdd(cv.work + 2, (unsigned long long)c);
    }
  }
  if (t1 == nsettle) {
    slot_store(D, env, st, cs, tau_m, tau_s, mu, epoch, A.SC.dt);
    cv.tick[pos] = CV_DONE;
  } else {
    wip_store(cv, col, st, cs);
    cv.tick[pos] = t1;
  }
}

__global__ void k_compact(const uint8_t* __restrict__ mask, int n, int* __restrict__ list) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && mask[i]) list[atomicAdd(list + n, 1)] = i;
}
