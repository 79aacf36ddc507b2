// qs_kernels.cu -- sm_100a kernels and the C ABI (include/qs_b200.h) of the
// batched Go1(+PEA) simulator.  One env per thread: the whole control step
// (action map -> [PD + PEA torque -> floating-base dynamics -> contact PGS ->
// integration] x action_repeat -> task / reward / done -> observation) runs out
// of registers; HBM is touched once per control step through SoA arrays
// ([component][env], coalesced).  No tensor cores: per-env matrices are <= 6x6.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "qs_env.cuh"
#include "qs_model_host.h"

using namespace qs;

// ============================================================================ args
struct KernelArgs {
  DeviceView D;
  EnvCfg C;
  RobotConst RC;
  ModelConstT<float> M;
  ModelLegPairsT<float> M2;  // M's leg tables for the leg pairs (packed per-leg passes of the tick, qs_packed.cuh)
  SolverConst SC;
  double time_step_d, max_time_d;
};
static_assert(sizeof(KernelArgs) <= 3600, "kernel parameter space (4 KB) also holds StepIO / Conveyor");

static thread_local std::string g_err;
static std::atomic<int64_t> g_launches{0};

static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return fail(QS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
  } while (0)

// ============================================================================ kernels
#include "qs_step_kernels.cuh"

// -------------------------------------------------------------------- observe / state I/O
__global__ void k_observe(const __grid_constant__ KernelArgs A, float* __restrict__ obs, int with_noise) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  if (env >= D.n) return;
  EnvState<float> st;
  ContactState<float> cs;
  load_state(D, env, st, cs, A.SC.dt);
  float Rb[9], rpy[3], ts[QS_TASK_DIM], o[QS_MAX_OBS];
  quat_to_R(st.quat, Rb);
  rpy_from_quat(st.quat, rpy);
#pragma unroll
  for (int i = 0; i < TS_END_ALL; i++) ts[i] = i < task_slots(A.C.task) ? D.task[i * D.n + env] : 0.f;
#pragma unroll
  for (int i = 0; i < QS_MAX_OBS; i++) o[i] = 0.f;
  observe(st, cs, ts, rpy, Rb, A.C.obs_mode, A.C.task, o);
  store_obs(obs + size_t(env) * A.C.obs_dim, o, A.C, A.RC, uint64_t(A.C.gid0 + env), D.reset_count[env],
            uint32_t(D.env_steps[env]) + 0x40000000u, with_noise != 0);
}

__global__ void k_set_state(DeviceView D, const float* __restrict__ src) {  // [N,37] -> SoA
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D.n * QS_STATE_DIM) return;
  const int env = i / QS_STATE_DIM, c = i % QS_STATE_DIM;
  D.state[c * D.n + env] = src[i];
  if (c == 0) {  // a teleported robot has no contact history
    D.contact[env] = 0;
    for (int k = 0; k < 4; k++) D.foot_force[k * D.n + env] = 0.f;
  }
}
__global__ void k_get_state(DeviceView D, float* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D.n * QS_STATE_DIM) return;
  const int env = i / QS_STATE_DIM, c = i % QS_STATE_DIM;
  dst[i] = D.state[c * D.n + env];
}

// -------------------------------------------------------------------- per-env masses written by the caller
__global__ void k_apply_masses(DeviceView D) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= D.n) return;
  float raw[8], em[EM_ROWS];
  for (int i = 0; i < 8; i++) raw[i] = D.mass_draw[size_t(i) * D.n + env];
  model_from_masses(raw, em);
  for (int i = 0; i < EM_ROWS; i++) D.model[size_t(i) * D.n + env] = em[i];
}

// -------------------------------------------------------------------- debug ticks (fp32 product / fp64 check)
template <typename T> struct DebugArgs {
  DeviceView D;
  ModelConstT<T> M;
  ModelLegPairsT<T> M2;
  SolverConst SC;
  int mass_randomizer;
  ExtForce ext;   // the attached push buffer (ext.ticks == nullptr: none); counted down by n_ticks like a step
};
template <typename T>
__global__ void __launch_bounds__(64)
k_debug_ticks(const __grid_constant__ DebugArgs<T> A, const float* __restrict__ tau, int n_ticks) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceView& D = A.D;
  if (env >= D.n) return;
  EnvState<float> sf;
  ContactState<float> cf;
  load_state(D, env, sf, cf, A.SC.dt);
  EnvState<T> st;
  ContactState<T> cs;
#pragma unroll
  for (int i = 0; i < 3; i++) { st.pos[i] = sf.pos[i]; st.vlin[i] = sf.vlin[i]; st.vang[i] = sf.vang[i]; }
#pragma unroll
  for (int i = 0; i < 4; i++) { st.quat[i] = sf.quat[i]; cs.lam_n[i] = cf.lam_n[i]; }
#pragma unroll
  for (int i = 0; i < 12; i++) { st.q[i] = sf.q[i]; st.qd[i] = sf.qd[i]; }
  cs.mask = cf.mask; cs.invalid = cf.invalid; cs.work_contacts = 0; cs.work_row_iters = 0;
  T t12[12];
#pragma unroll
  for (int i = 0; i < 12; i++) t12[i] = T(tau[size_t(env) * 12 + i]);
  const T mu = T(D.mu[env]);
  extern __shared__ __align__(16) unsigned char qs_smem_raw[];
  const Scratch<T> scr{reinterpret_cast<T*>(qs_smem_raw), int(blockDim.x), int(threadIdx.x)};
  const ExtPush pf = A.ext.ticks ? ext_push(A.ext, env, D.n) : ExtPush{};
  ExtWrench<T> w;
#pragma unroll
  for (int i = 0; i < 3; i++) { w.f[i] = T(pf.w.f[i]); w.p[i] = T(pf.w.p[i]); }
  for (int t = 0; t < n_ticks; t++)
    {
    const EnvModelRef em{A.mass_randomizer ? D.model : nullptr, D.n, env};
    const ExtWrench<T>* ext = t < pf.n ? &w : nullptr;
    if (physics_tick<T, true, 0, true, true>(st, t12, mu, cs, A.M, A.SC, true, scr, em, &A.M2, ext)) { T dl[12]; physics_tick_general<T, true, true>(st, t12, mu, cs, A.M, A.SC, em, dl, 1, ext); }
  }
  if (pf.n > 0) A.ext.ticks[env] = pf.n - min(pf.n, n_ticks);
#pragma unroll
  for (int i = 0; i < 3; i++) { sf.pos[i] = float(st.pos[i]); sf.vlin[i] = float(st.vlin[i]); sf.vang[i] = float(st.vang[i]); }
#pragma unroll
  for (int i = 0; i < 4; i++) { sf.quat[i] = float(st.quat[i]); cf.lam_n[i] = float(cs.lam_n[i]); }
#pragma unroll
  for (int i = 0; i < 12; i++) { sf.q[i] = float(st.q[i]); sf.qd[i] = float(st.qd[i]); }
  cf.mask = cs.mask; cf.invalid = cs.invalid;
  store_state(D, env, sf, cf, A.SC.dt);
}

// -------------------------------------------------------------------- push countdown (qs_set_external_force)
// After a step of `consumed` ticks: n -= min(n, consumed), and n = 0 where `ended` is set (the step's done flags under
// auto_reset: a push never carries into the next episode; the mask of a reset with consumed = 0).  ended == nullptr:
// no env ended.  consumed < 0: every count goes to 0 (a reset of every env).
__global__ void k_ext_countdown(int32_t* __restrict__ ticks, const uint8_t* __restrict__ ended, int consumed, int n) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  const int32_t c = ticks[env];
  if (consumed < 0 || (ended && ended[env])) { if (c != 0) ticks[env] = 0; }
  else if (c > 0) ticks[env] = c - min(c, consumed);
}

// -------------------------------------------------------------------- K3: analytic utilities
__global__ void k_action_to_command(const __grid_constant__ RobotConst RC, int control_mode, int action_mode,
                                    int adim, const float* __restrict__ a, float* __restrict__ cmd, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float act[12], a12[12], c[12];
#pragma unroll
  for (int j = 0; j < 12; j++) act[j] = j < adim ? a[size_t(i) * adim + j] : 0.f;
  expand_action(action_mode, control_mode == QS_CTRL_CARTESIAN_PD ? 1 : 0, act, a12);
  action12_to_command(RC, control_mode, a12, c);
#pragma unroll
  for (int j = 0; j < 12; j++) cmd[size_t(i) * 12 + j] = c[j];
}

struct TorqueArgs {
  float kp[12], kd[12], tau_max[12], spring[9];
  int has_spring, torque_mode;
};
__global__ void k_pd_pea(const __grid_constant__ TorqueArgs T, const float* __restrict__ cmd,
                         const float* __restrict__ q, const float* __restrict__ qd, float* __restrict__ tau_m,
                         float* __restrict__ tau_s, int n) {
  // one thread per (env, leg)
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 4) return;
  const int leg = i & 3;
  const size_t base = size_t(i >> 2) * 12 + 3 * leg;
  float ql[3], qdl[3];
#pragma unroll
  for (int j = 0; j < 3; j++) { ql[j] = q[base + j]; qdl[j] = qd[base + j]; }
#pragma unroll
  for (int j = 0; j < 3; j++)
    tau_m[base + j] = pd_torque1(T.kp[3 * leg + j], T.kd[3 * leg + j], T.tau_max[3 * leg + j], cmd[base + j], ql[j],
                                 qdl[j], T.torque_mode != 0);
  if (tau_s) {
    float ts3[3] = {0.f, 0.f, 0.f};
    if (T.has_spring) spring_torque_leg(leg, T.spring, T.spring + 3, T.spring + 6, ql, qdl, ts3);
#pragma unroll
    for (int j = 0; j < 3; j++) tau_s[base + j] = ts3[j];
  }
}

__global__ void k_fk(const float* __restrict__ q, const float* __restrict__ qd, float* __restrict__ pos,
                     float* __restrict__ jac, float* __restrict__ vel, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 4) return;
  const int leg = i & 3;
  const size_t base = size_t(i >> 2) * 12 + 3 * leg;
  float ql[3] = {q[base], q[base + 1], q[base + 2]}, p[3], J[9];
  fk_jacobian(ql, leg, p, J);
#pragma unroll
  for (int j = 0; j < 3; j++) pos[base + j] = p[j];
  if (jac) {
#pragma unroll
    for (int j = 0; j < 9; j++) jac[size_t(i) * 9 + j] = J[j];
  }
  if (vel && qd) {
    const float d0 = qd[base], d1 = qd[base + 1], d2 = qd[base + 2];
#pragma unroll
    for (int a = 0; a < 3; a++) vel[base + a] = J[3 * a] * d0 + J[3 * a + 1] * d1 + J[3 * a + 2] * d2;
  }
}

__global__ void k_ik(const float* __restrict__ xyz, float* __restrict__ q, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 4) return;
  const int leg = i & 3;
  const size_t base = size_t(i >> 2) * 12 + 3 * leg;
  float x[3] = {xyz[base], xyz[base + 1], xyz[base + 2]}, o[3];
  leg_ik(x, leg, o);
#pragma unroll
  for (int j = 0; j < 3; j++) q[base + j] = o[j];
}

// -------------------------------------------------------------------- K4: Hopf CPG + impedance law
// The oscillator state is kept in float64: the reference starts every phase exactly at 0 / +-pi,
// i.e. ON the swing/stance switch `sin(theta) > 0` (hopf_network.py:150-153), where a float32 pi
// would flip the branch.  It is ~60 FLOP per env and tick; the torque law below is fp32.
struct CpgArgs {
  double p[9], phi[16];
  float gains[8], foot_y;
};
// q / qd element (env i, joint j) at q[i * q_si + j * q_sj]: [N,12] row-major (12, 1) or the env's own SoA rows (1, N)
__global__ void k_cpg(const __grid_constant__ CpgArgs P, double* __restrict__ X, const float* __restrict__ q,
                      const float* __restrict__ qd, float* __restrict__ xs_o, float* __restrict__ zs_o,
                      float* __restrict__ tau, int n, int q_si, int q_sj) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double mu = P.p[0], om_sw = P.p[1], om_st = P.p[2], coup = P.p[3], dt = P.p[4], dstep = P.p[5],
               height = P.p[6], gc = P.p[7], gp = P.p[8];
  double r0[4], th0[4], r1[4], th1[4];
  float xs[4], zs[4];
#pragma unroll
  for (int k = 0; k < 4; k++) { r0[k] = X[size_t(i) * 8 + k]; th0[k] = X[size_t(i) * 8 + 4 + k]; }
  // hopf_network.py:137-173
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const double rd = 50.0 * (mu - r0[k] * r0[k]) * r0[k];
    double thd = sin(th0[k]) > 0.0 ? om_sw : om_st;
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (j != k) thd += r0[j] * coup * sin(th0[j] - th0[k] - P.phi[4 * k + j]);
    r1[k] = r0[k] + dt * rd;
    double th = fmod(th0[k] + dt * thd, 2 * QS_PI);
    if (th < 0.0) th += 2 * QS_PI;  // numpy % is a floored modulo
    th1[k] = th;
  }
#pragma unroll
  for (int k = 0; k < 4; k++) {
    X[size_t(i) * 8 + k] = r1[k];
    X[size_t(i) * 8 + 4 + k] = th1[k];
    double s, c;
    sincos(th1[k], &s, &c);
    xs[k] = float(-dstep * r1[k] * c);                              // hopf_network.py:126-133
    zs[k] = float(s > 0.0 ? -height + gc * s : -height + gp * s);
    if (xs_o) xs_o[size_t(i) * 4 + k] = xs[k];
    if (zs_o) zs_o[size_t(i) * 4 + k] = zs[k];
  }
  if (!tau) return;
  // hopf_network.py:241-289: joint PD on IK(xyz_d) + J^T (-Kp (x - x_d) - Kd J qd)
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const float xyz_d[3] = {xs[k], side_sign(k) * P.foot_y, zs[k]};
    float qdes[3], ql[3], qdl[3], J[9], p[3];
    leg_ik(xyz_d, k, qdes);
#pragma unroll
    for (int j = 0; j < 3; j++) { ql[j] = q[size_t(i) * q_si + size_t(3 * k + j) * q_sj]; qdl[j] = qd[size_t(i) * q_si + size_t(3 * k + j) * q_sj]; }
    fk_jacobian(ql, k, p, J);
    float F[3];
#pragma unroll
    for (int a = 0; a < 3; a++) {
      const float dx = J[3 * a] * qdl[0] + J[3 * a + 1] * qdl[1] + J[3 * a + 2] * qdl[2];
      F[a] = -P.gains[6] * (p[a] - xyz_d[a]) - P.gains[7] * dx;
    }
#pragma unroll
    for (int j = 0; j < 3; j++) {
      float t = -P.gains[j] * (ql[j] - qdes[j]) - P.gains[3 + j] * qdl[j];
      t += J[j] * F[0] + J[3 + j] * F[1] + J[6 + j] * F[2];
      tau[size_t(i) * 12 + 3 * k + j] = t;
    }
  }
}

// -------------------------------------------------------------------- K5: rollout statistics
// block reduce with warp shuffles, one atomic per block and statistic
__global__ void k_stats(DeviceView D, float* __restrict__ out) {
  __shared__ float sm[QS_STATS_DIM][8];
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float v[QS_STATS_DIM];
#pragma unroll
  for (int i = 0; i < QS_STATS_DIM; i++) v[i] = 0.f;
  if (env < D.n) {
#pragma unroll
    for (int i = 0; i < 12; i++) v[1 + i] = D.stats[i * D.n + env];
    v[0] = 1.f;
  }
  // rows 3 and 6 of v (stats rows 2, 5) are maxima, everything else sums
#pragma unroll
  for (int i = 0; i < QS_STATS_DIM; i++) {
    const bool is_max = (i == 3 || i == 6);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float t = __shfl_xor_sync(0xffffffffu, v[i], o);
      v[i] = is_max ? fmaxf(v[i], t) : v[i] + t;
    }
    if (lane == 0) sm[i][warp] = v[i];
  }
  __syncthreads();
  if (threadIdx.x < QS_STATS_DIM) {
    const int i = threadIdx.x;
    const bool is_max = (i == 3 || i == 6);
    float a = sm[i][0];
    for (int w = 1; w < (blockDim.x >> 5); w++) a = is_max ? fmaxf(a, sm[i][w]) : a + sm[i][w];
    if (is_max) atomicMax(reinterpret_cast<int*>(out + i), __float_as_int(fmaxf(a, 0.f)));  // non-negative floats order as ints
    else atomicAdd(out + i, a);
  }
}

// ============================================================================ host side
struct qs_env {
  qs_config cfg;
  int n, device;
  KernelArgs args;
  ModelConstT<double> model_d;
  void* pool;       // one allocation backing every SoA array
  size_t pool_bytes;
  int* lists;          // slow (n + 1) | reset (n + 1) | contact (n + 1) | flight (n + 1) | urgent (2 n) | conveyor fifo, tick, wip, control words
  int *slow_list, *reset_list, *contact_list, *flight_list;
  Conveyor cv;
  int wave_blocks;     // settle blocks resident at once (SMs x 2)
  int slice_min, slice_max, slice_early;
  int finish_pdl;  // device-buffer steps: k_finish next to k_step_slow (programmatic dependent launches)
  int flight_cap;      // envs per flight launch (k_pre sends the overflow to the contact kernel)
  int slow_spread;     // envs per warp in k_step_slow (power of two)
  cudaStream_t bg;     // the conveyor's slices run here, next to k_step_slow on the caller's stream
  cudaStream_t copy;   // qs_step_host: results go to the host while the slice is still running
  cudaEvent_t ev_results, ev_copied;
  uint32_t* host_urgent;  // pinned: urgent settles of the last step (their obs rows are written after the early copy)
  cudaEvent_t ev_fork, ev_join;
  float* dev_actions;  // staging for qs_step_host
  float* dev_obs;
  float* dev_reward;
  uint8_t* dev_done;
  uint8_t* dev_trunc;
  // qs_step_host: the results of the envs the general solver finishes last travel in a compact side buffer
  float* dev_late;     // [4 + late_cap * (O + 4)]: count | rows of (env, reward, done, truncated, obs[O])
  float* host_late;    // pinned twin
  int late_cap;
  cudaEvent_t ev_late;
  float* term_obs;     // caller-owned, optional (qs_set_terminal_obs)
  float* dev_demo;     // demonstration actions of the *_DEMO tasks (qs_set_demo)
  SubstepTrace trace;  // qs_set_substep_trace: caller-owned rows, column map in the pool (trace.buf == nullptr: off)
  ExtForce ext;        // qs_set_external_force: caller-owned wrench and tick counts (ext.ticks == nullptr: off)
  bool was_reset;
  // CUDA-event ring around k_step launches (roofline timing of the dominant kernel)
  static constexpr int kRing = 512;
  cudaEvent_t ev0[kRing], ev1[kRing];   // around k_step + k_step_contact, on the caller's stream
  cudaEvent_t ev4[kRing], ev5[kRing];   // around the early settle slice, on the second stream
  // CUDA graph of one step (qs_step): captured once per set of output buffers and timing-ring slot on the library's own
  // stream `main`, relaunched per step; the caller's stream is joined with two events.  Every data-dependent count of
  // the step lives on the device, so the graph never changes.
  static constexpr int kGraphSlots = 16, kGraphKeys = 4;
  struct GraphKey { float* obs; float* reward; uint8_t* done; uint8_t* trunc; float* term_obs; cudaGraphExec_t exec[kGraphSlots]; };
  GraphKey gkeys[kGraphKeys];
  int n_gkeys;
  int ring;            // timing ring in use: kRing (direct launches) or kGraphSlots (graph launches)
  bool use_graph;
  cudaStream_t main;   // the graph is launched here
  cudaEvent_t ev_in, ev_out;
  float* act_buf;      // the graph's action input [N, A]: the caller's actions are copied here first
  int launches_per_step;
  cudaEvent_t ev_fork0, ev_early_done;
  unsigned long long* stamps;   // [kRing][4] device: per step {late slice start, end, general solver start, end} (globaltimer ns)
  bool ev_ready;
  int64_t n_steps;
};

static inline unsigned grid_for(int n, int block) { return unsigned((n + block - 1) / block); }
// f(em, trace, push) for every instantiation of the tick kernels, as std::bool_constant arguments
template <typename F> static void for_each_tick_variant(F f) {
  using T = std::true_type;
  using N = std::false_type;
  f(N{}, N{}, N{}); f(T{}, N{}, N{}); f(N{}, T{}, N{}); f(T{}, T{}, N{});
  f(N{}, N{}, T{}); f(T{}, N{}, T{}); f(N{}, T{}, T{}); f(T{}, T{}, T{});
}
static int block_of(qs_handle) { return QS_BLOCK; }
static size_t smem_of(int block) { return size_t(block) * QS_TICK_SCRATCH * sizeof(float); }

extern "C" {

const char* qs_last_error(void) { return g_err.c_str(); }
int64_t qs_launch_count(void) { return g_launches.load(); }

int qs_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

void qs_default_config(qs_config* c) {
  std::memset(c, 0, sizeof(*c));
  c->enable_springs = 0;                       // quadruped_gym_env.py:63
  c->control_mode = QS_CTRL_PD;                // :57
  c->action_mode = QS_ACT_SYMMETRIC;           // :60
  c->task = QS_TASK_NO_TASK;                   // :58
  c->obs_mode = QS_OBS_ENCODER;                // :59
  c->action_repeat = 10;                       // :56
  c->is_rl_interface = 1;                      // :54
  c->enable_action_filter = 0;                 // :65
  c->ground_randomizer = 1;                    // :66
  c->settling_steps = 2500;                    // :115
  c->enable_noise = 1;
  c->auto_reset = 0;
  c->num_iterations = 0;
  c->enable_limits = 1;
  c->body_contact_response = 1;
  c->block_size = 0;
  c->seed = 0;
  c->env_id_offset = 0;
  c->time_step = 0.001;                        // :55
  c->max_episode_time = 10.0;                  // :35
  c->gravity_z = -9.8f;                        // :309
  c->mu_ground = 1.0f;
  c->contact_erp = 0.08f;
  c->limit_erp = 0.2f;
  c->linear_slop = 1e-5f;
  c->warmstart = 0.1f;
  c->residual_threshold = 1e-7f;
  c->max_coord_vel = 30.1f;                    // quadruped.py:678-683
  c->breaking_threshold = 0.02f;
  c->rand_leg_mass_err = 0.1f;                 // env_randomizer.py:5-14
  c->rand_payload_max = 1.0f;
  c->rand_payload_pos[0] = 0.1f; c->rand_payload_pos[1] = 0.0f; c->rand_payload_pos[2] = 0.1f;
  c->rand_spring_err = 0.1f;
  c->self_collision = 1;                       // quadruped.py:530-543
}

static int check_config(const qs_config* c) {
  if (!c) return fail(QS_ERR_ARG, "config is NULL");
  if (c->control_mode < 0 || c->control_mode > 2) return fail(QS_ERR_ARG, "unknown motor control mode");
  if (c->action_mode < 0 || c->action_mode > 2) return fail(QS_ERR_ARG, "unknown action space mode");
  if (c->task < 0 || c->task > QS_TASK_CONTINUOUS_JUMPING_FORWARD_DEMO) return fail(QS_ERR_ARG, "unknown task");
  if (c->block_size != 0 && c->block_size != QS_BLOCK) return fail(QS_ERR_ARG, "block_size is fixed at 128 (0 = default)");
  if (c->landing_mode < 0 || c->landing_mode > 5) return fail(QS_ERR_ARG, "unknown landing_mode");
  if (c->landing_mode >= 4 && c->action_mode != QS_ACT_SYMMETRIC)
    return fail(QS_ERR_ARG, "the backflip landing controllers script a SYMMETRIC action (landing_wrapper_backflip.py:21)");
  if (c->landing_mode == 3 && !(c->task >= QS_TASK_CONTINUOUS_JUMPING_FORWARD && c->task <= QS_TASK_CONTINUOUS_JUMPING_FORWARD_PPO))
    return fail(QS_ERR_ARG, "LandingWrapperContinuous needs a continuous-jumping task (task.get_jumping)");
  if (c->landing_mode && (c->control_mode == QS_CTRL_TORQUE || !c->is_rl_interface))
    return fail(QS_ERR_ARG, "landing controllers need the RL interface with PD or CARTESIAN_PD control");
  if (c->rest_mode && (c->control_mode == QS_CTRL_TORQUE || !c->is_rl_interface))
    return fail(QS_ERR_ARG, "the go-to-rest controller needs the RL interface with PD or CARTESIAN_PD control");
  if (c->mass_randomizer && (!(c->rand_leg_mass_err >= 0.f && c->rand_leg_mass_err < 1.f) || !(c->rand_payload_max >= 0.f) ||
                             c->rand_payload_max > 5.f))
    return fail(QS_ERR_ARG, "mass randomizer ranges out of bounds");
  if (!(c->rand_spring_err >= 0.f && c->rand_spring_err < 1.f)) return fail(QS_ERR_ARG, "rand_spring_err out of range");
  if (c->obs_mode < 0 || c->obs_mode > QS_OBS_PPO_CONTINUOUS_JUMPING_FORWARD) return fail(QS_ERR_ARG, "unknown observation space mode");
  if (c->action_repeat < 1 || c->action_repeat > 1000) return fail(QS_ERR_ARG, "action_repeat out of range");
  if (c->control_mode == QS_CTRL_TORQUE && c->is_rl_interface)  // quadruped_gym_env.py:167-168
    return fail(QS_ERR_ARG, "the motor control mode TORQUE not implemented yet for RL Gym interface.");
  if (!(c->time_step > 0)) return fail(QS_ERR_ARG, "time_step must be positive");
  return QS_OK;
}

int qs_config_obs_dim(const qs_config* c) { return c ? host::obs_dim_of(c->obs_mode) : QS_ERR_ARG; }
int qs_config_action_dim(const qs_config* c) { return c ? host::action_dim_of(c->is_rl_interface, c->action_mode) : QS_ERR_ARG; }

int qs_obs_noise_std(const qs_config* c, float* out) {
  if (int e = check_config(c)) return e;
  if (!out) return fail(QS_ERR_ARG, "out is NULL");
  RobotConst R;
  host::build_robot(*c, R);
  std::memcpy(out, R.obs_noise, sizeof(float) * QS_MAX_OBS);
  return QS_OK;
}

int qs_create(const qs_config* cfg, int n_envs, int device, qs_handle* out) {
  if (int e = check_config(cfg)) return e;
  if (!out) return fail(QS_ERR_ARG, "out handle is NULL");
  if (n_envs <= 0) return fail(QS_ERR_ARG, "n_envs must be positive");
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(QS_ERR_CUDA, "no such CUDA device (this library has no CPU fallback)");
  CUDA_TRY(cudaSetDevice(device));
  qs_env* h = new (std::nothrow) qs_env();
  if (!h) return fail(QS_ERR_STATE, "out of host memory");
  std::memset(static_cast<void*>(h), 0, sizeof(*h));
  h->cfg = *cfg;
  h->n = n_envs;
  h->device = device;
  KernelArgs& A = h->args;
  host::build_robot(*cfg, A.RC);
  host::build_model<float>(A.M, cfg->breaking_threshold);
  make_leg_pairs(A.M, A.M2);
  host::build_model<double>(h->model_d, cfg->breaking_threshold);
  A.SC.dt = float(cfg->time_step);
  A.SC.gravity_z = cfg->gravity_z;
  A.SC.contact_erp = cfg->contact_erp;
  A.SC.limit_erp = cfg->limit_erp;
  A.SC.linear_slop = cfg->linear_slop;
  A.SC.warmstart = cfg->warmstart;
  A.SC.residual_threshold = cfg->residual_threshold;
  A.SC.max_coord_vel = cfg->max_coord_vel;
  A.SC.mu_link = 1.0f;  // quadruped.py:670-676
  A.SC.num_iterations = cfg->num_iterations > 0 ? cfg->num_iterations : 300 / cfg->action_repeat;  // quadruped_gym_env.py:113
  A.SC.enable_limits = cfg->enable_limits;
  A.SC.body_response = cfg->body_contact_response;
  A.SC.self_collision = cfg->self_collision;
  if (const char* v = std::getenv("QS_SELF_COLLISION")) A.SC.self_collision = std::atoi(v);  // (experiments)
  A.time_step_d = cfg->time_step;
  A.max_time_d = cfg->max_episode_time;
  EnvCfg& C = A.C;
  C.enable_springs = cfg->enable_springs; C.control_mode = cfg->control_mode; C.action_mode = cfg->action_mode;
  C.task = cfg->task; C.obs_mode = cfg->obs_mode; C.action_repeat = cfg->action_repeat;
  C.is_rl = cfg->is_rl_interface; C.enable_filter = cfg->enable_action_filter; C.enable_noise = cfg->enable_noise;
  C.obs_dim = host::obs_dim_of(cfg->obs_mode);
  C.action_dim = host::action_dim_of(cfg->is_rl_interface, cfg->action_mode);
  C.settling_steps = cfg->settling_steps; C.ground_randomizer = cfg->ground_randomizer; C.auto_reset = cfg->auto_reset;
  C.landing_mode = cfg->landing_mode; C.spring_randomizer = cfg->spring_randomizer && cfg->enable_springs;
  C.rest_mode = cfg->rest_mode != 0;
  C.mass_randomizer = cfg->mass_randomizer != 0;
  C.leg_mass_err = cfg->rand_leg_mass_err; C.payload_max = cfg->rand_payload_max; C.spring_err = cfg->rand_spring_err;
  for (int i = 0; i < 3; i++) C.payload_pos[i] = cfg->rand_payload_pos[i];
  C.max_episode_time = float(cfg->max_episode_time); C.mu_ground = cfg->mu_ground;
  C.seed = cfg->seed; C.gid0 = cfg->env_id_offset;
  {  // RobotConst::settle_cmd = settle_command() as the device evaluates it
    float* d_cmd = nullptr;
    cudaError_t ec = cudaMalloc(&d_cmd, 12 * sizeof(float));
    if (ec == cudaSuccess) {
      k_settle_cmd<<<1, 1>>>(A, d_cmd);
      ec = cudaMemcpy(A.RC.settle_cmd, d_cmd, 12 * sizeof(float), cudaMemcpyDeviceToHost);
      cudaFree(d_cmd);
    }
    if (ec != cudaSuccess) { delete h; return fail(QS_ERR_CUDA, std::string("settle command: ") + cudaGetErrorString(ec)); }
  }

  // one pool for all SoA arrays (4-byte elements), 256 B aligned segments
  const size_t n = size_t(n_envs);
  const size_t rows = 37 + 12 + 12 + 12 + 12 + 9 + 1 + 4 + 1 + QS_TASK_DIM + 12 + 48 + 1 + 1 + 1 + QS_STATS_DIM + 1 + 3 + 12 + 1 + 1 + 1 + 2 + 1 + 14 + EM_ROWS + 8 + QS_SLOTS * (SLOT_ROWS + 1 + 1) + 1;
  // rows of one array are contiguous with stride n floats; each array starts 256 B aligned
  h->pool_bytes = rows * n * 4 + 64 * 256;
  cudaError_t e = cudaMalloc(&h->pool, h->pool_bytes);
  if (e != cudaSuccess) { delete h; return fail(QS_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
  cudaMemset(h->pool, 0, h->pool_bytes);
  char* p = static_cast<char*>(h->pool);
  auto carve = [&](size_t nrows) {
    void* r = p;
    size_t bytes = nrows * n * 4;
    bytes = ((bytes + 255) / 256) * 256;
    p += bytes;
    return r;
  };
  DeviceView& D = A.D;
  D.n = n_envs;
  D.state = (float*)carve(37); D.tau_motor = (float*)carve(12); D.tau_spring = (float*)carve(12);
  D.kp = (float*)carve(12); D.kd = (float*)carve(12); D.spring = (float*)carve(9); D.mu = (float*)carve(1);
  D.foot_force = (float*)carve(4); D.contact = (int32_t*)carve(1); D.task = (float*)carve(QS_TASK_DIM);
  D.last_action = (float*)carve(12); D.filt = (float*)carve(48); D.sim_steps = (int32_t*)carve(1);
  D.env_steps = (int32_t*)carve(1); D.ep_return = (float*)carve(1); D.stats = (float*)carve(QS_STATS_DIM);
  D.reset_count = (uint32_t*)carve(1);
  D.work = (uint32_t*)carve(3);
  D.cmd = (float*)carve(12); D.resume_tick = (int32_t*)carve(1);
  D.custom_gains = (uint8_t*)carve(1);
  D.land_mode = (int32_t*)carve(1); D.land_timer = (float*)carve(2);
  D.rest_active = (int32_t*)carve(1); D.rest = (float*)carve(14);
  D.model = (float*)carve(EM_ROWS); D.mass_draw = (float*)carve(8);
  D.slot = (float*)carve(QS_SLOTS * SLOT_ROWS); D.slot_contact = (int32_t*)carve(QS_SLOTS); D.slot_epoch = (uint32_t*)carve(QS_SLOTS);
  h->trace.col = (int32_t*)carve(1);
  if (size_t(p - static_cast<char*>(h->pool)) > h->pool_bytes) { cudaFree(h->pool); delete h; return fail(QS_ERR_STATE, "pool overflow"); }
  {
    // settle conveyor: window = one wave of settle blocks (2 per SM); the queue holds every ring entry
    // of every env several times over (duplicates after explicit resets)
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { cudaFree(h->pool); delete h; return fail(QS_ERR_CUDA, "cudaGetDeviceProperties"); }
    const int B = block_of(h);
    h->wave_blocks = prop.multiProcessorCount * std::max(1, 256 / B);
    Conveyor& cv = h->cv;
    cv.width = h->wave_blocks * B;
    size_t cap = 1024;
    // at least twice the slice window: two queue indices that share a position (a push dropped on a full queue keeps its
    // index) can then never be active in the same slice, whatever n
    while (cap < 4 * size_t(QS_SLOTS) * n || cap < 2 * size_t(cv.width)) cap <<= 1;
    cv.cap_mask = uint32_t(cap - 1);
    h->slice_min = 24;  // a settle never takes more than ~100 steps even when few episodes end (24 ticks hide behind the step's chain)
    h->slice_max = 1 << 20;  // no cap: the slice follows the demand
    h->flight_cap = h->wave_blocks * B;   // one wave of the flight kernel's blocks
    if (const char* v = std::getenv("QS_FLIGHT_CAP")) h->flight_cap = std::max(0, std::atoi(v));
    h->slice_early = 18;  // ticks of the early slice (round-2 sweep: 8 -> 1.443 ms per step, 12 -> 1.437, 16 -> 1.429, 20 -> 1.417, 24 -> 1.448, 32 -> 1.471)
    // envs per warp of the general solver.  Its duration is the longest env's chain, and lanes of a warp that take
    // different paths through it run one after the other: fewer envs per warp shorten it -- when there are idle SMs to put
    // the extra warps on (each of its blocks wants an SM of its own, see launch_conveyor).  With the GPU full (65536 envs)
    // 32 per warp is best (16: +11 % step time); at 4096 envs one env per warp takes the step from 0.89 to 0.70 ms.
    h->slow_spread = n_envs <= 8192 ? 1 : (n_envs <= 16384 ? 8 : 32);
    if (const char* v = std::getenv("QS_SLOW_SPREAD")) {
      const int k = std::atoi(v);
      if (k == 1 || k == 2 || k == 4 || k == 8 || k == 16 || k == 32) h->slow_spread = k;
    }
    h->finish_pdl = 1;
    if (const char* v = std::getenv("QS_FINISH_PDL")) h->finish_pdl = std::atoi(v) != 0;
    if (const char* v = std::getenv("QS_SETTLE_SLICE_EARLY")) h->slice_early = std::max(0, std::atoi(v));
    if (const char* v = std::getenv("QS_SETTLE_SLICE_MIN")) h->slice_min = std::max(1, std::atoi(v));
    if (const char* v = std::getenv("QS_SETTLE_SLICE_MAX")) h->slice_max = std::max(h->slice_min, std::atoi(v));
    const size_t w = size_t(cv.width);
    const size_t nints = 4 * (n + 1) + 2 * n + 2 * cap + cap + (WIP_ROWS + 1 + EM_ROWS) * w + CV_CTL_WORDS + 8;
    e = cudaMalloc(&h->lists, nints * sizeof(int));
    if (e != cudaSuccess) { cudaFree(h->pool); delete h; return fail(QS_ERR_CUDA, "cudaMalloc lists"); }
    cudaMemset(h->lists, 0, nints * sizeof(int));
    h->slow_list = h->lists;
    h->reset_list = h->slow_list + n + 1;
    h->contact_list = h->reset_list + n + 1;
    h->flight_list = h->contact_list + n + 1;
    cv.urgent_list = h->flight_list + n + 1;
    cv.fifo = cv.urgent_list + 2 * n;
    cv.tick = cv.fifo + 2 * cap;
    cv.wip = reinterpret_cast<float*>(cv.tick + cap);
    cv.wip_contact = reinterpret_cast<int*>(cv.wip + WIP_ROWS * w);
    cv.model = reinterpret_cast<float*>(cv.wip_contact + w);
    cv.ctl = reinterpret_cast<uint32_t*>(cv.model + EM_ROWS * w);
    cv.work = reinterpret_cast<unsigned long long*>(h->lists + ((size_t((cv.ctl + CV_CTL_WORDS) - reinterpret_cast<uint32_t*>(h->lists)) + 1) & ~size_t(1)));
    cudaMemset(cv.tick, 0xff, cap * sizeof(int));  // CV_DONE: nothing queued
    e = cudaStreamCreateWithFlags(&h->bg, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_results, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_copied, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMallocHost(&h->host_urgent, sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork0, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_early_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->main, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming);
    h->use_graph = true;
    if (const char* v = std::getenv("QS_GRAPH")) h->use_graph = std::atoi(v) != 0;
    h->ring = h->use_graph ? int(qs_env::kGraphSlots) : int(qs_env::kRing);
    if (e == cudaSuccess) e = cudaMalloc(&h->stamps, sizeof(unsigned long long) * 4 * qs_env::kRing);
    if (e == cudaSuccess) e = cudaMemset(h->stamps, 0, sizeof(unsigned long long) * 4 * qs_env::kRing);
    if (e != cudaSuccess) { cudaFree(h->pool); cudaFree(h->lists); delete h; return fail(QS_ERR_CUDA, "stream / event creation"); }
  }
  {
    const int max_smem = int(smem_of(256));
    // the tick kernels' eight instantiations <mass randomizer, substep trace, push>
    e = cudaSuccess;
    for_each_tick_variant([&](auto em, auto trace, auto push) {
      constexpr bool a = decltype(em)::value, b = decltype(trace)::value, c = decltype(push)::value;
      if (e == cudaSuccess) e = cudaFuncSetAttribute(k_step<a, b, c>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(k_step_contact<a, b, c>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    });
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_reset<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_reset<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_settle_urgent<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_settle_urgent<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_settle_slice<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_settle_slice<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_debug_ticks<double>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   int(64 * QS_TICK_SCRATCH * sizeof(double)));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_debug_ticks<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   int(64 * QS_TICK_SCRATCH * sizeof(float)));
    if (e != cudaSuccess) { cudaFree(h->pool); cudaFree(h->lists); delete h; return fail(QS_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e)); }
  }
  *out = h;
  return QS_OK;
}

static void drop_graphs(qs_handle h);

int qs_destroy(qs_handle h) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  cudaFree(h->pool);
  cudaFree(h->lists);
  if (h->dev_demo) cudaFree(h->dev_demo);
  cudaStreamDestroy(h->bg);
  cudaStreamDestroy(h->copy);
  cudaEventDestroy(h->ev_results);
  cudaEventDestroy(h->ev_copied);
  cudaFreeHost(h->host_urgent);
  cudaEventDestroy(h->ev_fork);
  cudaEventDestroy(h->ev_fork0);
  cudaEventDestroy(h->ev_join);
  cudaEventDestroy(h->ev_early_done);
  drop_graphs(h);
  cudaStreamDestroy(h->main);
  cudaEventDestroy(h->ev_in);
  cudaEventDestroy(h->ev_out);
  if (h->act_buf) cudaFree(h->act_buf);
  cudaFree(h->stamps);
  if (h->dev_actions) cudaFree(h->dev_actions);
  if (h->dev_obs) cudaFree(h->dev_obs);
  if (h->dev_reward) cudaFree(h->dev_reward);
  if (h->dev_done) cudaFree(h->dev_done);
  if (h->dev_late) { cudaFree(h->dev_late); cudaFreeHost(h->host_late); cudaEventDestroy(h->ev_late); }
  if (h->ev_ready)
    for (int i = 0; i < qs_env::kRing; i++) {
      cudaEventDestroy(h->ev0[i]); cudaEventDestroy(h->ev1[i]);
      cudaEventDestroy(h->ev4[i]); cudaEventDestroy(h->ev5[i]);
    }
  delete h;
  return QS_OK;
}

int qs_step_kernel_time(qs_handle h, int last_k, float* ms_sum) {
  // sum of the device durations of the last `last_k` k_step launches (CUDA events on the
  // launching stream; k_step + k_step_contact); the stream must have been synchronised by the caller
  if (!h || !ms_sum) return fail(QS_ERR_ARG, "NULL argument");
  if (last_k <= 0 || last_k > h->ring || last_k > h->n_steps) return fail(QS_ERR_ARG, "last_k out of range (qs_timing_window)");
  float tot = 0.f;
  for (int64_t i = h->n_steps - last_k; i < h->n_steps; i++) {
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0[i % h->ring], h->ev1[i % h->ring]));
    tot += ms;
  }
  *ms_sum = tot;
  return QS_OK;
}

int qs_settle_kernel_time(qs_handle h, int last_k, float* ms_sum) {
  // same for the k_settle_slice launches of the last `last_k` steps (events on the library's second stream)
  if (!h || !ms_sum) return fail(QS_ERR_ARG, "NULL argument");
  if (!h->cfg.auto_reset) return fail(QS_ERR_STATE, "no settle slices without auto_reset");
  if (last_k <= 0 || last_k > h->ring || last_k > h->n_steps) return fail(QS_ERR_ARG, "last_k out of range (qs_timing_window)");
  static unsigned long long host_st[4 * qs_env::kRing];
  CUDA_TRY(cudaMemcpy(host_st, h->stamps, sizeof(host_st), cudaMemcpyDeviceToHost));
  float tot = 0.f;
  for (int64_t i = h->n_steps - last_k; i < h->n_steps; i++) {
    float ms = 0.f;
    const unsigned long long* st = host_st + 4 * (i % h->ring);
    if (st[1] > st[0]) tot += float(double(st[1] - st[0]) * 1e-6);   // late slice: device-side stamps (it shares its stream)
    CUDA_TRY(cudaEventElapsedTime(&ms, h->ev4[i % h->ring], h->ev5[i % h->ring]));
    tot += ms;
  }
  *ms_sum = tot;
  return QS_OK;
}

int qs_slow_kernel_time(qs_handle h, int last_k, float* ms_sum) {
  // same for the k_step_slow launches (events on the caller's stream)
  if (!h || !ms_sum) return fail(QS_ERR_ARG, "NULL argument");
  if (last_k <= 0 || last_k > h->ring || last_k > h->n_steps) return fail(QS_ERR_ARG, "last_k out of range (qs_timing_window)");
  static unsigned long long host_st[4 * qs_env::kRing];
  CUDA_TRY(cudaMemcpy(host_st, h->stamps, sizeof(host_st), cudaMemcpyDeviceToHost));
  float tot = 0.f;
  for (int64_t i = h->n_steps - last_k; i < h->n_steps; i++) {
    const unsigned long long* st = host_st + 4 * (i % h->ring);
    if (st[3] > st[2]) tot += float(double(st[3] - st[2]) * 1e-6);
  }
  *ms_sum = tot;
  return QS_OK;
}

int64_t qs_step_count(qs_handle h) { return h ? h->n_steps : 0; }
int qs_timing_window(qs_handle h) { return h ? h->ring : QS_ERR_ARG; }

int qs_settle_work_counters(qs_handle h, uint64_t* out3, void* stream) {
  // totals of (settle ticks, foot-contact ticks, contact x PGS-sweep count) executed by k_settle_slice so far; synchronises
  if (!h || !out3) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  unsigned long long host[3];
  CUDA_TRY(cudaMemcpyAsync(host, h->cv.work, sizeof(host), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  for (int r = 0; r < 3; r++) out3[r] = host[r];
  return QS_OK;
}

int qs_work_counters(qs_handle h, uint64_t* out3, void* stream) {
  // totals over all envs of (ticks, contact-ticks, contact-sweeps) executed by k_step so far; synchronises
  if (!h || !out3) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t n = size_t(h->n);
  uint32_t* host = static_cast<uint32_t*>(std::malloc(3 * n * sizeof(uint32_t)));
  if (!host) return fail(QS_ERR_STATE, "out of host memory");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemcpyAsync(host, h->args.D.work, 3 * n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) { std::free(host); return fail(QS_ERR_CUDA, cudaGetErrorString(e)); }
  for (int r = 0; r < 3; r++) {
    uint64_t t = 0;
    for (size_t i = 0; i < n; i++) t += host[r * n + i];
    out3[r] = t;
  }
  std::free(host);
  return QS_OK;
}

int qs_debug_counters(qs_handle h, int32_t* out3, void* stream) {  // out3: 4 counters
  // {envs handed to the general solver, envs started on the urgent path (no settled slot was ready),
  // conveyor entries in flight, ticks of the last slice} as left by the last qs_step; synchronises
  if (!h || !out3) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemcpyAsync(out3 + 0, h->slow_list + h->n, sizeof(int), cudaMemcpyDeviceToHost, s));
  uint32_t ctl[CV_CTL_WORDS];
  CUDA_TRY(cudaMemcpyAsync(ctl, h->cv.ctl, sizeof(ctl), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  out3[1] = int32_t(ctl[CV_URGENT_LAST]);
  out3[2] = int32_t(ctl[CV_HEAD] - ctl[CV_TAIL]);
  out3[3] = int32_t(ctl[CV_SLICE]);
  return QS_OK;
}

int qs_action_dim(qs_handle h) { return h ? h->args.C.action_dim : QS_ERR_ARG; }
int qs_obs_dim(qs_handle h) { return h ? h->args.C.obs_dim : QS_ERR_ARG; }
int qs_num_envs(qs_handle h) { return h ? h->n : QS_ERR_ARG; }

int qs_get_state_ptrs(qs_handle h, qs_state_ptrs* o) {
  if (!h || !o) return fail(QS_ERR_ARG, "NULL argument");
  const DeviceView& D = h->args.D;
  o->state = D.state; o->tau_motor = D.tau_motor; o->tau_spring = D.tau_spring; o->kp = D.kp; o->kd = D.kd;
  o->spring = D.spring; o->mu = D.mu; o->foot_force = D.foot_force; o->contact = D.contact; o->task = D.task;
  o->last_action = D.last_action; o->sim_steps = D.sim_steps; o->env_steps = D.env_steps; o->ep_return = D.ep_return;
  o->custom_gains = D.custom_gains;
  o->land_mode = D.land_mode;
  o->rest_active = D.rest_active; o->rest = D.rest;
  o->mass_draw = D.mass_draw;
  o->filt = D.filt;
  o->work = D.work;
  return QS_OK;
}


// One turn of the settle conveyor.  In qs_step it runs on the second stream, forked after k_step and
// joined before the urgent pass, so that the slice shares the GPU with k_step_slow (a few latency-bound
// blocks); `flush` runs the whole window to completion in stream order (reset-time prefill).
static int launch_conveyor(qs_handle h, cudaStream_t s, int phase, int flush) {
  const int B = block_of(h);
  const int nsettle = h->cfg.is_rl_interface ? h->cfg.settling_steps : 1500;
  // the latency-bound kernel the slice of this phase runs next to, and how many of its envs cost the slice one block slot.
  // A block of the general solver (2 warps of slow_spread envs) costs TWO: an SM keeps one shared-memory / L1 split while
  // blocks are resident, that kernel lives on a large L1 (its solver rows are local memory; with the slice's split it
  // runs 2.4 x longer, measured), so an SM that holds one of its blocks takes no slice block at all.  Counting one slot
  // per block put the slice one wave + a few blocks past the free slots whenever more than ~1200 envs were in the
  // general solver, and those few blocks then ran as a second wave (+0.4 ms on the step).
  const int* busy = phase == 0 ? h->contact_list + h->n : h->slow_list + h->n;
  k_conveyor_ctl<<<1, 1024, 0, s>>>(h->cv, phase, busy, phase == 0 ? B : h->slow_spread, h->wave_blocks, B, h->n, nsettle,
                                    h->slice_min, h->slice_max, h->slice_early, flush);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}
// pdl: programmatic dependent launch behind the kernel just launched in `s` (k_step_slow, which issues
// griddepcontrol.launch_dependents on entry): the slice starts once every block of that kernel has been placed
static int launch_slice(qs_handle h, cudaStream_t s, int early, bool pdl = false, unsigned long long* stamps = nullptr) {
  const int B = block_of(h);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(unsigned(h->wave_blocks));
  cfg.blockDim = dim3(unsigned(B));
  cfg.dynamicSmemBytes = smem_of(B);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  if (h->args.C.mass_randomizer) CUDA_TRY(cudaLaunchKernelEx(&cfg, k_settle_slice<true>, h->args, h->cv, early, stamps));
  else CUDA_TRY(cudaLaunchKernelEx(&cfg, k_settle_slice<false>, h->args, h->cv, early, stamps));
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

static int need_demo(qs_handle h) {
  if (is_demo_task(h->args.C.task) && !h->args.C.demo)
    return fail(QS_ERR_STATE, "the *_DEMO tasks need a demonstration: call qs_set_demo first (tasks/task_base.py:169-176)");
  return QS_OK;
}

int qs_reset(qs_handle h, const uint8_t* mask, float* obs, void* stream) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  if (int e = need_demo(h)) return e;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(h->device));
  const int B = block_of(h);
  if (mask) {
    CUDA_TRY(cudaMemsetAsync(h->reset_list + h->n, 0, sizeof(int), s));
    k_compact<<<grid_for(h->n, 256), 256, 0, s>>>(mask, h->n, h->reset_list);
    if (h->args.C.mass_randomizer) k_reset<true><<<grid_for(h->n, B), B, smem_of(B), s>>>(h->args, h->reset_list, h->cv, obs); else k_reset<false><<<grid_for(h->n, B), B, smem_of(B), s>>>(h->args, h->reset_list, h->cv, obs);
    g_launches += 2;
  } else {
    if (h->args.C.mass_randomizer) k_reset<true><<<grid_for(h->n, B), B, smem_of(B), s>>>(h->args, nullptr, h->cv, obs); else k_reset<false><<<grid_for(h->n, B), B, smem_of(B), s>>>(h->args, nullptr, h->cv, obs);
    g_launches += 1;
  }
  CUDA_TRY(cudaGetLastError());
  if (h->cfg.auto_reset) {
    // settle the rings of the envs just reset, in stream order: every queued entry, one window at a time
    const size_t entries = size_t(QS_SLOTS) * size_t(h->n);
    const int rounds = int((entries + size_t(h->cv.width) - 1) / size_t(h->cv.width));
    for (int r = 0; r < rounds; r++) {
      if (int e = launch_conveyor(h, s, 1, 1)) return e;
      if (int e = launch_slice(h, s, 0)) return e;
    }
  }
  if (h->ext.ticks) {   // the reset envs' pushes end
    k_ext_countdown<<<grid_for(h->n, 256), 256, 0, s>>>(h->ext.ticks, mask, mask ? 0 : -1, h->n);
    g_launches += 1;
    CUDA_TRY(cudaGetLastError());
  }
  h->was_reset = true;
  return QS_OK;
}

// qs_step_host: rows of the envs k_step_slow finished, packed for one small copy (they are the only rows that change after
// k_step_contact; everything else is already on its way to the host while the general solver and the settle slice run)
__global__ void k_gather_late(const int* __restrict__ list, int n, int O, const float* __restrict__ obs,
                              const float* __restrict__ reward, const uint8_t* __restrict__ done,
                              const uint8_t* __restrict__ truncated, float* __restrict__ out, int cap) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int count = list[n];
  if (i == 0) out[0] = __int_as_float(count);
  if (i >= min(count, cap)) return;
  const int env = list[i];
  float* row = out + 4 + size_t(i) * size_t(O + 4);
  row[0] = __int_as_float(env);
  row[1] = reward[env];
  row[2] = float(done[env]);
  row[3] = float(truncated[env]);
  for (int k = 0; k < O; k++) row[4 + k] = obs[size_t(env) * O + k];
}

__global__ void k_zero3(int* a, int* b, int* c) {
  if (threadIdx.x == 0) { *a = 0; *b = 0; *c = 0; }
}

// host destinations of qs_step_host: copied as soon as the last step kernel has written them
struct HostOut {
  float* obs;
  float* reward;
  uint8_t* done;
  uint8_t* truncated;
};

static int ensure_events(qs_handle h) {
  if (!h->ev_ready) {
    for (int i = 0; i < qs_env::kRing; i++) {
      CUDA_TRY(cudaEventCreate(&h->ev0[i])); CUDA_TRY(cudaEventCreate(&h->ev1[i]));
      CUDA_TRY(cudaEventCreate(&h->ev4[i])); CUDA_TRY(cudaEventCreate(&h->ev5[i]));
    }
    h->ev_ready = true;
  }
  return QS_OK;
}
// a timing event: inside a stream capture it becomes an event-record node that can still be queried afterwards
static cudaError_t rec_timing(cudaEvent_t ev, cudaStream_t s, bool capturing) {
  return capturing ? cudaEventRecordWithFlags(ev, s, cudaEventRecordExternal) : cudaEventRecord(ev, s);
}

// The launches of one control step into stream s.  capture_slot >= 0: called under stream capture for the graph of
// timing-ring slot `capture_slot` (no host-side bookkeeping; the launcher does it per graph launch).
static int step_impl(qs_handle h, const float* actions, float* obs, float* reward, uint8_t* done, uint8_t* truncated,
                     void* stream, const HostOut* host, int capture_slot = -1) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  if (!actions || !obs || !reward || !done || !truncated) return fail(QS_ERR_ARG, "NULL buffer");
  if (!h->was_reset) return fail(QS_ERR_STATE, "qs_step before qs_reset");
  if (int e = need_demo(h)) return e;
  const bool capturing = capture_slot >= 0;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!capturing) CUDA_TRY(cudaSetDevice(h->device));
  const int B = block_of(h);
  const int64_t launches0 = g_launches.load();
  k_zero3<<<1, 32, 0, s>>>(h->slow_list + h->n, h->contact_list + h->n, h->flight_list + h->n);
  g_launches += 1;
  if (int e = ensure_events(h)) return e;
  StepIO io;
  io.actions = actions; io.obs = obs; io.reward = reward; io.done = done; io.truncated = truncated;
  io.term_obs = h->term_obs;
  io.slow_list = h->slow_list;
  io.contact_list = h->contact_list;
  io.flight_list = h->flight_list;
  io.cv = h->cv;
  const int slot = capturing ? capture_slot : int(h->n_steps % h->ring);
  io.stamps = h->stamps + 4 * slot;
  io.flight_cap = h->flight_cap;
  CUDA_TRY(rec_timing(h->ev0[slot], s, capturing));
  // the tick kernels' instantiation: <mass randomizer, substep trace, push>
  const SubstepTrace tr = h->trace;
  const ExtForce ef = h->ext;
  auto tick_kernels = [&](auto launch) {
    for_each_tick_variant([&](auto em, auto trace, auto push) {
      if (decltype(em)::value == bool(h->args.C.mass_randomizer) && decltype(trace)::value == (tr.buf != nullptr) &&
          decltype(push)::value == (ef.ticks != nullptr))
        launch(em, trace, push);
    });
  };
  k_pre<<<grid_for(h->n, 256), 256, 0, s>>>(h->args, io);
  g_launches += 1;
  tick_kernels([&](auto em, auto trace, auto push) {
    k_step<decltype(em)::value, decltype(trace)::value, decltype(push)::value><<<grid_for(h->n, B), B, smem_of(B), s>>>(h->args, io,
                                                                                                                   tr, ef);
  });
  if (h->cfg.auto_reset) {
    // conveyor, early slice: on the second stream, next to k_step_contact (about half a wave of blocks)
    if (int e = launch_conveyor(h, s, 0, 0)) return e;
    CUDA_TRY(cudaEventRecord(h->ev_fork0, s));
  }
  tick_kernels([&](auto em, auto trace, auto push) {
    k_step_contact<decltype(em)::value, decltype(trace)::value, decltype(push)::value><<<grid_for(h->n, B), B, smem_of(B), s>>>(
        h->args, io, tr, ef);
  });
  g_launches += 1;
  // The epilogue of every env whose ticks are done (all but the general solver's).  With host buffers it runs here, so
  // that the bulk of the results can leave for the host while k_step_slow and the late slice run.  With device buffers
  // it runs NEXT TO k_step_slow (a chain of programmatic dependent launches, below): the general solver's few blocks and
  // the late slice had come to end together, and this kernel's 0.08 ms in front of both was serial time.
  const bool finish_late = !host && h->cfg.auto_reset && h->finish_pdl;
  if (!finish_late) {
    if (h->args.C.mass_randomizer) k_finish<true><<<grid_for(h->n, QS_FINISH_BLOCK), QS_FINISH_BLOCK, 0, s>>>(h->args, io, nullptr); else k_finish<false><<<grid_for(h->n, QS_FINISH_BLOCK), QS_FINISH_BLOCK, 0, s>>>(h->args, io, nullptr);
    g_launches += 1;
  }
  CUDA_TRY(rec_timing(h->ev1[slot], s, capturing));
  if (!capturing) h->n_steps++;
  if (host) {
    // All rows but those of the envs now in the general solver's list are final: send everything to the host while
    // k_step_slow and the late settle slice run; the stragglers follow in a compact buffer (below), and rows an
    // urgent settle rewrites are fetched again by the caller (host_urgent).
    const size_t n = size_t(h->n), O = size_t(h->args.C.obs_dim);
    CUDA_TRY(cudaEventRecord(h->ev_results, s));
    CUDA_TRY(cudaStreamWaitEvent(h->copy, h->ev_results, 0));
    CUDA_TRY(cudaMemcpyAsync(host->obs, obs, n * O * sizeof(float), cudaMemcpyDeviceToHost, h->copy));
    CUDA_TRY(cudaMemcpyAsync(host->reward, reward, n * sizeof(float), cudaMemcpyDeviceToHost, h->copy));
    CUDA_TRY(cudaMemcpyAsync(host->done, done, n, cudaMemcpyDeviceToHost, h->copy));
    CUDA_TRY(cudaMemcpyAsync(host->truncated, truncated, n, cudaMemcpyDeviceToHost, h->copy));
  }
  if (h->cfg.auto_reset) {
    CUDA_TRY(cudaStreamWaitEvent(h->bg, h->ev_fork0, 0));
    CUDA_TRY(rec_timing(h->ev4[slot], h->bg, capturing));
    if (int e = launch_slice(h, h->bg, 1)) return e;
    CUDA_TRY(rec_timing(h->ev5[slot], h->bg, capturing));
    CUDA_TRY(cudaEventRecord(h->ev_early_done, h->bg));
    // the late slice works on the same entries: after the early one (over long before k_step_contact is)
    CUDA_TRY(cudaStreamWaitEvent(s, h->ev_early_done, 0));
    if (int e = launch_conveyor(h, s, 1, 0)) return e;
  }
  // envs parked for the general solver (joint limits / body contacts), then -- programmatic dependent launch -- the late
  // settle slice, which starts once every block of k_step_slow has been placed and runs next to it.  (Round 1 launched
  // the slice on a second stream: when the hardware placed it first, which it did on the three steps that follow a host
  // synchronisation, the general-solver blocks waited for the whole slice, +1 ms; a high-priority stream made it worse.)
  tick_kernels([&](auto em, auto trace, auto push) {
    k_step_slow<decltype(em)::value, decltype(trace)::value, decltype(push)::value><<<grid_for(h->n, 64), 64, 0, s>>>(
        h->args, io, h->slow_spread, tr, ef);
  });
  g_launches += 1;
  if (finish_late) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(grid_for(h->n, QS_FINISH_BLOCK)));
    cfg.blockDim = dim3(unsigned(QS_FINISH_BLOCK));
    cfg.dynamicSmemBytes = 0;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    const int* no_list = nullptr;
    if (h->args.C.mass_randomizer) CUDA_TRY(cudaLaunchKernelEx(&cfg, k_finish<true>, h->args, io, no_list));
    else CUDA_TRY(cudaLaunchKernelEx(&cfg, k_finish<false>, h->args, io, no_list));
    g_launches += 1;
  }
  if (h->cfg.auto_reset) {
    if (int e = launch_slice(h, s, 0, true, io.stamps)) return e;
  }
  if (host) {
    const int O = h->args.C.obs_dim;
    k_gather_late<<<grid_for(h->late_cap, 128), 128, 0, s>>>(h->slow_list, h->n, O, obs, reward, done, truncated, h->dev_late,
                                                             h->late_cap);
    g_launches += 1;
    CUDA_TRY(cudaEventRecord(h->ev_late, s));
    CUDA_TRY(cudaStreamWaitEvent(h->copy, h->ev_late, 0));
    CUDA_TRY(cudaMemcpyAsync(h->host_late, h->dev_late, (4 + size_t(h->late_cap) * size_t(O + 4)) * sizeof(float),
                             cudaMemcpyDeviceToHost, h->copy));
    CUDA_TRY(cudaEventRecord(h->ev_copied, h->copy));
  }
  if (h->cfg.auto_reset) {
    // envs that finished without a settled slot (rare): settled and started now
    if (h->args.C.mass_randomizer) k_settle_urgent<true><<<grid_for(h->n, B), B, smem_of(B), s>>>(h->args, h->cv, obs); else k_settle_urgent<false><<<grid_for(h->n, B), B, smem_of(B), s>>>(h->args, h->cv, obs);
    k_urgent_clear<<<1, 1, 0, s>>>(h->cv);
    g_launches += 2;
  }
  if (ef.ticks) {
    // the pushes' countdown, after every kernel that ran ticks of this step; ended episodes drop theirs
    k_ext_countdown<<<grid_for(h->n, 256), 256, 0, s>>>(ef.ticks, h->cfg.auto_reset ? done : nullptr, h->args.C.action_repeat, h->n);
    g_launches += 1;
  }
  CUDA_TRY(cudaGetLastError());
  h->launches_per_step = int(g_launches.load() - launches0);
  if (capturing) g_launches -= h->launches_per_step;   // counted per graph launch instead
  return QS_OK;
}

// qs_step through the step's CUDA graph (see qs_env::GraphKey); falls back to direct launches when the capture is not
// possible (more output-buffer sets than the cache holds, a driver that refuses the capture)
static int step_graph(qs_handle h, const float* actions, float* obs, float* reward, uint8_t* done, uint8_t* truncated,
                      void* stream) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  if (!h->use_graph) return step_impl(h, actions, obs, reward, done, truncated, stream, nullptr);
  if (!actions || !obs || !reward || !done || !truncated) return fail(QS_ERR_ARG, "NULL buffer");
  if (!h->was_reset) return fail(QS_ERR_STATE, "qs_step before qs_reset");
  if (int e = need_demo(h)) return e;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(h->device));
  if (int e = ensure_events(h)) return e;
  const size_t abytes = size_t(h->n) * size_t(h->args.C.action_dim) * sizeof(float);
  if (!h->act_buf) CUDA_TRY(cudaMalloc(&h->act_buf, size_t(h->n) * 12 * sizeof(float)));
  qs_env::GraphKey* key = nullptr;
  for (int i = 0; i < h->n_gkeys; i++) {
    qs_env::GraphKey& k = h->gkeys[i];
    if (k.obs == obs && k.reward == reward && k.done == done && k.trunc == truncated && k.term_obs == h->term_obs) { key = &k; break; }
  }
  if (!key) {
    if (h->n_gkeys == qs_env::kGraphKeys) return step_impl(h, actions, obs, reward, done, truncated, stream, nullptr);
    key = &h->gkeys[h->n_gkeys++];
    std::memset(key, 0, sizeof(*key));
    key->obs = obs; key->reward = reward; key->done = done; key->trunc = truncated; key->term_obs = h->term_obs;
  }
  const int v = int(h->n_steps % qs_env::kGraphSlots);
  if (!key->exec[v]) {
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamBeginCapture(h->main, cudaStreamCaptureModeThreadLocal);
    int rc = QS_OK;
    if (e == cudaSuccess) {
      rc = step_impl(h, h->act_buf, obs, reward, done, truncated, h->main, nullptr, v);
      e = cudaStreamEndCapture(h->main, &graph);
    }
    if (e == cudaSuccess && rc == QS_OK) e = cudaGraphInstantiate(&key->exec[v], graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (e != cudaSuccess || rc != QS_OK) {   // no graph on this system: direct launches from now on
      cudaGetLastError();
      key->exec[v] = nullptr;
      h->use_graph = false;
      h->ring = qs_env::kRing;
      return step_impl(h, actions, obs, reward, done, truncated, stream, nullptr);
    }
  }
  if (actions != h->act_buf) CUDA_TRY(cudaMemcpyAsync(h->act_buf, actions, abytes, cudaMemcpyDeviceToDevice, s));
  CUDA_TRY(cudaEventRecord(h->ev_in, s));
  CUDA_TRY(cudaStreamWaitEvent(h->main, h->ev_in, 0));
  CUDA_TRY(cudaGraphLaunch(key->exec[v], h->main));
  CUDA_TRY(cudaEventRecord(h->ev_out, h->main));
  CUDA_TRY(cudaStreamWaitEvent(s, h->ev_out, 0));
  g_launches += h->launches_per_step;
  h->n_steps++;
  return QS_OK;
}

static void drop_graphs(qs_handle h) {
  for (int i = 0; i < h->n_gkeys; i++)
    for (int v = 0; v < qs_env::kGraphSlots; v++)
      if (h->gkeys[i].exec[v]) cudaGraphExecDestroy(h->gkeys[i].exec[v]);
  h->n_gkeys = 0;
}

int qs_reset_to_state(qs_handle h, const uint8_t* mask, const float* states, float* obs, void* stream) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  if (!states) return fail(QS_ERR_ARG, "states is NULL");
  if (int e = need_demo(h)) return e;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(h->device));
  const int* list = nullptr;
  if (mask) {
    CUDA_TRY(cudaMemsetAsync(h->reset_list + h->n, 0, sizeof(int), s));
    k_compact<<<grid_for(h->n, 256), 256, 0, s>>>(mask, h->n, h->reset_list);
    g_launches += 1;
    list = h->reset_list;
  }
  if (h->args.C.mass_randomizer) k_reset_state<true><<<grid_for(h->n, 128), 128, 0, s>>>(h->args, list, states, h->cv, obs);
  else k_reset_state<false><<<grid_for(h->n, 128), 128, 0, s>>>(h->args, list, states, h->cv, obs);
  g_launches += 1;
  if (h->ext.ticks) {   // the reset envs' pushes end
    k_ext_countdown<<<grid_for(h->n, 256), 256, 0, s>>>(h->ext.ticks, mask, mask ? 0 : -1, h->n);
    g_launches += 1;
  }
  CUDA_TRY(cudaGetLastError());
  if (!mask) h->was_reset = true;
  return QS_OK;
}

int qs_set_demo(qs_handle h, const float* actions, int length) {
  if (!h || !actions) return fail(QS_ERR_ARG, "NULL argument");
  if (length < 1) return fail(QS_ERR_ARG, "a demonstration needs at least one row");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());  // no step may still be reading the old one
  if (h->dev_demo) CUDA_TRY(cudaFree(h->dev_demo));
  h->dev_demo = nullptr;
  const size_t bytes = size_t(length) * size_t(h->args.C.action_dim) * sizeof(float);
  CUDA_TRY(cudaMalloc(&h->dev_demo, bytes));
  CUDA_TRY(cudaMemcpy(h->dev_demo, actions, bytes, cudaMemcpyHostToDevice));
  h->args.C.demo = h->dev_demo;
  h->args.C.demo_len = length;
  drop_graphs(h);   // the kernel arguments are baked into the captured nodes
  return QS_OK;
}

int qs_set_substep_trace(qs_handle h, const int32_t* env_ids, int n_traced, float* trace) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());  // no step may still be reading the old map or writing the old rows
  std::vector<int32_t> col;
  if (trace) {
    if (n_traced < 1 || n_traced > h->n) return fail(QS_ERR_ARG, "n_traced must be in [1, N]");
    if (!env_ids) return fail(QS_ERR_ARG, "env_ids is NULL");
    std::vector<int32_t> ids(size_t(n_traced), 0);
    CUDA_TRY(cudaMemcpy(ids.data(), env_ids, ids.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
    col.assign(size_t(h->n), -1);
    for (int j = 0; j < n_traced; j++) {
      const int32_t e = ids[size_t(j)];
      if (e < 0 || e >= h->n) return fail(QS_ERR_ARG, "env id " + std::to_string(e) + " out of range");
      if (col[size_t(e)] >= 0) return fail(QS_ERR_ARG, "env id " + std::to_string(e) + " given twice");
      col[size_t(e)] = j;
    }
  }
  if (trace) CUDA_TRY(cudaMemcpy(h->trace.col, col.data(), col.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  h->trace.buf = trace;
  h->trace.n_traced = trace ? n_traced : 0;
  drop_graphs(h);   // the trace is a kernel argument of the captured nodes
  return QS_OK;
}

int qs_set_external_force(qs_handle h, float* wrench, int32_t* ticks) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  if ((wrench == nullptr) != (ticks == nullptr)) return fail(QS_ERR_ARG, "wrench and ticks must both be set or both be NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());  // no step may still be reading the old buffers
  h->ext.wrench = wrench;
  h->ext.ticks = ticks;
  drop_graphs(h);   // the buffers are kernel arguments of the captured nodes, and the tick kernels change
  return QS_OK;
}

int qs_apply_masses(qs_handle h, void* stream) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  if (!h->args.C.mass_randomizer)
    return fail(QS_ERR_STATE, "per-env masses need an env built with a mass randomizer mode (qs_config.mass_randomizer)");
  CUDA_TRY(cudaSetDevice(h->device));
  k_apply_masses<<<grid_for(h->n, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(h->args.D);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_set_terminal_obs(qs_handle h, float* term_obs) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  h->term_obs = term_obs;
  return QS_OK;
}

int qs_step(qs_handle h, const float* actions, float* obs, float* reward, uint8_t* done, uint8_t* truncated,
            void* stream) {
  return step_graph(h, actions, obs, reward, done, truncated, stream);
}

static int ensure_staging(qs_handle h) {
  const size_t n = size_t(h->n);
  if (!h->dev_actions) {
    CUDA_TRY(cudaMalloc(&h->dev_actions, n * 12 * sizeof(float)));
    CUDA_TRY(cudaMalloc(&h->dev_obs, n * QS_MAX_OBS * sizeof(float)));
    CUDA_TRY(cudaMalloc(&h->dev_reward, n * sizeof(float)));
    CUDA_TRY(cudaMalloc(&h->dev_done, 2 * n));
    h->dev_trunc = h->dev_done + n;
    h->late_cap = int(std::max<size_t>(1024, n / 16));
    if (const char* v = std::getenv("QS_LATE_CAP")) h->late_cap = std::max(1, std::atoi(v));  // (tests: force the overflow path)
    const size_t late_bytes = (4 + size_t(h->late_cap) * size_t(QS_MAX_OBS + 4)) * sizeof(float);
    CUDA_TRY(cudaMalloc(&h->dev_late, late_bytes));
    CUDA_TRY(cudaMallocHost(&h->host_late, late_bytes));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_late, cudaEventDisableTiming));
  }
  return QS_OK;
}

int qs_reset_host(qs_handle h, const uint8_t* mask, float* obs, void* stream) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(h->device));
  if (int e = ensure_staging(h)) return e;
  const size_t n = size_t(h->n), O = size_t(h->args.C.obs_dim);
  if (mask) CUDA_TRY(cudaMemcpyAsync(h->dev_done, mask, n, cudaMemcpyHostToDevice, s));
  if (obs && mask) CUDA_TRY(cudaMemcpyAsync(h->dev_obs, obs, n * O * sizeof(float), cudaMemcpyHostToDevice, s));
  if (int e = qs_reset(h, mask ? h->dev_done : nullptr, obs ? h->dev_obs : nullptr, stream)) return e;
  if (obs) CUDA_TRY(cudaMemcpyAsync(obs, h->dev_obs, n * O * sizeof(float), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  return QS_OK;
}

int qs_step_host(qs_handle h, const float* actions, float* obs, float* reward, uint8_t* done, uint8_t* truncated,
                 void* stream) {
  if (!h) return fail(QS_ERR_ARG, "handle is NULL");
  if (!actions || !obs || !reward || !done || !truncated) return fail(QS_ERR_ARG, "NULL buffer");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t n = size_t(h->n), A = size_t(h->args.C.action_dim), O = size_t(h->args.C.obs_dim);
  if (int e0 = ensure_staging(h)) return e0;
  CUDA_TRY(cudaMemcpyAsync(h->dev_actions, actions, n * A * sizeof(float), cudaMemcpyHostToDevice, s));
  const HostOut host{obs, reward, done, truncated};
  *h->host_urgent = 0;
  if (int e = step_impl(h, h->dev_actions, h->dev_obs, h->dev_reward, h->dev_done, h->dev_trunc, stream, &host)) return e;
  if (h->cfg.auto_reset)
    CUDA_TRY(cudaMemcpyAsync(h->host_urgent, h->cv.ctl + CV_URGENT_LAST, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamWaitEvent(s, h->ev_copied, 0));
  CUDA_TRY(cudaStreamSynchronize(s));
  int late = 0;
  std::memcpy(&late, h->host_late, sizeof(int));
  if (late > h->late_cap) {  // more stragglers than the side buffer holds (never seen; a robot pile-up): take everything again
    CUDA_TRY(cudaMemcpyAsync(obs, h->dev_obs, n * O * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(reward, h->dev_reward, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(done, h->dev_done, n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(truncated, h->dev_trunc, n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
  } else {
    for (int i = 0; i < late; i++) {  // the rows the general solver finished after the bulk copy had left
      const float* row = h->host_late + 4 + size_t(i) * (O + 4);
      int env;
      std::memcpy(&env, row, sizeof(int));
      reward[env] = row[1];
      done[env] = uint8_t(row[2]);
      truncated[env] = uint8_t(row[3]);
      std::memcpy(obs + size_t(env) * O, row + 4, O * sizeof(float));
    }
  }
  if (*h->host_urgent > 0 && late <= h->late_cap) {  // episodes settled and started after the copies: fetch their first obs
    CUDA_TRY(cudaMemcpyAsync(obs, h->dev_obs, n * O * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
  }
  return QS_OK;
}

int qs_set_state(qs_handle h, const float* state, void* stream) {
  if (!h || !state) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  k_set_state<<<grid_for(h->n * QS_STATE_DIM, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(h->args.D, state);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}
int qs_get_state(qs_handle h, float* state, void* stream) {
  if (!h || !state) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  k_get_state<<<grid_for(h->n * QS_STATE_DIM, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(h->args.D, state);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_observe(qs_handle h, float* obs, int with_noise, void* stream) {
  if (!h || !obs) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  k_observe<<<grid_for(h->n, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(h->args, obs, with_noise);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_debug_ticks(qs_handle h, const float* tau, int n_ticks, int use_f64, void* stream) {
  if (!h || !tau) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (use_f64) {
    DebugArgs<double> a;
    a.D = h->args.D; a.M = h->model_d; make_leg_pairs(a.M, a.M2); a.SC = h->args.SC; a.mass_randomizer = h->args.C.mass_randomizer;
    a.ext = h->ext;
    k_debug_ticks<double><<<grid_for(h->n, 64), 64, 64 * QS_TICK_SCRATCH * sizeof(double), s>>>(a, tau, n_ticks);
  } else {
    DebugArgs<float> a;
    a.D = h->args.D; a.M = h->args.M; a.M2 = h->args.M2; a.SC = h->args.SC; a.mass_randomizer = h->args.C.mass_randomizer;
    a.ext = h->ext;
    k_debug_ticks<float><<<grid_for(h->n, 64), 64, 64 * QS_TICK_SCRATCH * sizeof(float), s>>>(a, tau, n_ticks);
  }
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_action_to_command(const qs_config* cfg, const float* actions, float* cmd, int n, void* stream) {
  if (int e = check_config(cfg)) return e;
  if (!actions || !cmd || n <= 0) return fail(QS_ERR_ARG, "bad argument");
  RobotConst R;
  host::build_robot(*cfg, R);
  const int adim = host::action_dim_of(1, cfg->action_mode);
  k_action_to_command<<<grid_for(n, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(R, cfg->control_mode, cfg->action_mode,
                                                                                     adim, actions, cmd, n);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_pd_pea_torque(const float* cmd, const float* q, const float* qd, const float* kp12, const float* kd12,
                     const float* tau_max12, const float* spring9, int torque_mode, float* tau_motor,
                     float* tau_spring, int n, void* stream) {
  if (!cmd || !q || !qd || !kp12 || !kd12 || !tau_max12 || !tau_motor || n <= 0) return fail(QS_ERR_ARG, "bad argument");
  TorqueArgs T;
  std::memcpy(T.kp, kp12, sizeof T.kp);
  std::memcpy(T.kd, kd12, sizeof T.kd);
  std::memcpy(T.tau_max, tau_max12, sizeof T.tau_max);
  T.has_spring = spring9 != nullptr;
  if (spring9) std::memcpy(T.spring, spring9, sizeof T.spring); else std::memset(T.spring, 0, sizeof T.spring);
  T.torque_mode = torque_mode;
  k_pd_pea<<<grid_for(n * 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(T, cmd, q, qd, tau_motor, tau_spring, n);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_fk_jacobian(const float* q, const float* qd, float* pos, float* jac, float* vel, int n, void* stream) {
  if (!q || !pos || n <= 0) return fail(QS_ERR_ARG, "bad argument");
  k_fk<<<grid_for(n * 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(q, qd, pos, jac, vel, n);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_ik(const float* xyz, float* q, int n, void* stream) {
  if (!xyz || !q || n <= 0) return fail(QS_ERR_ARG, "bad argument");
  k_ik<<<grid_for(n * 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(xyz, q, n);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_cpg_update(double* X, const double* params9, const double* phi16, const float* q, const float* qd,
                  const float* gains8, float foot_y, float* xs, float* zs, float* tau, int n, void* stream) {
  if (!X || !params9 || !phi16 || n <= 0) return fail(QS_ERR_ARG, "bad argument");
  if (tau && (!q || !qd || !gains8)) return fail(QS_ERR_ARG, "torque output needs q, qd and gains");
  CpgArgs P;
  std::memcpy(P.p, params9, sizeof P.p);
  std::memcpy(P.phi, phi16, sizeof P.phi);
  if (gains8) std::memcpy(P.gains, gains8, sizeof P.gains); else std::memset(P.gains, 0, sizeof P.gains);
  P.foot_y = foot_y;
  k_cpg<<<grid_for(n, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(P, X, q, qd, xs, zs, tau, n, 12, 1);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_cpg_steps(qs_handle h, double* X, const double* params9, const double* phi16, const float* gains8, float foot_y,
                 int n_ticks, float* obs, float* reward, uint8_t* done, uint8_t* truncated, void* stream) {
  // hopf_network.py:241-289 for n_ticks control ticks without leaving the library: per tick the oscillators advance and the
  // torque law reads the joint state straight from the env's rows (k_cpg), then the env steps on those torques (the step's
  // CUDA graph).  Same numbers as the caller's own loop over qs_cpg_update + qs_step.
  if (!h || !X || !params9 || !phi16 || !gains8) return fail(QS_ERR_ARG, "NULL argument");
  if (h->args.C.is_rl || h->args.C.control_mode != QS_CTRL_TORQUE)
    return fail(QS_ERR_STATE, "the CPG drives a TORQUE-mode env built with isRLGymInterface=False (hopf_network.py:183-190)");
  if (n_ticks < 1) return fail(QS_ERR_ARG, "n_ticks must be positive");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!h->act_buf) CUDA_TRY(cudaMalloc(&h->act_buf, size_t(h->n) * 12 * sizeof(float)));
  CpgArgs P;
  std::memcpy(P.p, params9, sizeof P.p);
  std::memcpy(P.phi, phi16, sizeof P.phi);
  std::memcpy(P.gains, gains8, sizeof P.gains);
  P.foot_y = foot_y;
  const float* q = h->args.D.state + size_t(13) * h->n;
  const float* qd = h->args.D.state + size_t(25) * h->n;
  for (int t = 0; t < n_ticks; t++) {
    k_cpg<<<grid_for(h->n, 128), 128, 0, s>>>(P, X, q, qd, nullptr, nullptr, h->act_buf, h->n, 1, h->n);
    g_launches += 1;
    if (int e = step_graph(h, h->act_buf, obs, reward, done, truncated, stream)) return e;
  }
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

int qs_reduce_stats(qs_handle h, float* out, void* stream) {
  if (!h || !out) return fail(QS_ERR_ARG, "NULL argument");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemsetAsync(out, 0, QS_STATS_DIM * sizeof(float), s));
  k_stats<<<grid_for(h->n, 256), 256, 0, s>>>(h->args.D, out);
  g_launches += 1;
  CUDA_TRY(cudaGetLastError());
  return QS_OK;
}

}  // extern "C"
