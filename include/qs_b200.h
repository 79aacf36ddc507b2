/*
 * qs_b200.h -- C ABI of the B200-native batched Go1(+PEA) simulator.
 *
 * This is the drop-in boundary for the hot path of
 * francescovezzi/quadruped-springs: QuadrupedGymEnv.step / reset for N
 * independent environments (reference: quadruped_spring/env/quadruped_gym_env.py).
 * The reference is pure Python over pybullet and has no FFI of its own, so each
 * entry point cites the reference Python interface it replaces; INTEGRATION.md
 * shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain C types only; every buffer is caller-owned unless stated; device
 *     buffers are fp32 row-major [N, k] unless stated;
 *   - int return: 0 = ok, negative = QS_ERR_*; qs_last_error() gives the text
 *     (thread-local) -- replaces the reference's Python exceptions
 *     (quadruped_gym_env.py:168, quadruped.py:75);
 *   - every launch is asynchronous on the given cudaStream_t (passed as void*),
 *     no host synchronisation inside qs_step / qs_reset;
 *   - one handle per device, not re-entrant;
 *   - there is NO CPU fallback: every call fails with QS_ERR_CUDA if no sm_100
 *     device / driver is present.
 */
#ifndef QS_B200_H
#define QS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QS_OK 0
#define QS_ERR_ARG (-1)
#define QS_ERR_CUDA (-2)
#define QS_ERR_STATE (-3)

#define QS_STATE_DIM 37 /* pos3 quat4(xyzw) linvel3 angvel3 q12 qd12 (world frame) */
#define QS_MAX_OBS 32
#define QS_TASK_DIM 48
#define QS_STATS_DIM 16

/* registry keys of the reference, as integers (string -> id mapping lives in
 * the host layer and keeps the reference's names):
 * control_interface/collection.py:21-49, tasks/task_collection.py:19-37,
 * sensors/sensor_collection.py:92-105 */
enum qs_control_mode { QS_CTRL_PD = 0, QS_CTRL_CARTESIAN_PD = 1, QS_CTRL_TORQUE = 2 };
enum qs_action_mode { QS_ACT_DEFAULT = 0, QS_ACT_SYMMETRIC = 1, QS_ACT_SYMMETRIC_NO_HIP = 2 };
enum qs_task {
  QS_TASK_NO_TASK = 0,
  QS_TASK_JUMPING_IN_PLACE = 1,
  QS_TASK_JUMPING_FORWARD = 2,
  QS_TASK_BACKFLIP = 3,
  QS_TASK_JUMPING_IN_PLACE_PPO = 4,
  QS_TASK_JUMPING_FORWARD_PPO = 5,
  QS_TASK_BACKFLIP_PPO = 6,
  QS_TASK_JUMPING_IN_PLACE_PPO_HP = 7,
  QS_TASK_JUMPING_FORWARD_PPO_HP = 8,
  QS_TASK_CONTINUOUS_JUMPING_FORWARD = 9,      /* robot_tasks.py:102-131 */
  QS_TASK_CONTINUOUS_JUMPING_FORWARD2 = 10,    /* robot_tasks.py:134-166 */
  QS_TASK_CONTINUOUS_JUMPING_FORWARD3 = 11,    /* robot_tasks.py:169-212 */
  QS_TASK_CONTINUOUS_JUMPING_FORWARD_PPO = 12, /* robot_tasks.py:553-698 */
  /* imitation tasks (tasks/task_base.py:169-220, robot_tasks.py:222-241): per-step reward exp(-0.35 |a_demo - a|) / (rows
   * left at reset), episode ends with the demonstration; the demonstration is given with qs_set_demo */
  QS_TASK_JUMPING_IN_PLACE_DEMO = 13,
  QS_TASK_JUMPING_FORWARD_DEMO = 14,
  QS_TASK_BACKFLIP_DEMO = 15,
  QS_TASK_CONTINUOUS_JUMPING_FORWARD_DEMO = 16 /* TaskJumpingDemo2, tasks/task_base.py:402-452, robot_tasks.py:244-247 */
};
enum qs_obs_mode {
  QS_OBS_ENCODER = 0,
  QS_OBS_ENCODER_2,
  QS_OBS_CARTESIAN_NO_IMU,
  QS_OBS_ARS_BASIC,
  QS_OBS_ARS_SENSOR,
  QS_OBS_LANDING_SENSOR,
  QS_OBS_PPO_BASIC,
  QS_OBS_PPO_BASIC_X,
  QS_OBS_PPO_BASIC_CONTACT,
  QS_OBS_ARS_BACKFLIP,
  QS_OBS_PPO_BACKFLIP,
  QS_OBS_PPO_CONTINUOUS_JUMPING_FORWARD
};

/* Constructor arguments of QuadrupedGymEnv (quadruped_gym_env.py:52-70) plus the
 * physics-engine parameters the reference sets on pybullet
 * (quadruped_gym_env.py:301-309, quadruped.py:663-683).  Fill with
 * qs_default_config() first. */
typedef struct qs_config {
  int32_t enable_springs;        /* enable_springs */
  int32_t control_mode;          /* motor_control_mode */
  int32_t action_mode;           /* action_space_mode */
  int32_t task;                  /* task_env */
  int32_t obs_mode;              /* observation_space_mode */
  int32_t action_repeat;         /* action_repeat (10) */
  int32_t is_rl_interface;       /* isRLGymInterface */
  int32_t enable_action_filter;  /* enable_action_filter */
  int32_t ground_randomizer;     /* env_randomizer_mode == GROUND_RANDOMIZER: mu ~ U[0.5,1) per reset */
  int32_t settling_steps;        /* 2500 (quadruped_gym_env.py:115) */
  int32_t enable_noise;          /* sensor noise (sensors/sensor.py:25-60) */
  int32_t auto_reset;            /* reset finished envs inside qs_step (SB3 VecEnv behaviour) */
  int32_t num_iterations;        /* int(300/action_repeat) unless overridden (>0) */
  int32_t enable_limits;         /* joint-limit constraint rows */
  int32_t body_contact_response; /* non-foot shapes touching the ground are constrained too (general solver) */
  int32_t block_size;            /* CUDA block size of the step kernels: 0 or 128 (compiled in) */
  uint64_t seed;                 /* Philox key; streams are indexed by GLOBAL env id */
  int64_t env_id_offset;         /* global id of local env 0 (multi-GPU sharding) */
  double time_step;              /* 0.001; double so that sim_time > 10 s fires on control step 1001 like the reference */
  double max_episode_time;       /* EPISODE_LENGTH = 10 s (quadruped_gym_env.py:35) */
  float gravity_z;               /* -9.8 */
  float mu_ground;               /* used when ground_randomizer == 0 */
  float contact_erp, limit_erp, linear_slop, warmstart, residual_threshold;
  float max_coord_vel;           /* 30.1 */
  float breaking_threshold;      /* 0.02 */
  int32_t landing_mode;          /* 0 none; 1 LandingWrapper (env/wrappers/landing_wrapper.py:18-69): after take-off the action is
                                  * held until the predicted apex, then the landing action with gains 60 / 1.5 until the
                                  * episode ends; 2 LandingWrapper2 (landing_wrapper_2.py:39-78): default gains, landing until
                                  * touch-down, once per episode; 3 LandingWrapperContinuous (landing_wrapper_continuous.py:38-70):
                                  * triggered by every detected jump, landing until the jump is over; 4 / 5
                                  * LandingWrapperBackflip / Backflip2 (landing_wrapper_backflip*.py:47-80): scripted take-off
                                  * action until the backflip pitch reaches 5 pi / 8, then landing until the episode ends /
                                  * until touch-down.  The wrappers' inner env.step loops run as a per-env mode
                                  * machine: one qs_step = one control step, scripted envs ignore the action passed in */
  int32_t spring_randomizer;     /* EnvRandomizerSprings (env_randomizers/env_randomizer.py:86-122): every reset draws the
                                  * spring stiffness and damping of hip / thigh / calf within +-10 % of the nominal values;
                                  * the settle of that episode already runs on them.  No effect without springs */
  int32_t rest_mode;             /* 1: GoToRestWrapper (env/wrappers/go_to_rest_wrapper.py:43-95) outside the landing controller:
                                  * once the robot has jumped, stands on four feet and its base rises again, the env ramps from
                                  * its pose to the init action (1 s with springs, 0.3 s without) on gains 60 / 0.8 (60 / 1.5
                                  * without springs) and holds it until the episode ends; the action passed in is ignored */
  int32_t mass_randomizer;       /* EnvRandomizerMasses (env_randomizers/env_randomizer.py:19-84): every reset draws the hip /
                                  * thigh / calf link masses (the same for the four legs) within +-rand_leg_mass_err of nominal,
                                  * welds a block of U[0, rand_payload_max) kg to the trunk at U[-rand_payload_pos, +rand_payload_pos]
                                  * (base frame) and sets the trunk mass so that the total stays 12.01301 kg; the settle of that
                                  * episode already runs on them.  The reference's block is a second body on a JOINT_FIXED
                                  * constraint (quadruped.py:778-819); here it is welded on (folded into the trunk's inertia) */
  float rand_leg_mass_err;       /* 0.1; the *_CURRICULUM modes interpolate towards 0.2 (env_randomizer.py:148-169) */
  float rand_payload_max;        /* 1 kg -> 4 kg */
  float rand_payload_pos[3];     /* (0.1, 0, 0.1) m -> (0.2, 0, 0.2) */
  float rand_spring_err;         /* relative range of the spring stiffness / damping draws: 0.1 -> 0.3 (:242-262) */
  int32_t self_collision;        /* URDF_USE_SELF_COLLISION (quadruped.py:530-543): calf-involved self contacts count as
                                  * invalid contacts (quadruped.py:236-241); detection only.  Default 1 */
} qs_config;

typedef struct qs_env* qs_handle;

/* device pointers into the handle-owned structure-of-arrays state; every array
 * is [dim][N] (component-major, env-minor => coalesced).  Valid until
 * qs_destroy.  Replaces the Quadruped accessor surface (quadruped.py:82-222). */
typedef struct qs_state_ptrs {
  float* state;        /* [37][N] */
  float* tau_motor;    /* [12][N] last substep's clipped motor torque = GetMotorTorques() */
  float* tau_spring;   /* [12][N] */
  float* kp;           /* [12][N] per-env PD gains (quadruped_motor.py:45-99) */
  float* kd;           /* [12][N] */
  float* spring;       /* [9][N]  k3, b3, rest3 (springs.py:28-74) */
  float* mu;           /* [N] ground friction */
  float* foot_force;   /* [4][N] normal force of the last tick (quadruped.py:256) */
  int32_t* contact;    /* [N] bits 0-3: foot in contact, bits 8-: invalid (non-foot) contact count */
  float* task;         /* [QS_TASK_DIM][N] task state (tasks/task_base.py:40-59) */
  float* last_action;  /* [12][N] */
  int32_t* sim_steps;  /* [N] */
  int32_t* env_steps;  /* [N] */
  float* ep_return;    /* [N] */
  uint8_t* custom_gains; /* [N] set non-zero after writing kp/kd of an env: the kernels then read its gains from
                          * the arrays instead of the config constants; cleared by every reset of that env */
  int32_t* land_mode;  /* [N] landing controller mode: 0 policy, 1 take-off hold, 2 landing, 3 spent, 4 backflip take-off */
  int32_t* rest_active; /* [N] go-to-rest controller engaged (go_to_rest_wrapper.py:58-81) */
  float* rest;         /* [14][N] go-to-rest: h_actual, sim step of activation, start action[12] */
  float* mass_draw;    /* [8][N] mass randomizer, current episode: hip, thigh, calf link mass, trunk mass, block mass, block
                        * position[3] (Quadruped.GetLegMasses / get_offset_mass_value / get_offset_mass_position) */
  float* filt;         /* [4][12][N] action-filter history x[t-1], x[t-2], y[t-1], y[t-2] (utils/action_filter.py:110-127);
                        * y[t-1] is env.get_last_filtered_action() when the filter is on */
  uint32_t* work;      /* [3][N] per-env work counters of the step kernels: physics ticks, foot-contact ticks,
                        * contact x PGS-sweep count (cumulative; bench / diagnostics) */
} qs_state_ptrs;

void qs_default_config(qs_config* cfg);
/* host-only helpers (no GPU needed): per-element sensor noise std of cfg->obs_mode
 * (go1/configs_*.py:215-230 through sensors/robot_sensors.py), and the
 * observation/action dimensions for a config. */
int qs_obs_noise_std(const qs_config* cfg, float* out /*QS_MAX_OBS*/);
int qs_config_obs_dim(const qs_config* cfg);
int qs_config_action_dim(const qs_config* cfg);
const char* qs_last_error(void);
int qs_device_count(void);

/* QuadrupedGymEnv.__init__ (quadruped_gym_env.py:52-155) for n_envs envs */
int qs_create(const qs_config* cfg, int n_envs, int device, qs_handle* out);
/* QuadrupedGymEnv.close (quadruped_gym_env.py:337) */
int qs_destroy(qs_handle h);
int qs_action_dim(qs_handle h);
int qs_obs_dim(qs_handle h);
int qs_num_envs(qs_handle h);
int qs_get_state_ptrs(qs_handle h, qs_state_ptrs* out);

/* QuadrupedGymEnv.reset (quadruped_gym_env.py:278-297): re-initialise and
 * settle the envs whose mask byte is non-zero (all when mask == NULL); writes
 * the first observation of those envs into obs[N, O] when obs != NULL. */
int qs_reset(qs_handle h, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* QuadrupedGymEnv.step (quadruped_gym_env.py:227-256) for all N envs:
 * actions [N, A] -> obs [N, O], reward [N], done [N], truncated [N]
 * (infos["TimeLimit.truncated"]). */
int qs_step(qs_handle h, const float* actions_dev, float* obs_dev, float* reward_dev,
            uint8_t* done_dev, uint8_t* truncated_dev, void* stream);

/* TaskJumpingDemo.demo_list (tasks/task_base.py:169-176): the demonstration of the *_DEMO tasks, `length` rows of
 * action_dim actions in HOST memory (the action block of the rows GetDemonstrationWrapper records,
 * env/wrappers/get_demonstration_wrapper.py:35-57); copied to the device.  Must be set before qs_reset for those tasks.
 * The per-env position in it is task-state row QS_TS_DEMO_COUNTER (set_demo_counter, task_base.py:218-219). */
int qs_set_demo(qs_handle h, const float* actions_host, int length);
#define QS_TS_DEMO_COUNTER 29
/* ... and for QS_TASK_CONTINUOUS_JUMPING_FORWARD_DEMO, whose continuous-jumping bookkeeping occupies those rows */
#define QS_TS_DEMO2_COUNTER 42

/* Quadruped.SetLegMasses / SetBaseMass / _add_base_mass_offset (quadruped.py:744-819) on the batch: after the caller
 * wrote qs_state_ptrs.mass_draw, recompute the per-env mass properties the physics reads.  Needs
 * qs_config.mass_randomizer (the next reset of an env draws again). */
int qs_apply_masses(qs_handle h, void* stream);

/* Optional device buffer [N, O] (caller-owned; NULL detaches it): with auto_reset, qs_step writes there the LAST
 * observation of every env whose episode ended in that step -- infos[i]["terminal_observation"] of the
 * stable-baselines3 VecEnv the reference is trained through (load_model.py:109-113 make_vec_env -> DummyVecEnv);
 * rows of envs that did not finish are left untouched. */
int qs_set_terminal_obs(qs_handle h, float* term_obs_dev);

/* QuadrupedGymEnv.reset with env.set_robot_desired_state(...) (quadruped_gym_env.py:288-289,401; quadruped.py:470-471,
 * 521-525; ReferenceStateInitializationWrapper): the masked envs (all when mask == NULL) start a new episode from the
 * given physical state, rows of states_dev [N, 37] = pos3 quat4(xyzw) lin_vel3 ang_vel3 q12 qd12, WITHOUT the settle;
 * _last_action is zero, the task is reset on that state.  obs_dev [N, O] (optional) gets their first observation. */
int qs_reset_to_state(qs_handle h, const uint8_t* mask_dev, const float* states_dev, float* obs_dev, void* stream);

/* qs_reset with HOST buffers: mask_host [N] bytes or NULL (all), obs_host [N, O] or NULL;
 * synchronises the stream. */
int qs_reset_host(qs_handle h, const uint8_t* mask_host, float* obs_host, void* stream);

/* same call with HOST buffers (pinned or pageable): H2D of actions, the step,
 * D2H of the four results, all on `stream`; returns after the stream is
 * synchronised.  This is the end-to-end path a numpy caller (SB3 VecEnv) uses. */
int qs_step_host(qs_handle h, const float* actions_host, float* obs_host, float* reward_host,
                 uint8_t* done_host, uint8_t* truncated_host, void* stream);

/* Quadruped.reset_desired_state / env.set_robot_desired_state
 * (quadruped.py:521-525): overwrite the physical state [N,37] (row-major) */
int qs_set_state(qs_handle h, const float* state_dev /*[N,37]*/, void* stream);
int qs_get_state(qs_handle h, float* state_dev /*[N,37]*/, void* stream);
/* the clean observation of the current state (SensorList.get_obs, sensor.py:101-105) */
int qs_observe(qs_handle h, float* obs_dev, int with_noise, void* stream);

/* TEST HOOK: advance n_ticks physics ticks (pybullet.stepSimulation,
 * quadruped_gym_env.py:218-219) with fixed joint torques tau[N,12]; no task
 * bookkeeping.  use_f64 != 0 runs the double-precision instantiation of the
 * same kernel (algorithm check against the oracle, not a product path). */
int qs_debug_ticks(qs_handle h, const float* tau_dev, int n_ticks, int use_f64, void* stream);

/* ---- stand-alone analytic kernels (Quadruped / motor-model accessor surface) ---- */
/* ActionWrapper._transform_action_to_motor_command (interface_base.py:162-164) */
int qs_action_to_command(const qs_config* cfg, const float* actions_dev /*[N,A]*/,
                         float* cmd_dev /*[N,12]*/, int n, void* stream);
/* QuadrupedMotorModel.convert_to_torque + compute_spring_torques
 * (quadruped_motor.py:45-104).  kp/kd/tau_max are [12] host arrays, spring9 =
 * k3,b3,rest3 host array or NULL (no springs); outputs [N,12]. */
int qs_pd_pea_torque(const float* cmd_dev, const float* q_dev, const float* qd_dev,
                     const float* kp12, const float* kd12, const float* tau_max12,
                     const float* spring9, int torque_mode, float* tau_motor_dev,
                     float* tau_spring_dev, int n, void* stream);
/* Quadruped.ComputeJacobianAndPosition + ComputeFeetPosAndVel
 * (quadruped.py:348-397,440-449): q,qd [N,12] -> pos [N,12], J [N,4,9], vel [N,12] */
int qs_fk_jacobian(const float* q_dev, const float* qd_dev, float* pos_dev, float* jac_dev,
                   float* vel_dev, int n, void* stream);
/* Quadruped.ComputeInverseKinematics (quadruped.py:399-438): xyz [N,12] -> q [N,12] */
int qs_ik(const float* xyz_dev, float* q_dev, int n, void* stream);
/* HopfNetwork.update (hopf_network.py:117-173) + the Cartesian impedance law of
 * hopf_network.py:241-289.  X [N,8] float64 (r[4], theta[4]) is updated in place
 * (float64 because the reference starts every phase ON the sin(theta) > 0 switch);
 * params9 = mu, omega_swing, omega_stance, coupling, dt, des_step_len,
 * robot_height, ground_clearance, ground_penetration; phi16 row-major PHI;
 * gains8 = kp3, kd3, kpCartesian, kdCartesian.  tau [N,12] out (may be NULL);
 * xs, zs [N,4] out (may be NULL). */
int qs_cpg_update(double* X_dev, const double* params9, const double* phi16, const float* q_dev,
                  const float* qd_dev, const float* gains8, float foot_y, float* xs_dev,
                  float* zs_dev, float* tau_dev, int n, void* stream);
/* n_ticks turns of the reference's CPG loop (hopf_network.py:241-289) inside the library: per tick qs_cpg_update's
 * oscillator step and torque law on the env's own joint state, then qs_step on those torques.  The env must be a
 * TORQUE-mode env with is_rl_interface = 0 (hopf_network.py:183-190).  Outputs as qs_step, of the last tick. */
int qs_cpg_steps(qs_handle h, double* X_dev, const double* params9, const double* phi16, const float* gains8,
                 float foot_y, int n_ticks, float* obs_dev, float* reward_dev, uint8_t* done_dev,
                 uint8_t* truncated_dev, void* stream);
/* rollout statistics of this shard (EvaluationWrapper infos,
 * evaluation_wrapper.py:43-53; task maxima, task_base.py:51-57): out[QS_STATS_DIM]
 * floats on the device: count, finished episodes, sum/max of max_height,
 * rel_max_height, max_forward_distance, max_flight_time, flip completion,
 * return sum, length sum, terminated count. */
int qs_reduce_stats(qs_handle h, float* out_dev, void* stream);

/* measurement hooks (bench.py): device time of the last `last_k` step-kernel launches
 * (CUDA events on the launching stream; synchronise first), and the algorithmic-work
 * counters the step kernel keeps: out3 = {physics ticks, foot-contact ticks,
 * contact x PGS-sweep count} summed over all envs since creation. */
int qs_step_kernel_time(qs_handle h, int last_k, float* ms_sum);
int qs_work_counters(qs_handle h, uint64_t* out3, void* stream);
/* the same two for the settle slices (k_settle_slice, the kernel that pre-computes reset()'s 2500-tick settle,
 * control_interface/interface_base.py:182-200): device time of the launches of the last `last_k` steps, and
 * {settle ticks, foot-contact ticks, contact x PGS-sweep count} done so far */
int qs_settle_kernel_time(qs_handle h, int last_k, float* ms_sum);
int qs_settle_work_counters(qs_handle h, uint64_t* out3, void* stream);
/* device time of the general-solver launches (k_step_slow: joint limits, body contacts) of the last `last_k` steps,
 * and the number of qs_step / qs_step_host calls made on this handle so far */
int qs_slow_kernel_time(qs_handle h, int last_k, float* ms_sum);
int64_t qs_step_count(qs_handle h);
/* how many of the last steps the three timing hooks can look back on: 512 with direct launches, 16 when qs_step replays
 * the step's CUDA graph (one captured graph per timing slot; QS_GRAPH=0 in the environment turns the graph off) */
int qs_timing_window(qs_handle h);
/* diagnostics of the last qs_step: out4 = {envs handed to the general solver, envs whose next episode was
 * settled on the spot because no settled slot was ready, entries on the settle conveyor, ticks of its last
 * slice}; synchronises the stream */
int qs_debug_counters(qs_handle h, int32_t* out4, void* stream);

/* Per-substep trace (what QuadrupedGymEnv.set_sub_step_callback / MonitorState read after every stepSimulation,
 * quadruped_gym_env.py:152,222-223, utils/monitor_state.py:391-396): every later qs_step, qs_step_host and qs_cpg_steps
 * writes, for the n_traced envs env_ids_dev[0..n_traced) (device int32, distinct, in [0, N)), the values after each of
 * its action_repeat physics ticks into trace_dev [action_repeat][QS_TRACE_DIM][n_traced] (device float32, caller-owned;
 * column j = env env_ids_dev[j]).  Row t of the first index is tick t of the step:
 *   QS_TR_STATE       37 words in qs_get_state order (pos3 quat4 vlin3 vang3 q12 qd12)
 *   QS_TR_TAU_MOTOR   12 clipped motor torques applied in that tick (GetMotorTorques)
 *   QS_TR_TAU_SPRING  12 spring torques applied in that tick
 *   QS_TR_FOOT_FORCE  4 foot normal forces, 0 for a foot not in contact (GetContactInfo)
 *   QS_TR_CONTACT     contact word (mask & 15) | invalid << 8 as a float (exact)
 * With auto_reset, the rows of an env whose episode ends in the step are the ticks of that episode (the NaN / Inf guard
 * does not clear them).  Resets, settles and qs_debug_ticks write nothing.  The ids are checked on the host (the call
 * synchronises the device); QS_ERR_ARG when n_traced is not in [1, N] or an id repeats or is out of range.
 * trace_dev == NULL clears the trace.  Steps without a trace run the same kernels as before the feature existed. */
#define QS_TRACE_DIM 66
#define QS_TR_STATE 0
#define QS_TR_TAU_MOTOR 37
#define QS_TR_TAU_SPRING 49
#define QS_TR_FOOT_FORCE 61
#define QS_TR_CONTACT 65
int qs_set_substep_trace(qs_handle h, const int32_t* env_ids_dev, int n_traced, float* trace_dev);

/* Quadruped.apply_external_force (quadruped.py:338-343) for the batch: a push on the base, applied inside the step
 * kernels tick by tick.  wrench_dev [QS_EXT_DIM][N] and ticks_dev [N] are caller-owned device buffers, component-major
 * like the qs_state_ptrs arrays.  Env i's push is the force F = wrench rows 0-2 (world frame, N) at the point p = rows
 * 3-5 (base frame, from the base position GetBasePosition, m): in each tick it acts on, it is Bullet's
 * applyExternalForce(robot, -1, F, pos + R p, WORLD_FRAME) made before that stepSimulation, the moment recomputed from
 * that tick's orientation.  ticks_dev[i] = n is the number of physics ticks the push still lasts:
 *   qs_step / qs_step_host / qs_cpg_steps  tick t (0-based) of the step's R = action_repeat ticks is pushed iff t < n
 *                                          at the start of the step; after the step n -= min(n, R), and with auto_reset
 *                                          n = 0 for an env whose episode ended in the step (NaN / Inf guard included)
 *   qs_reset / qs_reset_host / qs_reset_to_state  n = 0 for the reset envs
 *   qs_debug_ticks                         the same rule over its n_ticks
 *   settles (the conveyor's included)      never pushed, consume nothing
 * The library decrements and clears ticks_dev; between steps the caller may write new values into both buffers without
 * another call.  An env with n = 0 runs exactly the arithmetic of an unpushed step.  Both NULL detaches the buffers (the
 * steps run the same kernels as before the feature existed); QS_ERR_ARG when exactly one is NULL.  Attaching or
 * detaching synchronises the device and drops the captured step graphs. */
#define QS_EXT_DIM 6   /* rows: force xyz (world, N), point xyz (base frame, from the base position, m) */
int qs_set_external_force(qs_handle h, float* wrench_dev /*[QS_EXT_DIM][N]*/, int32_t* ticks_dev /*[N]*/);

/* Camera images of robots (QuadrupedGymEnv.render(mode="rgb_array") -> pybullet getCameraImage,
 * quadruped_gym_env.py render; utils/video_recording.py): image i shows the robot of states_dev row i (qs_get_state
 * rows, so recorded states render as well) on the ground plane, seen by camera row i = pybullet's view matrix (16) then
 * projection matrix (16), column-major as computeViewMatrix* / computeProjectionMatrix* return them.  Stateless, needs
 * no handle.  Drawn: the plane z = 0 (1 m checkerboard) and the 18 collision primitives the contact code collides (the
 * mass randomizer's payload block is not drawn), one flat colour per link kind, one directional light with shadows of
 * the robot.  Pixel (r, c), row 0 at the top, is the ray through its centre, x_ndc = 2 (c + 0.5) / W - 1,
 * y_ndc = 1 - 2 (r + 0.5) / H, unprojected through inverse(P V) from the near to the far plane; no anti-aliasing.
 *   rgb_dev   [k][H][W][3] uint8, sky colour for a miss
 *   depth_dev [k][H][W] metric eye-space depth -z_eye (pybullet's depth buffer d linearised as
 *             far near / (far - (far - near) d)); far for a miss
 *   seg_dev   [k][H][W] ER_SEGMENTATION_MASK_OBJECT_AND_LINKINDEX: objectUniqueId + ((linkIndex + 1) << 24), plane 0
 *             (object 0, link -1), robot object 1 with URDF link indices (trunk 0, imu 1, then hip, thigh, calf, foot of
 *             FR, FL, RR, RL: feet 5, 9, 13, 17); -1 for a miss
 * Any of the three may be NULL, not all.  A state row with a non-finite word draws no robot.  QS_ERR_ARG when k < 1,
 * width or height is outside [1, 4096], or no output is given.  Launches one kernel on `stream`. */
#define QS_CAM_DIM 32
int qs_render(const float* states_dev /*[k, QS_STATE_DIM]*/, const float* cams_dev /*[k, QS_CAM_DIM]*/, int k, int width,
              int height, uint8_t* rgb_dev, float* depth_dev, int32_t* seg_dev, void* stream);

/* ---- ARS training (sb3_contrib.ars.ARS with one candidate policy per group of envs; quadruped_springs_b200/ars.py) ----
 * Two stateless entry points, run once per control step beside qs_step.  Neither synchronises the host. */

/* Running observation statistics (VecNormalize.obs_rms, RunningMeanStd.update, float64) and episode bookkeeping.
 * Statistics (mean_dev, var_dev, count_dev all non-NULL): the rows r of obs_dev [n, o] with alive_dev[r] != 0 (every row
 * when alive_dev is NULL) form one batch; its mean and population variance are merged into the running mean, var and
 * count (Chan et al.) exactly as RunningMeanStd.update merges them.  No alive row leaves all three unchanged.  count_dev
 * lives on the device because the host does not know how many rows are alive.  mean_dev == NULL skips the statistics
 * (obs_dev may then be NULL).
 * Bookkeeping (reward_dev, done_dev, ret_dev, len_dev all non-NULL; alive_dev required): for every row r,
 *   if alive[r]: ret[r] += reward[r] (float64), len[r] += 1;  then alive[r] &= !done[r]
 * after the row has been read for the statistics, so the statistics of a step see the envs that were alive before it.
 * QS_ERR_ARG when n < 1, o is outside [1, QS_MAX_OBS] (with statistics), or neither part is requested.  One launch of
 * one 8-block cluster: the result does not depend on the launch, only on the rows and their order. */
int qs_obs_stats(const float* obs_dev /*[n, o]*/, uint8_t* alive_dev /*[n] or NULL*/, int n, int o, double* mean_dev,
                 double* var_dev, double* count_dev /*[1]*/, const float* reward_dev, const uint8_t* done_dev,
                 double* ret_dev, int32_t* len_dev, void* stream);

/* The policy network of sb3-contrib's ARSPolicy / ARSLinearPolicy: Linear layers (weight [out, in] row-major, then bias
 * when `bias`), `activation` after each hidden layer, tanh on the output when `squash`. */
#define QS_ARS_MAX_HIDDEN 64
#define QS_ARS_MAX_ACT 12
#define QS_ARS_RELU 0
#define QS_ARS_TANH 1
typedef struct {
  int32_t obs_dim;      /* [1, QS_MAX_OBS] */
  int32_t act_dim;      /* [1, QS_ARS_MAX_ACT] */
  int32_t n_hidden;     /* 0, 1 or 2 */
  int32_t hidden[2];    /* each in [1, QS_ARS_MAX_HIDDEN] (the first n_hidden) */
  int32_t activation;   /* QS_ARS_RELU or QS_ARS_TANH */
  int32_t bias;         /* 0 or 1 */
  int32_t squash;       /* 0 or 1 */
} qs_ars_arch;

/* Actions of ARS candidate policies.  Env e (row e of obs_dev) runs candidate c = first_candidate + e / envs_per_candidate,
 * whose parameter vector is theta + delta_std * deltas[c] for c < n_delta and theta - delta_std * deltas[c - n_delta]
 * otherwise (each product rounded to fp32 before the sum, as torch computes it); deltas_dev == NULL means theta itself
 * for every env.  theta [P] is parameters_to_vector of the policy (layer by layer: weight row-major, then bias).  The
 * observation is first normalised as VecNormalize does, in float64: clip((obs - mean) / sqrt(var + eps), +-clip_obs),
 * rounded to fp32 (mean_dev == NULL: no normalisation).  Output actions_dev [n, act_dim], clipped to [-1, 1].
 * A block evaluates envs of one candidate, forming that candidate's weights once into shared memory; an env's action
 * does not depend on the other envs of the call.  QS_ERR_ARG for an arch outside the ranges above, n < 1,
 * envs_per_candidate < 1, n_delta < 1, or a candidate index outside [0, 2 n_delta).  One launch. */
int qs_ars_act(const float* obs_dev /*[n, obs_dim]*/, const double* mean_dev, const double* var_dev, double clip_obs,
               double eps, const float* theta_dev /*[P]*/, const float* deltas_dev /*[n_delta, P] or NULL*/,
               float delta_std, int n_delta, int first_candidate, int envs_per_candidate, const qs_ars_arch* arch,
               float* actions_dev /*[n, act_dim]*/, int n, void* stream);

/* ---- PPO training (stable_baselines3.PPO with VecNormalize over the batch; quadruped_springs_b200/ppo.py) ----
 * Three stateless entry points.  Per control step qs_ppo_act runs before qs_step, qs_obs_stats (statistics only) and
 * qs_ppo_reward after it; qs_ppo_gae runs once per rollout.  None synchronises the host.  Rollout buffers are step-major:
 * row t of a [n_steps, n, ...] array holds step t of every env. */

/* The network of SB3's ActorCriticPolicy with the default MlpExtractor and one net_arch for both heads.  theta is
 * parameters_to_vector of MlpPolicyTorch, in this order (torch lists a module's own parameters before its children's;
 * each Linear: weight [out, in] row-major, then bias [out]):
 *   log_std                   [act_dim]
 *   mlp_extractor.policy_net  n_hidden Linear layers (obs_dim -> hidden[0] -> hidden[1])
 *   mlp_extractor.value_net   the same shapes
 *   action_net                Linear(last, act_dim), last = hidden[n_hidden - 1] or obs_dim
 *   value_net                 Linear(last, 1)
 * `activation` follows every hidden layer. */
typedef struct {
  int32_t obs_dim;      /* [1, QS_MAX_OBS] */
  int32_t act_dim;      /* [1, QS_ARS_MAX_ACT] */
  int32_t n_hidden;     /* 0, 1 or 2 */
  int32_t hidden[2];    /* each in [1, QS_ARS_MAX_HIDDEN] (the first n_hidden) */
  int32_t activation;   /* QS_ARS_RELU or QS_ARS_TANH */
} qs_ppo_arch;

/* Pointers and scalars of one qs_ppo_act call (device pointers; NULL where a field is not used). */
typedef struct {
  const float* obs;                /* [n, obs_dim] raw observations of step `step` */
  const double* obs_mean;          /* [obs_dim] running statistics (VecNormalize.obs_rms); NULL: no normalisation */
  const double* obs_var;           /* [obs_dim] */
  const float* theta;              /* [P], see qs_ppo_arch */
  const uint8_t* episode_start;    /* [n] 1 where step `step` starts an episode (the previous step's done) */
  const uint8_t* prev_truncated;   /* [n] the previous step's TimeLimit.truncated; NULL: no bootstrap */
  const float* terminal_obs;       /* [n, obs_dim] raw terminal observations of the previous step (qs_set_terminal_obs) */
  float* actions;                  /* [n, act_dim] the env action: the sample (or the mean) clipped to [-1, 1] */
  float* buf_obs;                  /* [n_steps, n, obs_dim] normalised observations */
  float* buf_actions;              /* [n_steps, n, act_dim] unclipped samples */
  float* buf_values;               /* [n_steps, n] */
  float* buf_log_probs;            /* [n_steps, n] */
  float* buf_episode_starts;       /* [n_steps, n] 0 / 1 */
  float* buf_rewards;              /* [n_steps, n] the bootstrap adds to row step - 1 */
  float* last_values;              /* [n] values_only: V of the observations */
  float* mean_out;                 /* [n, act_dim] or NULL: the actor mean */
  double clip_obs, epsilon;        /* VecNormalize's clip_obs and epsilon */
  uint64_t seed;                   /* key of the policy noise */
  int64_t env_id_offset;           /* global id of row 0 (shards) */
  float gamma;                     /* discount of the bootstrap */
  int32_t iteration;               /* rollout index: part of the noise key */
  int32_t step;                    /* in [0, n_steps) for a sampling call, in [0, n_steps] otherwise */
  int32_t n_steps;
  int32_t n;
  int32_t values_only;             /* 1: last_values and the bootstrap only */
  int32_t deterministic;           /* 1: actions = clipped mean, nothing else is written (but mean_out) */
} qs_ppo_args;

/* Actor and critic of every env (one thread per env).  The observation is normalised as VecNormalize does, in float64:
 * clip((obs - mean) / sqrt(var + eps), +-clip_obs), rounded to fp32 (the same bits as VecNormalizeTorch.normalize_obs).
 * A sampling call draws eps ~ N(0, 1) per action entry from Philox keyed by (seed, env_id_offset + row, iteration, step),
 * a = mean + exp(log_std) eps, log_prob = sum_i log N(a_i; mean_i, std_i), and writes row `step` of every buffer
 * (normalised obs, a, V, log_prob, episode start) and the clipped env action.  Where episode_start and prev_truncated
 * are both set, buf_rewards[step - 1] += gamma V(normalised terminal_obs), SB3's time-limit bootstrap; the terminal
 * observation is normalised with the same statistics as the step's own.  values_only writes last_values and that
 * bootstrap (call it with step = n_steps after the last step).  QS_ERR_ARG for an arch outside its ranges, n < 1, a
 * step outside [0, n_steps) for a sampling call or outside [0, n_steps] for the others, or a missing pointer the call
 * needs.  One launch. */
int qs_ppo_act(const qs_ppo_args* args, const qs_ppo_arch* arch, void* stream);

/* VecNormalize's reward path and Monitor's episode totals for one step of n envs (one 8-block cluster):
 *   ret = ret * gamma + reward (float64); every row's ret merged into ret_rms (mean, var, count [1] each; Chan et al. in
 *   a fixed order, then RunningMeanStd.update_from_moments); reward_out = clip(reward / sqrt(var + epsilon),
 *   +-clip_reward) with the updated var, rounded to fp32; ret = 0 where done.
 *   ep_return += reward (float64), ep_length += 1; where done they are added to totals[0..2] = {episodes, sum of returns,
 *   sum of lengths} and cleared; totals[3] += the sum of every row's reward (fixed order; totals [4] may be NULL).
 * ret, ret_mean, ret_var and ret_count all NULL: no normalisation, reward_out = reward.  The result does not depend on
 * the launch, only on the rows and their order. */
int qs_ppo_reward(const float* reward_dev, const uint8_t* done_dev, int n, double* ret_dev, double* ret_mean_dev,
                  double* ret_var_dev, double* ret_count_dev, double gamma, double epsilon, double clip_reward,
                  float* reward_out_dev, double* ep_return_dev, int32_t* ep_length_dev, double* totals_dev,
                  void* stream);

/* RolloutBuffer.compute_returns_and_advantage over step-major [n_steps, n] arrays, fp32 operation for operation:
 * next_non_terminal = 1 - last_dones (last step) or 1 - episode_starts[t + 1], next_values = last_values or
 * values[t + 1], delta = rewards[t] + gamma next_values next_non_terminal - values[t],
 * adv[t] = delta + gamma gae_lambda next_non_terminal adv[t + 1]; returns = adv + values.  One launch. */
int qs_ppo_gae(const float* rewards_dev, const float* values_dev, const float* episode_starts_dev,
               const float* last_values_dev /*[n]*/, const uint8_t* last_dones_dev /*[n]*/, int n_steps, int n,
               double gamma, double gae_lambda, float* advantages_dev, float* returns_dev, void* stream);

/* number of kernels launched by this library since load (bench bookkeeping) */
int64_t qs_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
