"""Build + ctypes binding of the C-ABI library (include/qs_b200.h).

The CUDA library is the only implementation of the hot path: if it cannot be
built or loaded this module raises -- there is no eager/PyTorch/CPU fallback.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(CSRC, "libqs_b200.so")
SOURCES = ["qs_kernels.cu", "qs_render.cu", "qs_ars.cu", "qs_ppo.cu", "qs_step_kernels.cuh", "qs_env.cuh", "qs_physics.cuh", "qs_packed.cuh", "qs_robot.cuh", "qs_types.h", "qs_model_host.h"]
HEADER = os.path.join(os.path.dirname(_HERE), "include", "qs_b200.h")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
]

QS_MAX_OBS = 32
QS_TASK_DIM = 48
QS_STATS_DIM = 16
QS_STATE_DIM = 37
QS_TRACE_DIM = 66   # row of the per-substep trace (qs_set_substep_trace)
QS_EXT_DIM = 6      # rows of the push wrench (qs_set_external_force): force xyz (world, N), point xyz (base frame, m)
QS_CAM_DIM = 32     # camera row of qs_render: view matrix (16) then projection matrix (16), column-major
QS_ARS_MAX_HIDDEN = 64
QS_ARS_MAX_ACT = 12
QS_ARS_RELU, QS_ARS_TANH = 0, 1


class QsConfig(C.Structure):
    _fields_ = [
        ("enable_springs", C.c_int32), ("control_mode", C.c_int32), ("action_mode", C.c_int32),
        ("task", C.c_int32), ("obs_mode", C.c_int32), ("action_repeat", C.c_int32),
        ("is_rl_interface", C.c_int32), ("enable_action_filter", C.c_int32),
        ("ground_randomizer", C.c_int32), ("settling_steps", C.c_int32), ("enable_noise", C.c_int32),
        ("auto_reset", C.c_int32), ("num_iterations", C.c_int32), ("enable_limits", C.c_int32),
        ("body_contact_response", C.c_int32), ("block_size", C.c_int32),
        ("seed", C.c_uint64), ("env_id_offset", C.c_int64),
        ("time_step", C.c_double), ("max_episode_time", C.c_double),
        ("gravity_z", C.c_float), ("mu_ground", C.c_float), ("contact_erp", C.c_float),
        ("limit_erp", C.c_float), ("linear_slop", C.c_float), ("warmstart", C.c_float),
        ("residual_threshold", C.c_float), ("max_coord_vel", C.c_float),
        ("breaking_threshold", C.c_float), ("landing_mode", C.c_int32),
        ("spring_randomizer", C.c_int32), ("rest_mode", C.c_int32), ("mass_randomizer", C.c_int32), ("rand_leg_mass_err", C.c_float),
        ("rand_payload_max", C.c_float), ("rand_payload_pos", C.c_float * 3), ("rand_spring_err", C.c_float),
        ("self_collision", C.c_int32),
    ]


class QsArsArch(C.Structure):
    """qs_ars_arch: the network of sb3-contrib's ARSPolicy / ARSLinearPolicy that qs_ars_act evaluates"""
    _fields_ = [("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("n_hidden", C.c_int32), ("hidden", C.c_int32 * 2),
                ("activation", C.c_int32), ("bias", C.c_int32), ("squash", C.c_int32)]


class QsPpoArch(C.Structure):
    """qs_ppo_arch: the actor-critic network of SB3's ActorCriticPolicy that qs_ppo_act evaluates"""
    _fields_ = [("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("n_hidden", C.c_int32), ("hidden", C.c_int32 * 2),
                ("activation", C.c_int32)]


class QsPpoArgs(C.Structure):
    """qs_ppo_args: the pointers and scalars of one qs_ppo_act call"""
    _fields_ = [(n, C.c_void_p) for n in (
        "obs", "obs_mean", "obs_var", "theta", "episode_start", "prev_truncated", "terminal_obs", "actions", "buf_obs",
        "buf_actions", "buf_values", "buf_log_probs", "buf_episode_starts", "buf_rewards", "last_values", "mean_out")] + [
        ("clip_obs", C.c_double), ("epsilon", C.c_double), ("seed", C.c_uint64), ("env_id_offset", C.c_int64),
        ("gamma", C.c_float), ("iteration", C.c_int32), ("step", C.c_int32), ("n_steps", C.c_int32), ("n", C.c_int32),
        ("values_only", C.c_int32), ("deterministic", C.c_int32)]


class QsStatePtrs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "state", "tau_motor", "tau_spring", "kp", "kd", "spring", "mu", "foot_force", "contact", "task",
        "last_action", "sim_steps", "env_steps", "ep_return", "custom_gains", "land_mode", "rest_active", "rest", "mass_draw", "filt", "work")]


def nvcc_path():
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if p and (os.path.isabs(p) and os.path.exists(p) or not os.path.isabs(p)):
            return p
    return "nvcc"


def needs_build():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [HEADER]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """nvcc cross-compiles for sm_100a (works without a GPU)."""
    if not force and not needs_build():
        return SO_PATH
    # several processes may get here at once (torchrun ranks on a fresh checkout): one builds under a file lock into a
    # temporary file that is renamed into place, the others wait and then find the library up to date
    import fcntl
    with open(SO_PATH + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return SO_PATH
            tmp = f"{SO_PATH}.{os.getpid()}.tmp"
            cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [
                "-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES if s.endswith(".cu")]
            res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            if res.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + res.stdout)
            os.replace(tmp, SO_PATH)
            if verbose:
                print(res.stdout)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return SO_PATH


EXPORTS = {
    "qs_default_config": (None, [C.POINTER(QsConfig)]),
    "qs_obs_noise_std": (C.c_int, [C.POINTER(QsConfig), C.POINTER(C.c_float)]),
    "qs_config_obs_dim": (C.c_int, [C.POINTER(QsConfig)]),
    "qs_config_action_dim": (C.c_int, [C.POINTER(QsConfig)]),
    "qs_last_error": (C.c_char_p, []),
    "qs_device_count": (C.c_int, []),
    "qs_create": (C.c_int, [C.POINTER(QsConfig), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "qs_destroy": (C.c_int, [C.c_void_p]),
    "qs_action_dim": (C.c_int, [C.c_void_p]),
    "qs_obs_dim": (C.c_int, [C.c_void_p]),
    "qs_num_envs": (C.c_int, [C.c_void_p]),
    "qs_get_state_ptrs": (C.c_int, [C.c_void_p, C.POINTER(QsStatePtrs)]),
    "qs_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "qs_step": (C.c_int, [C.c_void_p] * 7),
    "qs_step_host": (C.c_int, [C.c_void_p] * 7),
    "qs_set_terminal_obs": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qs_apply_masses": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qs_set_demo": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "qs_set_substep_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "qs_set_external_force": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "qs_reset_to_state": (C.c_int, [C.c_void_p] * 5),
    "qs_reset_host": (C.c_int, [C.c_void_p] * 4),
    "qs_set_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "qs_get_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "qs_observe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "qs_debug_ticks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "qs_action_to_command": (C.c_int, [C.POINTER(QsConfig), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "qs_pd_pea_torque": (C.c_int, [C.c_void_p] * 3 + [C.POINTER(C.c_float)] * 4 + [C.c_int, C.c_void_p, C.c_void_p,
                                                                                C.c_int, C.c_void_p]),
    "qs_fk_jacobian": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_void_p]),
    "qs_ik": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "qs_cpg_update": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.c_void_p,
                                C.POINTER(C.c_float), C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                C.c_void_p]),
    "qs_cpg_steps": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_float),
                               C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "qs_reduce_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "qs_step_kernel_time": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_float)]),
    "qs_work_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "qs_debug_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "qs_settle_kernel_time": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_float)]),
    "qs_settle_work_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "qs_slow_kernel_time": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_float)]),
    "qs_step_count": (C.c_int64, [C.c_void_p]),
    "qs_timing_window": (C.c_int, [C.c_void_p]),
    "qs_render": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                            C.c_void_p]),
    "qs_obs_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 8),
    "qs_ars_act": (C.c_int, [C.c_void_p] * 3 + [C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_float, C.c_int,
                             C.c_int, C.c_int, C.POINTER(QsArsArch), C.c_void_p, C.c_int, C.c_void_p]),
    "qs_ppo_act": (C.c_int, [C.POINTER(QsPpoArgs), C.POINTER(QsPpoArch), C.c_void_p]),
    "qs_ppo_reward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_double] * 3 +
                      [C.c_void_p] * 5),
    "qs_ppo_gae": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_double, C.c_double] + [C.c_void_p] * 3),
    "qs_launch_count": (C.c_int64, []),
}

_LIB = None


def lib():
    """Load (building first if needed) the CUDA library; raises if unavailable."""
    global _LIB
    if _LIB is not None:
        return _LIB
    build()
    try:
        L = C.CDLL(SO_PATH)
    except OSError as e:  # pragma: no cover
        raise RuntimeError(f"cannot load {SO_PATH}: {e} (the CUDA extension is mandatory; no fallback)") from e
    for name, (res, args) in EXPORTS.items():
        f = getattr(L, name)  # AttributeError if the header and the library drift apart
        f.restype = res
        f.argtypes = args
    _LIB = L
    return L


class QsError(RuntimeError):
    pass


def check(code):
    if code != 0:
        msg = lib().qs_last_error().decode()
        if code == -1:
            raise ValueError(msg)
        raise QsError(f"[{code}] {msg}")
