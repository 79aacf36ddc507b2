"""Batched, GPU-resident mirror of the reference's gym interface.

`BatchedQuadrupedGymEnv` keeps the constructor keywords, registry keys and the
reset/step contract of QuadrupedGymEnv (quadruped_spring/env/quadruped_gym_env.py:41-256)
for `num_envs` independent robots.  All arithmetic runs in the CUDA library
behind the C ABI (include/qs_b200.h); this file only owns buffers, string->id
registries and zero-copy tensor views.  There is no CPU path.
"""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import torch

from . import _lib
from .configs import SENSOR_SETS, go1_config, observation_layout

ACTION_EPS = 0.01       # quadruped_gym_env.py:33
OBSERVATION_EPS = 0.01  # quadruped_gym_env.py:34
EPISODE_LENGTH = 10     # quadruped_gym_env.py:35


class _Collection:
    """utils/base_collection.py:1-15 with the same keys; unknown keys raise
    ValueError (the reference prints and returns None, then fails later)."""

    def __init__(self, element_type, keys):
        self._element_type = element_type
        self._dict = {k: i for i, k in enumerate(keys)}

    def get_el(self, keyword):
        try:
            return self._dict[keyword]
        except KeyError:
            raise ValueError(f"the {self._element_type} {keyword} is not implemented yet.") from None

    def keys(self):
        return list(self._dict)


# control_interface/collection.py:21-49
MotorInterfaceCollection = lambda: _Collection("motor control mode", ["PD", "CARTESIAN_PD", "TORQUE"])
ActionInterfaceCollection = lambda: _Collection("action space mode", ["DEFAULT", "SYMMETRIC", "SYMMETRIC_NO_HIP"])
# tasks/task_collection.py:19-37 (the *_DEMO tasks replay recorded trajectories on the host: SURVEY.md section 2 #8)
TaskCollection = lambda: _Collection("task", [
    "NO_TASK", "JUMPING_IN_PLACE", "JUMPING_FORWARD", "BACKFLIP", "JUMPING_IN_PLACE_PPO", "JUMPING_FORWARD_PPO",
    "BACKFLIP_PPO", "JUMPING_IN_PLACE_PPO_HP", "JUMPING_FORWARD_PPO_HP", "CONTINUOUS_JUMPING_FORWARD",
    "CONTINUOUS_JUMPING_FORWARD2", "CONTINUOUS_JUMPING_FORWARD3", "CONTINUOUS_JUMPING_FORWARD_PPO",
    "JUMPING_IN_PLACE_DEMO", "JUMPING_FORWARD_DEMO", "BACKFLIP_DEMO", "CONTINUOUS_JUMPING_FORWARD_DEMO"])
# sensors/sensor_collection.py:92-105
SensorCollection = lambda: _Collection("sensor package", list(SENSOR_SETS))
# env_randomizers/env_randomizer_collection.py:15-21 (mass / curriculum randomizers: SURVEY.md 8f "next")
EnvRandomizerCollection = lambda: _Collection("env randomizer", [
    "GROUND_RANDOMIZER", "NO_RANDOMIZER", "SPRING_RANDOMIZER", "MASS_RANDOMIZER", "TEST_RANDOMIZER",
    "TEST_RANDOMIZER_CURRICULUM"])


class Box:
    """Minimal stand-in for gym.spaces.Box (gym is not a dependency)."""

    def __init__(self, low, high, dtype=np.float32):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = np.dtype(dtype)

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)

    def __repr__(self):
        return f"Box({self.shape}, {self.dtype})"


class _DevArray:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def _view(ptr, shape, typestr, device):
    """zero-copy torch view of handle-owned device memory"""
    with torch.cuda.device(device):
        return torch.as_tensor(_DevArray(ptr, shape, typestr), device=device)


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class BatchedQuadruped:
    """Accessor surface of env/quadruped.py:82-449 on [N, ...] tensors.

    Getters return views of kernel-owned state (no copies); component-major
    arrays are exposed transposed so that indexing reads like the reference
    (`GetMotorAngles()[env, motor]`)."""

    def __init__(self, env):
        self._env = env
        self._robot_config = env._robot_config
        self.num_motors, self.num_legs = 12, 4
        v = env._views
        s = v["state"]
        self._pos, self._quat = s[0:3].t(), s[3:7].t()
        self._vlin, self._vang = s[7:10].t(), s[10:13].t()
        self._q, self._qd = s[13:25].t(), s[25:37].t()

    def getHeight(self):
        return self._pos[:, 2]

    def GetBasePosition(self):                      # quadruped.py:107-114
        return self._pos

    def GetBaseOrientation(self):                   # :116-129 (xyzw)
        return self._quat

    def GetBaseOrientationMatrix(self):             # :172-175
        x, y, z, w = self._quat.unbind(-1)
        s = 2.0 / (x * x + y * y + z * z + w * w)
        R = torch.stack([1 - s * (y * y + z * z), s * (x * y - w * z), s * (x * z + w * y),
                         s * (x * y + w * z), 1 - s * (x * x + z * z), s * (y * z - w * x),
                         s * (x * z - w * y), s * (y * z + w * x), 1 - s * (x * x + y * y)], dim=-1)
        return R.view(-1, 3, 3)

    def GetBaseOrientationRollPitchYaw(self):       # :131-139 (pybullet getEulerFromQuaternion)
        x, y, z, w = self._quat.unbind(-1)
        sarg = -2 * (x * z - w * y)
        roll = torch.atan2(2 * (y * z + w * x), w * w - x * x - y * y + z * z)
        pitch = torch.asin(sarg.clamp(-1, 1))
        yaw = torch.atan2(2 * (x * y + w * z), w * w + x * x - y * y - z * z)
        lo, hi = sarg <= -0.99999, sarg >= 0.99999
        roll = torch.where(lo | hi, torch.zeros_like(roll), roll)
        pitch = torch.where(lo, torch.full_like(pitch, -0.5 * np.pi), torch.where(hi, torch.full_like(pitch, 0.5 * np.pi), pitch))
        yaw = torch.where(lo, 2 * torch.atan2(x, -y), torch.where(hi, 2 * torch.atan2(-x, y), yaw))
        return torch.stack([roll, pitch, yaw], dim=-1)

    def GetTrueBaseRollPitchYawRate(self):          # :141-170: R^T omega
        return torch.einsum("nji,nj->ni", self.GetBaseOrientationMatrix(), self._vang)

    def GetBaseLinearVelocity(self):                # :177-180
        return self._vlin

    def GetBaseAngularVelocity(self):               # :182-185
        return self._vang

    def GetMotorAngles(self):                       # :187-195
        return self._q

    def GetMotorVelocities(self):                   # :197-207
        return self._qd

    def GetMotorTorques(self):                      # :209-216 (clipped PD torque of the last substep)
        return self._env._views["tau_motor"].t()

    def GetSpringTorques(self):
        return self._env._views["tau_spring"].t()

    def GetContactInfo(self):                       # :224-258
        c = self._env._views["contact"]
        in_contact = torch.stack([(c >> k) & 1 for k in range(4)], dim=-1)
        forces = self._env._views["foot_force"].t() * in_contact
        return in_contact.sum(-1), c >> 8, forces, in_contact

    def _is_flying(self):                           # :260-262
        return (self._env._views["contact"] & 15) == 0

    # --- kinematics (kernels K3)
    def _fk_all(self, q=None, qd=None):
        env = self._env
        q = (self._q if q is None else q).contiguous()
        n = q.shape[0]
        pos = torch.empty(n, 12, device=q.device)
        jac = torch.empty(n, 4, 3, 3, device=q.device)
        vel = torch.empty(n, 12, device=q.device) if qd is not None else None
        qdc = qd.contiguous() if qd is not None else None
        _lib.check(env._L.qs_fk_jacobian(_p(q), _p(qdc), _p(pos), _p(jac), _p(vel), n, _stream_ptr(env.device)))
        return pos, jac, vel

    def ComputeJacobianAndPosition(self, legID):    # :394-397
        pos, jac, _ = self._fk_all()
        return jac[:, legID], pos[:, 3 * legID:3 * legID + 3]

    def ComputeInverseKinematics(self, legID, xyz_coord):   # :399-438
        env = self._env
        xyz = torch.as_tensor(xyz_coord, dtype=torch.float32, device=env.device)
        if xyz.dim() == 1:
            xyz = xyz.expand(env.num_envs, 3)
        full = torch.zeros(xyz.shape[0], 12, device=env.device)
        full[:, 3 * legID:3 * legID + 3] = xyz
        out = torch.empty_like(full)
        _lib.check(env._L.qs_ik(_p(full), _p(out), full.shape[0], _stream_ptr(env.device)))
        return out[:, 3 * legID:3 * legID + 3]

    def ComputeFeetPosAndVel(self):                 # :440-449
        pos, _, vel = self._fk_all(qd=self._qd)
        return pos, vel

    # --- per-env motor / spring parameters (runtime, quadruped.py:720-742, landing_wrapper.py:21-33)
    def set_motor_gains(self, kp, kd, env_ids=None):
        v = self._env._views
        kp = torch.as_tensor(kp, dtype=torch.float32, device=self._env.device).expand(12)
        kd = torch.as_tensor(kd, dtype=torch.float32, device=self._env.device).expand(12)
        if env_ids is None:
            v["kp"][:] = kp[:, None]
            v["kd"][:] = kd[:, None]
            v["custom_gains"][:] = 1
        else:
            v["kp"][:, env_ids] = kp[:, None]
            v["kd"][:, env_ids] = kd[:, None]
            v["custom_gains"][env_ids] = 1

    def get_spring_nominal_params(self):
        sp = self._env._views["spring"]
        return sp[0:3].t(), sp[3:6].t(), sp[6:9].t()

    # --- mass randomizer read-outs (quadruped.py:685-718): the current episode's draw, zero-copy views
    def GetLegMasses(self):
        """[N, 3] hip, thigh, calf link mass (the same for the four legs, env_randomizer.py:62-71)"""
        return self._env._views["mass_draw"][0:3].t()

    def GetBaseMass(self):
        return self._env._views["mass_draw"][3]

    def get_offset_mass_value(self):
        return self._env._views["mass_draw"][4]

    def get_offset_mass_position(self):
        return self._env._views["mass_draw"][5:8].t()

    def set_masses(self, leg_masses=None, base_mass=None, offset_mass=None, offset_position=None):
        """SetLegMasses ([N, 3] or [3]: hip, thigh, calf), SetBaseMass, _add_base_mass_offset (quadruped.py:744-819) for
        the current episode; needs a mass randomizer mode (the next reset draws again)."""
        v, dev = self._env._views["mass_draw"], self._env.device
        f = lambda x: torch.as_tensor(x, dtype=torch.float32, device=dev)
        if leg_masses is not None:
            v[0:3] = f(leg_masses).reshape(-1, 3).t().expand(3, self._env.num_envs)
        if base_mass is not None:
            v[3] = f(base_mass)
        if offset_mass is not None:
            v[4] = f(offset_mass)
        if offset_position is not None:
            v[5:8] = f(offset_position).reshape(-1, 3).t().expand(3, self._env.num_envs)
        _lib.check(self._env._L.qs_apply_masses(self._env._h, _stream_ptr(dev)))

    def set_spring_stiffness(self, stiffness):
        self._env._views["spring"][0:3] = torch.as_tensor(stiffness, dtype=torch.float32, device=self._env.device).view(3, -1)

    def set_spring_damping(self, damping):
        self._env._views["spring"][3:6] = torch.as_tensor(damping, dtype=torch.float32, device=self._env.device).view(3, -1)

    def set_spring_rest_angles(self, rest):
        self._env._views["spring"][6:9] = torch.as_tensor(rest, dtype=torch.float32, device=self._env.device).view(3, -1)

    # --- external push on the base (quadruped.py:338-343), applied tick by tick inside the step kernels
    def apply_external_force(self, force, position=None, n_ticks=1, env_ids=None):
        """Push the base of the envs `env_ids` (indices, a bool mask of [N], or None for every env) with `force` ([3] or
        [k, 3], world frame, N) at `position` ([3] or [k, 3], base frame from GetBasePosition, m; default the base
        position) for the next `n_ticks` physics ticks (int or [k] ints >= 0; a control step is action_repeat ticks).

        In every tick it lasts, the push is Bullet's applyExternalForce(robot, -1, force, pos + R position, WORLD_FRAME)
        made before that stepSimulation (qs_set_external_force has the full rule).  The count runs down by the ticks each
        step runs; an episode end under auto_reset and a reset of the env set it to 0.  A call overwrites the selected
        envs' force, point and count (n_ticks=0 cancels): unlike Bullet, where the calls made before one stepSimulation
        add up.  The first call attaches the library's push buffers (clear_external_force detaches them)."""
        env = self._env
        dev, n = env.device, env.num_envs
        if env_ids is None:
            ids = torch.arange(n)
        else:
            ids = torch.as_tensor(env_ids).cpu()
            if ids.dtype == torch.bool:
                if ids.shape != (n,):
                    raise ValueError(f"a bool env_ids mask must have shape ({n},), got {tuple(ids.shape)}")
                ids = ids.nonzero().flatten()
            elif ids.dtype in (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8) and ids.dim() <= 1:
                ids = ids.reshape(-1).long()
                if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= n):
                    raise ValueError(f"env_ids must lie in [0, {n})")
                if ids.unique().numel() != ids.numel():
                    raise ValueError("env_ids must be distinct")
            else:
                raise ValueError(f"env_ids must be indices or a bool mask, got {ids.dtype} of shape {tuple(ids.shape)}")
        k = ids.numel()

        def rows(x, name):
            t = torch.as_tensor(x, dtype=torch.float64).cpu()
            if t.shape == (3,):
                t = t.expand(k, 3)
            if t.shape != (k, 3):
                raise ValueError(f"{name} must have shape (3,) or ({k}, 3), got {tuple(t.shape)}")
            if not bool(torch.isfinite(t).all()):
                raise ValueError(f"{name} must be finite")
            return t.to(torch.float32)

        f = rows(force, "force")
        p = rows(torch.zeros(3) if position is None else position, "position")
        nt = torch.as_tensor(n_ticks).cpu()
        if nt.dtype.is_floating_point or nt.dtype == torch.bool or nt.dtype.is_complex:
            raise ValueError(f"n_ticks must be integers, got {nt.dtype}")
        if nt.dim() == 0:
            nt = nt.expand(k)
        if nt.shape != (k,):
            raise ValueError(f"n_ticks must be an int or have shape ({k},), got {tuple(nt.shape)}")
        if k and (int(nt.min()) < 0 or int(nt.max()) > 2**31 - 1):
            raise ValueError("n_ticks must lie in [0, 2**31)")
        if getattr(self, "_ext_ticks", None) is None:
            wrench = torch.zeros(_lib.QS_EXT_DIM, n, device=dev)
            ticks = torch.zeros(n, dtype=torch.int32, device=dev)
            _lib.check(env._L.qs_set_external_force(env._h, _p(wrench), _p(ticks)))
            self._ext_wrench, self._ext_ticks = wrench, ticks   # the library reads and counts them down: keep them alive
        if k == 0:
            return
        ids = ids.to(dev)
        self._ext_wrench[0:3, ids] = f.t().to(dev)
        self._ext_wrench[3:6, ids] = p.t().to(dev)
        self._ext_ticks[ids] = nt.to(device=dev, dtype=torch.int32)

    def get_external_force(self):
        """(force [N, 3], position [N, 3], ticks_left [N] int32): views of the attached push buffers (None when none is
        attached).  ticks_left reads what the steps enqueued so far leave."""
        if getattr(self, "_ext_ticks", None) is None:
            return None
        return self._ext_wrench[0:3].t(), self._ext_wrench[3:6].t(), self._ext_ticks

    def clear_external_force(self):
        """Detach the push buffers: every later step runs the kernels of an env that was never pushed."""
        env = self._env
        _lib.check(env._L.qs_set_external_force(env._h, None, None))
        self._ext_wrench = self._ext_ticks = None


class _ActionInterface:
    """control_interface/interface_base.py + motor_interface.py on batches."""

    def __init__(self, env):
        self._env = env
        c = env._robot_config
        self._motor_control_mode = env._motor_control_mode
        self._motor_control_mode_ROB = "TORQUE" if env._motor_control_mode == "TORQUE" else "PD"
        self._action_space_mode = env._action_space_mode
        if env._motor_control_mode == "CARTESIAN_PD":
            self._lower_lim, self._upper_lim = c.RL_LOWER_CARTESIAN_POS.copy(), c.RL_UPPER_CARTESIAN_POS.copy()
            self._init_pose, self._settling_pose, self._landing_pose = (
                c.NOMINAL_FOOT_POS_LEG_FRAME, c.CARTESIAN_SETTLING_POSE, c.CARTESIAN_LANDING_POSE)
            self._symm_idx = 1
        elif env._motor_control_mode == "PD":
            self._lower_lim, self._upper_lim = c.RL_LOWER_ANGLE_JOINT.copy(), c.RL_UPPER_ANGLE_JOINT.copy()
            if env.task_env == "BACKFLIP":              # motor_interface.py:20-22
                self._upper_lim[[7, 10]] = np.pi / 2
            self._init_pose, self._settling_pose, self._landing_pose = (
                c.INIT_MOTOR_ANGLES, c.ANGLE_SETTLING_POSE, c.ANGLE_LANDING_POSE)
            self._symm_idx = 0
        else:
            self._lower_lim, self._upper_lim = -c.TORQUE_LIMITS, c.TORQUE_LIMITS
            self._init_pose = np.zeros(12)
            self._settling_pose = self._landing_pose = None
            self._symm_idx = 0

    def get_action_space_mode(self):
        return self._action_space_mode

    def get_action_space_dim(self):
        return self._env.action_dim

    def get_motor_control_mode(self):
        return self._motor_control_mode

    def get_init_pose(self):
        return self._init_pose

    def get_landing_pose(self):
        return self._landing_pose

    def get_settling_pose(self):
        return self._settling_pose

    def _transform_action_to_motor_command(self, action):   # interface_base.py:162-164
        env = self._env
        a = torch.as_tensor(action, dtype=torch.float32, device=env.device)
        single = a.dim() == 1
        a = a.view(-1, env.action_dim).contiguous()
        out = torch.empty(a.shape[0], 12, device=env.device)
        _lib.check(env._L.qs_action_to_command(C.byref(env._cfg), _p(a), _p(out), a.shape[0], _stream_ptr(env.device)))
        return out[0] if single else out

    def _convert_to_actual_action_space(self, action12):    # action_interface.py:17-18,41-44,67-74
        m = self._action_space_mode
        if m == "DEFAULT":
            return action12
        fr, rr = action12[..., 0:3], action12[..., 6:9]
        if m == "SYMMETRIC":
            return torch.cat([fr, rr], dim=-1)
        keep = [j for j in range(3) if j != self._symm_idx]
        return torch.cat([fr[..., keep], rr[..., keep]], dim=-1)

    def _transform_motor_command_to_action(self, command):  # interface_base.py:92-100,166-168
        env = self._env
        lo = torch.as_tensor(self._lower_lim, dtype=torch.float32, device=env.device)
        hi = torch.as_tensor(self._upper_lim, dtype=torch.float32, device=env.device)
        c = torch.as_tensor(command, dtype=torch.float32, device=env.device)
        c = torch.minimum(torch.maximum(c, lo), hi)
        a = (-1 + 2 * (c - lo) / (hi - lo)).clamp(-1, 1)
        return self._convert_to_actual_action_space(a)

    def get_landing_action(self):
        return self._transform_motor_command_to_action(self.get_landing_pose())

    def get_init_action(self):
        return self._transform_motor_command_to_action(self.get_init_pose())

    def get_last_reference(self):
        return self._transform_action_to_motor_command(self._env._last_action[:, :self._env.action_dim])


_TASK_FIELDS = {  # reference attribute name -> task-state slot (csrc/qs_types.h TaskSlot)
    "_switched_controller": 0, "_all_feet_in_the_air": 1, "_time_take_off": 2, "_init_height": 6,
    "_max_flight_time": 8, "_max_forward_distance": 9, "_max_pitch": 10, "_relative_max_height": 11,
    "_max_delta_x": 12, "_max_height": 13, "max_pitch": 14, "old_fwd": 15, "actual_fwd": 16,
    # continuous-jumping tasks (task_base.py:222-400)
    "is_jumping": 29, "cumulative_fwd": 30, "cumulative_flight_time": 31, "first_jump": 32, "jump_counter": 33,
    "good_jump_counter": 34, "max_jump_height": 35, "end_jump": 41,
}
_DEMO_TASK_FIELDS = {"demo_counter": 29, "delta_demo": 30}   # imitation tasks (task_base.py:169-220) reuse those rows


class _Task:
    """Read access to the per-env task state the kernels maintain
    (tasks/task_base.py:40-59 attribute names)."""

    def __init__(self, env):
        self._env = env

    def __getattr__(self, name):
        if name in _DEMO_TASK_FIELDS and self._env.task_env.endswith("_DEMO"):
            return self._env._views["task"][self._demo_row(name)]
        if name in _TASK_FIELDS:
            return self._env._views["task"][_TASK_FIELDS[name]]
        raise AttributeError(name)

    def _demo_row(self, name):
        # TaskJumpingDemo2 keeps the continuous-jumping rows: its two imitation rows come after them (QS_TS_DEMO2_COUNTER)
        off = 13 if self._env.task_env == "CONTINUOUS_JUMPING_FORWARD_DEMO" else 0
        return _DEMO_TASK_FIELDS[name] + off

    def set_demo_counter(self, value, mask=None):    # task_base.py:218-219, 451-452
        row = self._env._views["task"][self._demo_row("demo_counter")]
        v = torch.as_tensor(value, dtype=torch.float32, device=self._env.device)
        if mask is None:
            row[:] = v
        else:
            row[mask] = v

    @property
    def _robot_pose_take_off(self):
        return self._env._views["task"][3:6].t()

    def is_switched_controller(self):
        return self._env._views["task"][0] != 0

    def get_jumping(self):                           # task_base.py:277,355
        return self._env._views["task"][29] != 0

    def get_cumulative_fwd(self):                    # task_base.py:358 (sum of the per-jump fwd array)
        return self._env._views["task"][36]

    def get_avg_performance(self):                   # task_base.py:392-399 (zero-padded to >= 3 jumps)
        t = self._env._views["task"]
        return t[38] / t[33].clamp_min(3)

    def get_entropy_fwd(self):                       # task_base.py:376-383
        t = self._env._views["task"]
        n, S, Q = t[33], t[36], t[37]
        ent = (torch.log2(S.clamp_min(1e-30)) - Q / S.clamp_min(1e-30)) / torch.log2(n.clamp_min(3))
        return torch.where((n > 0) & (S >= 0.05), ent, torch.zeros_like(ent))

    def compute_jumping_distance(self):              # task_base.py:109-116
        t = self._env._views["task"]
        pos = self._env.robot.GetBasePosition()
        yaw = t[7]
        dx, dy = pos[:, 0] - t[3], pos[:, 1] - t[4]
        return (torch.cos(yaw) * dx - torch.sin(yaw) * dy).clamp_min(0)


class BatchedQuadrupedGymEnv:
    """QuadrupedGymEnv for `num_envs` robots on one GPU (same kwargs, same keys)."""

    metadata = {"render.modes": ["rgb_array"]}

    def __init__(
        self,
        num_envs=1,
        device="cuda:0",
        isRLGymInterface=True,
        time_step=0.001,
        action_repeat=10,
        motor_control_mode="PD",
        task_env="NO_TASK",
        observation_space_mode="ENCODER",
        action_space_mode="SYMMETRIC",
        on_rack=False,
        render=False,
        enable_springs=False,
        enable_action_interpolation=False,
        enable_action_filter=False,
        env_randomizer_mode="GROUND_RANDOMIZER",
        camera_mode="CLASSIC",
        curriculum_level=0.0,
        verbose=0,
        # batched-only options
        seed=0,
        env_id_offset=0,
        auto_reset=True,
        enable_noise=True,
        solver=None,
        block_size=0,
        landing_wrapper=None,
        go_to_rest_wrapper=False,
    ):
        """landing_wrapper: None, "LandingWrapper" (env/wrappers/landing_wrapper.py:18-69), "LandingWrapper2"
        (landing_wrapper_2.py:39-78), "LandingWrapperContinuous" (landing_wrapper_continuous.py:38-70),
        "LandingWrapperBackflip" or "LandingWrapperBackflip2" (landing_wrapper_backflip*.py:47-80).  The reference wraps the env and loops env.step inside one wrapper step; here
        the same controller runs per env inside the step kernel: every call is one control step, envs whose
        controller is scripted (infos["landing_mode"] != 0 and != 3) ignore the action they are given.
        go_to_rest_wrapper: GoToRestWrapper (env/wrappers/go_to_rest_wrapper.py:8-95) around that: once the robot has
        jumped, stands on its four feet and its base rises again, the env ramps to the init action on gains 60 / 0.8
        (60 / 1.5 without springs) until the episode ends (infos["rest_active"])."""
        if render or on_rack:
            raise ValueError("render=True (the pybullet GUI) and on_rack are not provided; camera images come from "
                             "env.render('rgb_array') and env.render_images()")
        self._L = _lib.lib()
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedQuadrupedGymEnv needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device)
        self.num_envs = int(num_envs)
        self.verbose = verbose
        self._enable_springs = bool(enable_springs)
        self._robot_config = go1_config(self._enable_springs)
        self._isRLGymInterface = bool(isRLGymInterface)
        self.sim_time_step = time_step
        self._action_repeat = int(action_repeat)
        self.env_time_step = self._action_repeat * self.sim_time_step
        self._on_rack, self._is_render = False, False
        # no-op in the reference as well (step() overwrites _last_action first, quadruped_gym_env.py:187-205,229-234)
        self._enable_action_interpolation = bool(enable_action_interpolation)
        self._enable_action_filter = bool(enable_action_filter)
        self._num_bullet_solver_iterations = int(300 / action_repeat)
        self._MAX_EP_LEN = EPISODE_LENGTH
        self._settling_steps = 2500
        self.task_env = task_env
        self._motor_control_mode = motor_control_mode
        self._action_space_mode = action_space_mode
        self._observation_space_mode = observation_space_mode
        self._env_randomizer_mode = env_randomizer_mode
        self.curriculum_level = 0.0

        cfg = _lib.QsConfig()
        self._L.qs_default_config(C.byref(cfg))
        cfg.enable_springs = int(enable_springs)
        cfg.control_mode = MotorInterfaceCollection().get_el(motor_control_mode)
        cfg.action_mode = ActionInterfaceCollection().get_el(action_space_mode)
        cfg.task = TaskCollection().get_el(task_env)
        cfg.obs_mode = SensorCollection().get_el(observation_space_mode)
        rnd = EnvRandomizerCollection().get_el(env_randomizer_mode)
        # env_randomizer_collection.py:15-21: every mode but NO_RANDOMIZER starts with the ground randomizer
        cfg.ground_randomizer = int(rnd != 1)
        cfg.spring_randomizer = int(rnd in (2, 4, 5))
        cfg.mass_randomizer = int(rnd in (3, 4, 5))
        if rnd == 5:
            # *Curriculum randomizers (env_randomizer.py:125-262): ranges interpolated by the level, which the env
            # raises once at construction (quadruped_gym_env.py:147-150)
            lvl = float(np.clip(curriculum_level, 0.0, 1.0))
            self.curriculum_level = lvl
            mix = lambda lo, hi: (1.0 - lvl) * lo + lvl * hi
            cfg.rand_leg_mass_err = mix(0.1, 0.2)
            cfg.rand_payload_max = mix(1.0, 4.0)
            cfg.rand_payload_pos = (C.c_float * 3)(mix(0.1, 0.2), 0.0, mix(0.1, 0.2))
            cfg.rand_spring_err = mix(0.1, 0.3)
        cfg.action_repeat = self._action_repeat
        cfg.is_rl_interface = int(isRLGymInterface)
        cfg.enable_action_filter = int(enable_action_filter)
        cfg.settling_steps = self._settling_steps
        cfg.enable_noise = int(enable_noise)
        cfg.auto_reset = int(auto_reset)
        cfg.seed = int(seed)
        cfg.env_id_offset = int(env_id_offset)
        cfg.time_step = float(time_step)
        cfg.max_episode_time = float(EPISODE_LENGTH)
        cfg.block_size = int(block_size)
        try:
            cfg.landing_mode = {None: 0, "LandingWrapper": 1, "LandingWrapper2": 2, "LandingWrapperContinuous": 3,
                                "LandingWrapperBackflip": 4, "LandingWrapperBackflip2": 5}[landing_wrapper]
        except KeyError:
            raise ValueError(f"the landing wrapper {landing_wrapper} is not implemented yet.") from None
        cfg.rest_mode = int(bool(go_to_rest_wrapper))
        for k, v in (solver or {}).items():
            if not hasattr(cfg, k):
                raise ValueError(f"unknown solver parameter {k}")
            setattr(cfg, k, v)
        self._cfg = cfg
        self._auto_reset = bool(auto_reset)

        h = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _lib.check(self._L.qs_create(C.byref(cfg), self.num_envs, idx, C.byref(h)))
        self._h = h
        self.action_dim = self._L.qs_action_dim(h)
        self.obs_dim = self._L.qs_obs_dim(h)
        self.setupActionSpace(self.action_dim)
        self.setupObservationSpace()

        ptrs = _lib.QsStatePtrs()
        _lib.check(self._L.qs_get_state_ptrs(h, C.byref(ptrs)))
        n, dev = self.num_envs, self.device
        self._views = {
            "state": _view(ptrs.state, (37, n), "<f4", dev), "tau_motor": _view(ptrs.tau_motor, (12, n), "<f4", dev),
            "tau_spring": _view(ptrs.tau_spring, (12, n), "<f4", dev), "kp": _view(ptrs.kp, (12, n), "<f4", dev),
            "kd": _view(ptrs.kd, (12, n), "<f4", dev), "spring": _view(ptrs.spring, (9, n), "<f4", dev),
            "mu": _view(ptrs.mu, (n,), "<f4", dev), "foot_force": _view(ptrs.foot_force, (4, n), "<f4", dev),
            "contact": _view(ptrs.contact, (n,), "<i4", dev), "task": _view(ptrs.task, (_lib.QS_TASK_DIM, n), "<f4", dev),
            "last_action": _view(ptrs.last_action, (12, n), "<f4", dev),
            "sim_steps": _view(ptrs.sim_steps, (n,), "<i4", dev), "env_steps": _view(ptrs.env_steps, (n,), "<i4", dev),
            "ep_return": _view(ptrs.ep_return, (n,), "<f4", dev),
            "custom_gains": _view(ptrs.custom_gains, (n,), "|u1", dev),
            "land_mode": _view(ptrs.land_mode, (n,), "<i4", dev),
            "rest_active": _view(ptrs.rest_active, (n,), "<i4", dev), "rest": _view(ptrs.rest, (14, n), "<f4", dev),
            "mass_draw": _view(ptrs.mass_draw, (8, n), "<f4", dev), "filt": _view(ptrs.filt, (4, 12, n), "<f4", dev),
            "work": _view(ptrs.work, (3, n), "<i4", dev),
        }
        self.robot = BatchedQuadruped(self)
        self.task = _Task(self)
        self._ac_interface = _ActionInterface(self)
        self._obs = torch.zeros(n, self.obs_dim, device=dev)
        self._reward = torch.zeros(n, device=dev)
        self._done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._trunc = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._last_host_obs = None      # where the latest observation lives when it came through the host path
        self.sub_step_callback = None
        self._trace = self._trace_ids = None
        self.robot_desired_state = None
        if self.verbose > 0:
            self.print_info()

    # ------------------------------------------------------------------ spaces (quadruped_gym_env.py:160-182)
    def setupObservationSpace(self):
        self._obs_layout, hi, lo = observation_layout(self._observation_space_mode, self._robot_config)
        if self.task_env == "BACKFLIP" and self._motor_control_mode == "PD":
            pass  # JOINT_ANGLES_HIGH aliases the mutated RL_UPPER_ANGLE_JOINT upstream (App. D.7); bounds only
        self.observation_space = Box(lo - OBSERVATION_EPS, hi + OBSERVATION_EPS, dtype=np.float32)

    def setupActionSpace(self, action_dim):
        action_high = np.array([1] * action_dim)
        self.action_space = Box(-action_high, action_high, dtype=np.float32)

    # ------------------------------------------------------------------ reset / step
    def reset(self, mask=None):
        """QuadrupedGymEnv.reset (quadruped_gym_env.py:278-297) for all envs, or for
        the envs selected by a bool/uint8 mask [N].  Returns obs [N, O]."""
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        if self._last_host_obs is not None:   # a partial reset leaves the other rows as the last (host-path) step left them
            self._obs.copy_(torch.as_tensor(self._last_host_obs, device=self.device))
            self._last_host_obs = None
        _lib.check(self._L.qs_reset(self._h, _p(m), _p(self._obs), _stream_ptr(self.device)))
        return self._obs

    def step(self, action):
        """QuadrupedGymEnv.step (quadruped_gym_env.py:227-256): action [N, A] ->
        (obs [N, O], reward [N], done [N] bool, infos).  With auto_reset the obs row
        of a finished env is the first observation of its next episode."""
        a = torch.as_tensor(action, dtype=torch.float32, device=self.device)
        if a.dim() == 1:
            a = a.expand(self.num_envs, -1)
        if a.shape != (self.num_envs, self.action_dim):
            raise ValueError(f"action must have shape {(self.num_envs, self.action_dim)}, got {tuple(a.shape)}")
        a = a.contiguous()
        _lib.check(self._L.qs_step(self._h, _p(a), _p(self._obs), _p(self._reward), _p(self._done), _p(self._trunc),
                                   _stream_ptr(self.device)))
        self._last_host_obs = None
        infos = {"TimeLimit.truncated": self._trunc.bool()}
        if self._cfg.landing_mode:
            infos["landing_mode"] = self._views["land_mode"]
        if self._cfg.rest_mode:
            infos["rest_active"] = self._views["rest_active"]
        return self._obs, self._reward, self._done.bool(), infos

    def reset_to_state(self, states, mask=None):
        """reset() with `set_robot_desired_state(states)` (quadruped_gym_env.py:288-289,401): the selected envs start a new
        episode from rows of states [N, 37] (pos3 quat4 lin_vel3 ang_vel3 q12 qd12), without the settle."""
        s = torch.as_tensor(states, dtype=torch.float32, device=self.device).contiguous()
        if s.shape != (self.num_envs, 37):
            raise ValueError(f"states must have shape {(self.num_envs, 37)}")
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        _lib.check(self._L.qs_reset_to_state(self._h, _p(m), _p(s), _p(self._obs), _stream_ptr(self.device)))
        return self._obs

    def get_last_filtered_action(self):
        """quadruped_gym_env.py:385-387: the filter's last output; zeros when the filter is off (the reference only
        assigns it inside `if self._enable_action_filter`, :232-234)"""
        if self._enable_action_filter:
            return self._views["filt"][2].t()[:, :self.action_dim]
        return torch.zeros(self.num_envs, self.action_dim, device=self.device)

    def set_demo(self, demo, rows_are_actions=False):
        """the demonstration of the *_DEMO tasks (TaskJumpingDemo.demo_list, tasks/task_base.py:169-176): an array of
        GetDemonstrationWrapper rows [L, A + 38] (or of bare actions [L, A])"""
        d = np.asarray(demo, dtype=np.float32)
        a = np.ascontiguousarray(d if rows_are_actions else d[:, :self.action_dim])
        if a.ndim != 2 or a.shape[1] != self.action_dim:
            raise ValueError(f"demonstration rows must start with {self.action_dim} action values")
        self.demo_list, self.demo_length = d, int(a.shape[0])
        _lib.check(self._L.qs_set_demo(self._h, a.ctypes.data_as(C.c_void_p), int(a.shape[0])))

    def set_terminal_obs_buffer(self, buf):
        """device tensor [N, O] (or None) that receives the last observation of every env whose episode ends inside
        step() under auto_reset: SB3's infos["terminal_observation"] (qs_set_terminal_obs)"""
        if buf is not None:
            if buf.shape != (self.num_envs, self.obs_dim) or buf.dtype != torch.float32 or not buf.is_contiguous() \
                    or buf.device.type != "cuda":
                raise ValueError(f"terminal-obs buffer must be a contiguous float32 cuda tensor {(self.num_envs, self.obs_dim)}")
        self._term_obs = buf        # keep it alive
        _lib.check(self._L.qs_set_terminal_obs(self._h, _p(buf)))

    def reset_host(self, mask_np=None):
        """numpy twin of reset(): returns the host observation array [N, O]"""
        out = np.zeros((self.num_envs, self.obs_dim), np.float32)
        m = None
        if mask_np is not None:
            # rows of the envs that are NOT reset keep the observation of the last step, wherever that step left it:
            # the host array step_host / reset_host returned, or the device tensor of step() / reset()
            m = np.ascontiguousarray(mask_np, dtype=np.uint8)
            out[:] = self._last_host_obs if self._last_host_obs is not None else self._obs.cpu().numpy()
        _lib.check(self._L.qs_reset_host(self._h, m.ctypes.data_as(C.c_void_p) if m is not None else None,
                                         out.ctypes.data_as(C.c_void_p), _stream_ptr(self.device)))
        self._last_host_obs = out
        return out

    def step_host(self, action_np, out=None):
        """End-to-end numpy path (what an SB3 VecEnv adapter calls): host action
        [N, A] float32 -> host (obs, reward, done, truncated); copies are inside."""
        a = np.ascontiguousarray(action_np, dtype=np.float32)
        if out is None:
            out = (np.empty((self.num_envs, self.obs_dim), np.float32), np.empty(self.num_envs, np.float32),
                   np.empty(self.num_envs, np.uint8), np.empty(self.num_envs, np.uint8))
        o, r, d, t = out
        _lib.check(self._L.qs_step_host(self._h, a.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p),
                                        r.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p),
                                        t.ctypes.data_as(C.c_void_p), _stream_ptr(self.device)))
        self._last_host_obs = o
        return out

    def close(self):
        if getattr(self, "_h", None):
            self._L.qs_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ state I/O (checkpoint / parity harness)
    def get_state(self):
        out = torch.empty(self.num_envs, 37, device=self.device)
        _lib.check(self._L.qs_get_state(self._h, _p(out), _stream_ptr(self.device)))
        return out

    def set_state(self, state):
        s = torch.as_tensor(state, dtype=torch.float32, device=self.device).contiguous()
        assert s.shape == (self.num_envs, 37)
        _lib.check(self._L.qs_set_state(self._h, _p(s), _stream_ptr(self.device)))

    def set_robot_desired_state(self, state):        # quadruped_gym_env.py:401
        self.set_state(state)

    def debug_ticks(self, tau, n_ticks=1, use_f64=False):
        t = torch.as_tensor(tau, dtype=torch.float32, device=self.device).contiguous()
        assert t.shape == (self.num_envs, 12)
        _lib.check(self._L.qs_debug_ticks(self._h, _p(t), int(n_ticks), int(use_f64), _stream_ptr(self.device)))

    # ------------------------------------------------------------------ camera images (quadruped_springs_b200/render.py)
    def render(self, mode="rgb_array"):
        """QuadrupedGymEnv.render: env 0's image of the follow camera as a numpy uint8 [360, 480, 3] for "rgb_array",
        an empty array for any other mode (there is no GUI)."""
        if mode != "rgb_array":
            return np.array([])
        return self.render_images([0])["rgb"][0].cpu().numpy()

    def render_images(self, env_ids=None, width=480, height=360, camera=None, depth=False, segmentation=False):
        """Camera images of the envs `env_ids` (all when None) in their current state: render.render_states of
        get_state()[env_ids] through `camera` ([k, 32] or [32], pybullet's view then projection matrix) or, by default,
        the follow camera of each robot.  Returns a dict of CUDA tensors ("rgb", and "depth" / "segmentation" when
        asked).  Reads the state only: no env value changes."""
        from .render import follow_cameras, render_states
        states = self.get_state()
        if env_ids is not None:
            states = states[torch.as_tensor(env_ids, dtype=torch.long, device=self.device)]
        cams = camera if camera is not None else follow_cameras(states[:, :3], width, height)
        return render_states(states, cams, width, height, rgb=True, depth=depth, segmentation=segmentation)

    # ------------------------------------------------------------------ getters (quadruped_gym_env.py:343-426)
    def get_observation(self, with_noise=True):
        out = torch.empty(self.num_envs, self.obs_dim, device=self.device)
        _lib.check(self._L.qs_observe(self._h, _p(out), int(with_noise and self._cfg.enable_noise), _stream_ptr(self.device)))
        return out

    def get_observation_dict(self, obs=None):
        """the reference returns a dict keyed by sensor name (sensor.py:107-111)"""
        obs = self._obs if obs is None else obs
        return {name: obs[:, a:b] for name, a, b in self._obs_layout}

    def get_sim_time(self):
        return self._views["sim_steps"].to(torch.float64) * self.sim_time_step

    def get_motor_control_mode(self):
        return self._motor_control_mode

    def get_robot_config(self):
        return self._robot_config

    def are_springs_enabled(self):
        return self._enable_springs

    def get_init_pose(self):
        return self._ac_interface.get_init_pose()

    def get_landing_action(self):
        return self._ac_interface.get_landing_action()

    @property
    def _last_action(self):
        return self._views["last_action"].t()

    def get_last_action(self):
        return self._last_action[:, :self.action_dim]

    def get_observation_space_mode(self):
        return self._observation_space_mode

    def get_curriculum_level(self):
        return self.curriculum_level

    def get_randomizer_mode(self):
        return self._env_randomizer_mode

    def get_ac_interface(self):
        return self._ac_interface

    def set_sub_step_callback(self, callback):
        raise NotImplementedError("per-substep Python callbacks cannot run inside the fused step kernel "
                                  "(SURVEY.md section 5); set_substep_trace records every substep instead")

    def set_substep_trace(self, env_ids):
        """Per-substep trace of the envs `env_ids` (qs_set_substep_trace): what a sub_step_callback reading the Quadruped
        accessors after every stepSimulation would see (quadruped_gym_env.py:222-223).  Returns the float32 tensor
        [action_repeat, 66, len(env_ids)] that every later step() rewrites: row t = the values after tick t of that step,
        column j = env env_ids[j]; rows 0-36 state (get_state order), 37-48 motor torque, 49-60 spring torque, 61-64 foot
        normal force (0 off contact), 65 contact word (mask | invalid << 8, exact as a float).  Under auto_reset, the
        rows of an env whose episode ended in the step are the ticks of that episode.  None clears the trace; the last
        buffer is then left as it is.  See substep.SubstepRecorder for a recording over many steps."""
        if env_ids is None:
            _lib.check(self._L.qs_set_substep_trace(self._h, None, 0, None))
            self._trace = self._trace_ids = None
            return None
        ids = torch.as_tensor(env_ids)
        if ids.dtype not in (torch.int32, torch.int64) or ids.dim() != 1:
            raise ValueError(f"env_ids must be a 1-D integer sequence, got {ids.dtype} of shape {tuple(ids.shape)}")
        host = ids.cpu()
        if host.numel() == 0:
            raise ValueError("env_ids is empty (set_substep_trace(None) clears the trace)")
        if int(host.min()) < 0 or int(host.max()) >= self.num_envs:
            raise ValueError(f"env_ids must lie in [0, {self.num_envs})")
        if host.unique().numel() != host.numel():
            raise ValueError("env_ids must be distinct")
        ids = ids.to(device=self.device, dtype=torch.int32).contiguous()
        buf = torch.full((self._action_repeat, _lib.QS_TRACE_DIM, ids.numel()), float("nan"), device=self.device)
        _lib.check(self._L.qs_set_substep_trace(self._h, _p(ids), ids.numel(), _p(buf)))
        self._trace, self._trace_ids = buf, ids      # the library writes into them: keep them alive
        return buf

    def rollout_stats(self):
        """per-shard statistics vector (kernel K5); see stats.gather_rollout_stats"""
        out = torch.zeros(_lib.QS_STATS_DIM, device=self.device)
        _lib.check(self._L.qs_reduce_stats(self._h, _p(out), _stream_ptr(self.device)))
        return out

    def print_info(self):
        print("\n*** Environment Info ***")
        print(f"task environment -> {self.task_env}")
        print(f"spring enabled -> {self._enable_springs}")
        print(f"low-pass action filter > {self._enable_action_filter}")
        print(f"sensors -> {self._observation_space_mode}")
        print(f"env randomizer -> {self._env_randomizer_mode}")
        print(f"num envs -> {self.num_envs} on {self.device}")
        print("")
