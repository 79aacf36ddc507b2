"""Recording of every physics tick over many control steps: the batched counterpart of the recording half of the
reference's MonitorState (utils/monitor_state.py:20-21,391-396), which patches step_simulation to sample the robot after
every stepSimulation.  Here the step kernels write each tick into the env's substep trace
(BatchedQuadrupedGymEnv.set_substep_trace) and the recorder copies it, device to device, after every step."""
import numpy as np
import torch

from ._lib import QS_TRACE_DIM

# rows of a trace column (include/qs_b200.h QS_TR_*): accessor name -> (first row, rows)
_ROWS = {
    "base_position": (0, 3), "base_orientation": (3, 4), "base_linear_velocity": (7, 3),
    "base_angular_velocity": (10, 3), "motor_angles": (13, 12), "motor_velocities": (25, 12),
    "motor_torques": (37, 12), "spring_torques": (49, 12), "feet_normal_forces": (61, 4),
}
_CONTACT_ROW = 65


class SubstepRecorder:
    """Every tick of `steps` control steps for the envs `env_ids`.

    `data` is [steps, action_repeat, 66, n] float32 on the env's device; the named views below are [recorded steps,
    action_repeat, n, k] (k dropped for scalars) and cover the steps recorded so far.  Step the env through
    `recorder.step(action)`: it reads the traced envs' tick counters, steps, and copies the step's trace."""

    def __init__(self, env, env_ids, steps):
        self.env = env
        self.trace = env.set_substep_trace(env_ids)
        self.env_ids = torch.as_tensor(env_ids).to(torch.int64)
        self.steps = int(steps)
        R, _, n = self.trace.shape
        dev = self.trace.device
        self.data = torch.full((self.steps, R, QS_TRACE_DIM, n), float("nan"), device=dev)
        self._ticks0 = torch.zeros(self.steps, n, dtype=torch.int64, device=dev)   # sim steps before each step
        self._dt = float(env.sim_time_step)
        self.count = 0

    def step(self, action):
        """env.step(action), then the copy of its trace; returns what env.step returns"""
        if self.count >= self.steps:
            raise RuntimeError(f"the recorder holds {self.steps} steps")
        self._ticks0[self.count] = self.env._views["sim_steps"][self.env_ids.to(self.trace.device)].to(torch.int64)
        out = self.env.step(action)
        self.data[self.count].copy_(self.trace)
        self.count += 1
        return out

    def _rows(self, first, k):
        return self.data[:self.count, :, first:first + k].transpose(-1, -2)

    def __getattr__(self, name):
        if name in _ROWS:
            return self._rows(*_ROWS[name])
        raise AttributeError(name)

    @property
    def _contact(self):
        return self.data[:self.count, :, _CONTACT_ROW].to(torch.int32)

    @property
    def feet_in_contact(self):
        """[steps, action_repeat, n, 4] bool (GetContactInfo's foot contact flags)"""
        c = self._contact
        return torch.stack([((c >> k) & 1).bool() for k in range(4)], dim=-1)

    @property
    def invalid_contacts(self):
        """[steps, action_repeat, n] number of non-foot contacts (GetContactInfo's invalid count)"""
        return self._contact >> 8

    @property
    def sim_time(self):
        """[steps, action_repeat, n] float64 episode time after each tick (the env's get_sim_time)"""
        R = self.data.shape[1]
        t = torch.arange(1, R + 1, device=self.data.device)
        return (self._ticks0[:self.count, None, :] + t[None, :, None]).to(torch.float64) * self._dt

    def save(self, path):
        """every view and the env ids to an .npz (numpy arrays)"""
        out = {name: getattr(self, name).cpu().numpy() for name in _ROWS}
        out.update(feet_in_contact=self.feet_in_contact.cpu().numpy(), invalid_contacts=self.invalid_contacts.cpu().numpy(),
                   sim_time=self.sim_time.cpu().numpy(), env_ids=self.env_ids.cpu().numpy())
        np.savez(path, **out)
