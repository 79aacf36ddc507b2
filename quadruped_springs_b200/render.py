"""Camera images of the robots, ray cast on the GPU (`qs_render`, include/qs_b200.h).

The reference's `QuadrupedGymEnv.render(mode="rgb_array")` returns a pybullet `getCameraImage` of a camera that follows
the robot, `utils/video_recording.py` turns such images into mp4s, and stable-baselines3's `VecVideoRecorder` calls
`VecEnv.get_images()`.  Here one kernel renders the collision shapes of any batch of states on the ground plane: RGB,
metric depth and pybullet's segmentation encoding.  What is drawn is what the contact code collides (no visual meshes;
the mass randomizer's payload block is not drawn).

* `compute_view_matrix_from_yaw_pitch_roll`, `compute_projection_matrix_fov` -- pybullet's camera matrices, batched.
* `follow_cameras`  -- the camera of the reference's `render()`.
* `render_states`   -- the one wrapper over `qs_render`: states [k, 37] and cameras -> dict of CUDA tensors.
* `tile_images`     -- stable-baselines3's `tile_images`, restated.
* `VideoRecorder`   -- follow-camera frames of chosen envs in a device buffer, written out as mp4 with cv2.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib

# The reference's render() camera.  Its values come from the pybullet_envs minitaur env that the reference's render()
# descends from (the reference source is not part of this project); only these defaults depend on them.
FOLLOW_DISTANCE = 1.0
FOLLOW_YAW = 0.0
FOLLOW_PITCH = -30.0
FOLLOW_FOV = 60.0
FOLLOW_NEAR = 0.1
FOLLOW_FAR = 100.0
RENDER_WIDTH = 480
RENDER_HEIGHT = 360


def _batch(x, k, device):
    t = torch.as_tensor(x, dtype=torch.float64, device=device)
    return t.expand(k) if t.dim() == 0 else t.reshape(k)


def compute_view_matrix_from_yaw_pitch_roll(target, distance, yaw, pitch, roll=0.0):
    """pybullet.computeViewMatrixFromYawPitchRoll(target, distance, yaw, pitch, roll, upAxisIndex=2) for a batch:
    target [k, 3] (or [3]), distance / yaw / pitch in degrees as numbers or [k] tensors -> [k, 16] float32, column-major
    like pybullet's list.  Bullet's b3ComputeViewMatrixFromYawPitchRoll rotates the eye offset (0, -distance, 0) and the
    up vector (0, 0, 1) by Rz(yaw) Rx(pitch) about the target; it sets roll to 0 whatever is passed, and so does this
    function.  With yaw 0 and pitch -30 the eye sits at target + distance (0, -cos 30, sin 30)."""
    del roll  # ignored by Bullet as well
    tgt = torch.as_tensor(target, dtype=torch.float64)
    tgt = tgt.reshape(-1, 3)
    k, dev = tgt.shape[0], tgt.device
    d = _batch(distance, k, dev)
    y = torch.deg2rad(_batch(yaw, k, dev))
    p = torch.deg2rad(_batch(pitch, k, dev))
    cy, sy, cp, sp = torch.cos(y), torch.sin(y), torch.cos(p), torch.sin(p)
    eye = tgt + torch.stack([d * cp * sy, -d * cp * cy, -d * sp], 1)
    up = torch.stack([sp * sy, -sp * cy, cp], 1)
    # b3ComputeViewMatrixFromPositions: the gluLookAt basis
    f = torch.nn.functional.normalize(tgt - eye, dim=1)
    u = torch.nn.functional.normalize(up, dim=1)
    s = torch.nn.functional.normalize(torch.cross(f, u, dim=1), dim=1)
    u = torch.cross(s, f, dim=1)
    V = torch.zeros(k, 4, 4, dtype=torch.float64, device=dev)   # V[:, col, row]: column-major flat
    V[:, 0:3, 0] = s
    V[:, 0:3, 1] = u
    V[:, 0:3, 2] = -f
    V[:, 3, 0] = -(s * eye).sum(1)
    V[:, 3, 1] = -(u * eye).sum(1)
    V[:, 3, 2] = (f * eye).sum(1)
    V[:, 3, 3] = 1.0
    return V.reshape(k, 16).to(torch.float32)


def compute_projection_matrix_fov(fov, aspect, near, far):
    """pybullet.computeProjectionMatrixFOV(fov, aspect, nearVal, farVal) (Bullet's b3ComputeProjectionMatrixFOV, the
    OpenGL perspective): [16] float32, column-major.  fov is the vertical field of view in degrees."""
    y = 1.0 / math.tan(math.radians(fov) / 2.0)
    P = np.zeros(16, dtype=np.float64)
    P[0] = y / aspect
    P[5] = y
    P[10] = (near + far) / (near - far)
    P[11] = -1.0
    P[14] = 2.0 * far * near / (near - far)
    return torch.tensor(P, dtype=torch.float32)


def follow_cameras(base_pos, width=RENDER_WIDTH, height=RENDER_HEIGHT, distance=FOLLOW_DISTANCE, yaw=FOLLOW_YAW,
                   pitch=FOLLOW_PITCH, fov=FOLLOW_FOV, near=FOLLOW_NEAR, far=FOLLOW_FAR):
    """The camera of the reference's render(): aimed at GetBasePosition() from `distance` at `yaw` / `pitch`, with a
    `fov` perspective of aspect width / height.  base_pos [k, 3] -> cameras [k, QS_CAM_DIM] on base_pos's device."""
    pos = torch.as_tensor(base_pos, dtype=torch.float32).reshape(-1, 3)
    V = compute_view_matrix_from_yaw_pitch_roll(pos, distance, yaw, pitch)
    P = compute_projection_matrix_fov(fov, width / height, near, far).to(pos.device)
    return torch.cat([V, P.expand(pos.shape[0], 16)], 1).contiguous()


def _launch(states, cameras, width, height, rgb, depth, seg):
    _lib.check(_lib.lib().qs_render(
        C.c_void_p(states.data_ptr()), C.c_void_p(cameras.data_ptr()), states.shape[0], int(width), int(height),
        *(C.c_void_p(t.data_ptr()) if t is not None else None for t in (rgb, depth, seg)),
        C.c_void_p(torch.cuda.current_stream(states.device).cuda_stream)))


def _inputs(states, cameras):
    if not (isinstance(states, torch.Tensor) and states.is_cuda):
        raise ValueError("states must be a CUDA tensor [k, 37] (there is no CPU renderer)")
    if states.dim() != 2 or states.shape[1] != _lib.QS_STATE_DIM:
        raise ValueError(f"states must have shape (k, {_lib.QS_STATE_DIM}), got {tuple(states.shape)}")
    k = states.shape[0]
    cams = torch.as_tensor(cameras, dtype=torch.float32, device=states.device)
    if cams.shape == (_lib.QS_CAM_DIM,):
        cams = cams.expand(k, -1)
    if cams.shape != (k, _lib.QS_CAM_DIM):
        raise ValueError(f"cameras must have shape ({_lib.QS_CAM_DIM},) or ({k}, {_lib.QS_CAM_DIM}), got {tuple(cams.shape)}")
    return states.to(torch.float32).contiguous(), cams.contiguous()


def render_states(states, cameras, width=RENDER_WIDTH, height=RENDER_HEIGHT, rgb=True, depth=False, segmentation=False):
    """Render robot i in state states[i] (qs_get_state rows: env.get_state(), SubstepRecorder rows, recorded
    demonstrations) through camera cameras[i] ([k, 32] or one [32] camera for all): view matrix then projection matrix,
    column-major as pybullet returns them.  Launches one kernel on the current stream and returns a dict of CUDA tensors:
      "rgb"           [k, H, W, 3] uint8
      "depth"         [k, H, W] float32, metric eye-space depth (far plane where nothing is hit)
      "segmentation"  [k, H, W] int32, objectUniqueId + ((linkIndex + 1) << 24): plane 0, robot links 1 + ((link + 1)
                      << 24) with URDF link indices (trunk 0, imu 1, hip / thigh / calf / foot of FR, FL, RR, RL), -1 sky
    A state row with a non-finite word is drawn as ground and sky only.  ValueError on bad shapes or sizes."""
    states, cams = _inputs(states, cameras)
    k, dev = states.shape[0], states.device
    shape = (k, max(int(height), 0), max(int(width), 0))
    out = {}
    if rgb:
        out["rgb"] = torch.empty(shape + (3,), dtype=torch.uint8, device=dev)
    if depth:
        out["depth"] = torch.empty(shape, dtype=torch.float32, device=dev)
    if segmentation:
        out["segmentation"] = torch.empty(shape, dtype=torch.int32, device=dev)
    _launch(states, cams, width, height, out.get("rgb"), out.get("depth"), out.get("segmentation"))
    return out


def tile_images(images):
    """stable-baselines3's tile_images: n images [n, H, W, c] -> one image of ceil(sqrt(n)) rows and
    ceil(n / rows) columns of them, row by row, the empty cells zero."""
    img = np.asarray(images)
    n, h, w, c = img.shape
    rows = int(np.ceil(np.sqrt(n)))
    cols = int(np.ceil(float(n) / rows))
    img = np.concatenate([img, np.zeros((rows * cols - n, h, w, c), dtype=img.dtype)], 0)
    return img.reshape(rows, cols, h, w, c).transpose(0, 2, 1, 3, 4).reshape(rows * h, cols * w, c)


class VideoRecorder:
    """Follow-camera frames of `env_ids` of a BatchedQuadrupedGymEnv, one per `capture()`, kept in a preallocated device
    buffer of `max_frames` frames (480 x 360 RGB is 0.5 MB per env and frame).  `frames` is [T, n, H, W, 3] uint8 on the
    device; `save_mp4` writes them tiled (tile_images) with cv2, as the reference's utils/video_recording.py does."""

    def __init__(self, env, env_ids=(0,), width=RENDER_WIDTH, height=RENDER_HEIGHT, max_frames=1000):
        self.env = env
        self.env_ids = torch.as_tensor(list(env_ids), dtype=torch.long, device=env.device)
        if self.env_ids.numel() < 1 or int(self.env_ids.min()) < 0 or int(self.env_ids.max()) >= env.num_envs:
            raise ValueError(f"env_ids must be a non-empty list of env indices in [0, {env.num_envs})")
        if max_frames < 1:
            raise ValueError("max_frames must be at least 1")
        self.width, self.height = int(width), int(height)
        self._buf = torch.empty(int(max_frames), self.env_ids.numel(), self.height, self.width, 3, dtype=torch.uint8,
                                device=env.device)
        self._count = 0

    def capture(self):
        """Render the current state of the envs into the next frame (call it after reset() and after each step)."""
        if self._count == self._buf.shape[0]:
            raise RuntimeError(f"VideoRecorder buffer is full ({self._buf.shape[0]} frames)")
        st = self.env.get_state().index_select(0, self.env_ids)
        cams = follow_cameras(st[:, :3], self.width, self.height)
        st, cams = _inputs(st, cams)
        _launch(st, cams, self.width, self.height, self._buf[self._count], None, None)
        self._count += 1

    @property
    def frames(self):
        return self._buf[:self._count]

    def reset(self):
        self._count = 0

    def save_mp4(self, path, fps=None):
        """Write the captured frames, tiled, to `path` (mp4v).  fps defaults to the control rate 1 / env_time_step."""
        try:
            import cv2
        except ImportError as e:
            raise RuntimeError("VideoRecorder.save_mp4 needs OpenCV (the cv2 module), which is not installed") from e
        if self._count == 0:
            raise RuntimeError("no frame captured")
        fps = float(fps) if fps is not None else 1.0 / self.env.env_time_step
        frames = self.frames.cpu().numpy()
        first = tile_images(frames[0])
        writer = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"mp4v"), fps, (first.shape[1], first.shape[0]))
        if not writer.isOpened():
            raise RuntimeError(f"cv2 cannot open a video writer for {path}")
        try:
            for f in frames:
                writer.write(np.ascontiguousarray(tile_images(f)[:, :, ::-1]))   # cv2 takes BGR
        finally:
            writer.release()
