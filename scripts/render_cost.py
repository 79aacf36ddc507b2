"""Cost of qs_render (quadruped_springs_b200/render.py render_states) at three sizes a user runs.

  video         16 envs at 480 x 360 (the follow camera of env.render / VideoRecorder)
  batch_128     1024 envs at 128 x 128
  pixel_obs_64  4096 envs at 64 x 64 (pixel observations)

The states come from bench.py configuration 3 after a short random rollout (robots standing, jumping and landing), one
follow camera per env.  Each size renders RGB + depth + segmentation into preallocated outputs, warmed up, then timed
with CUDA events over at least `--seconds` of back-to-back calls.  Reported per size: time per call, images/s, Mrays/s
(one primary ray per pixel; shadow rays are not counted), and the bytes the call writes per second against the 7.7 TB/s
HBM bound of a B200.  One JSON line, with the device name and its power limit.

    python scripts/render_cost.py [--seconds 1.0] [--rollout 40]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12
SIZES = {"video": (16, 480, 360), "batch_128": (1024, 128, 128), "pixel_obs_64": (4096, 64, 64)}


def power_limit(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rollout", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()

    import numpy as np
    import torch

    import bench
    import quadruped_springs_b200 as qs
    from quadruped_springs_b200 import render

    if not torch.cuda.is_available():
        raise SystemExit("render_cost.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    cfg = bench.CONFIGS[3]["env"]
    n_max = max(n for n, _, _ in SIZES.values())
    env = qs.BatchedQuadrupedGymEnv(num_envs=n_max, device=dev, seed=0, auto_reset=True, enable_noise=True, **cfg)
    env.reset()
    rng = np.random.default_rng(0)
    for _ in range(args.rollout):
        env.step(torch.tensor(rng.uniform(-1, 1, (n_max, env.action_dim)), dtype=torch.float32, device=dev))
    all_states = env.get_state()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {}
    for name, (k, W, H) in SIZES.items():
        states = all_states[:k].contiguous()
        cams = render.follow_cameras(states[:, :3], W, H)
        rgb = torch.empty(k, H, W, 3, dtype=torch.uint8, device=dev)
        depth = torch.empty(k, H, W, device=dev)
        seg = torch.empty(k, H, W, dtype=torch.int32, device=dev)
        call = lambda: render._launch(states, cams, W, H, rgb, depth, seg)
        for _ in range(args.warmup):
            call()
        torch.cuda.synchronize()
        e0.record()          # size the timed window from one probe
        call()
        e1.record()
        e1.synchronize()
        reps = max(20, int(args.seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)) + 1)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out_bytes = k * H * W * (3 + 4 + 4)
        res[name] = {"envs": k, "width": W, "height": H, "calls": reps, "timed_s": ms * reps / 1e3,
                     "ms_per_call": ms, "images_per_s": k / (ms / 1e3), "mrays_per_s": k * W * H / (ms / 1e3) / 1e6,
                     "robot_pixel_share": float((seg > 0).float().mean()),
                     "out_bytes": out_bytes, "out_gb_per_s": out_bytes / (ms / 1e3) / 1e9,
                     "share_of_hbm_write_bound": out_bytes / HBM_BYTES_PER_S / (ms / 1e3)}
    print(json.dumps({"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(dev.index or 0),
                      "sizes": res}))


if __name__ == "__main__":
    main()
