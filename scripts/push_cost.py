"""Step time with and without the external push (qs_set_external_force) on BASELINE configuration 3.

One process, one GPU: bench.py's job (65536 envs, auto_reset, noise, random actions) pre-rolled to the stationary regime
as bench.py does, then four arms alternated `--repeats` times in rotating order -- no push buffer, the buffers attached
with every count 0, `--pushed` envs pushed on every tick, every env pushed on every tick -- each timed over `--steps`
steps with CUDA events after a warm-up that recaptures the step's graphs (attaching or detaching the buffers drops them).
The pushed arms write the pushed envs' counts before every step (an episode end clears a count), one small torch kernel
per step that is timed with the arm.  The push is a horizontal force of 30 N at a random point of the trunk.  Prints one
JSON line: per arm the median step time and the spread over the repeats, with the device name and its power limit.

    python scripts/push_cost.py [--envs 65536] [--steps 300] [--repeats 5] [--pushed 1024]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--pushed", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=40)
    args = ap.parse_args()

    import torch
    import bench
    from quadruped_springs_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("push_cost.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    L = _lib.lib()
    job = bench.Job(bench.CONFIGS[3], args.envs, dev, 0, seed=0)
    info = bench.preroll(job, L, _lib, 600, 1, None, dev, 150)
    env = job.env
    gen = torch.Generator().manual_seed(5)
    n, R = args.envs, env._action_repeat
    ang = torch.rand(n, generator=gen) * 6.283185307179586
    force = torch.stack([30 * ang.cos(), 30 * ang.sin(), torch.zeros(n)], 1)
    point = (torch.rand(n, 3, generator=gen) * 2 - 1) * torch.tensor([0.1881, 0.04675, 0.057])
    arms = {"no_buffer": None, "idle_buffer": torch.zeros(0, dtype=torch.long),
            f"pushed_{args.pushed}": torch.randperm(n, generator=gen)[:args.pushed].sort().values.to(dev),
            "pushed_all": torch.arange(n, device=dev)}
    names = list(arms)
    times = {k: [] for k in names}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep in range(args.repeats):
        for k in names[rep % 4:] + names[:rep % 4]:
            ids = arms[k]
            if ids is None:
                env.robot.clear_external_force()
            else:
                env.robot.apply_external_force(force, point, n_ticks=0)      # attaches; every count 0
            ticks = env.robot.get_external_force()[2] if ids is not None and ids.numel() else None

            def step():
                if ticks is not None:
                    ticks.index_fill_(0, ids, R)      # pushed on every tick of this step
                job.step(job.next_input())

            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / args.steps)
    env.robot.clear_external_force()
    res = {k: {"step_ms_median": statistics.median(v), "step_ms_min": min(v), "step_ms_max": max(v), "repeats": v}
           for k, v in times.items()}
    print(json.dumps({"config": bench.CONFIGS[3]["name"], "envs": args.envs, "steps_per_repeat": args.steps,
                      "device": torch.cuda.get_device_name(dev), "power_limit": power_limit(dev.index or 0),
                      "preroll": info, "arms": res}))


if __name__ == "__main__":
    main()
