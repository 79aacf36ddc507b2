"""Step time with and without the per-substep trace (qs_set_substep_trace) on BASELINE configuration 3.

One process, one GPU: bench.py's job (65536 envs, auto_reset, noise, random actions) pre-rolled to the stationary regime
as bench.py does, then three arms alternated `--repeats` times in rotating order -- no trace, a trace of `--traced` envs,
a trace of every env -- each timed over `--steps` steps with CUDA events after a warm-up that recaptures the step's
graphs (setting or clearing a trace drops them).  Prints one JSON line: per arm the median step time and the spread over
the repeats, with the device name and its power limit.

    python scripts/trace_cost.py [--envs 65536] [--steps 300] [--repeats 5] [--traced 1024]
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
    ap.add_argument("--traced", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=40)
    args = ap.parse_args()

    import torch
    import bench
    from quadruped_springs_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("trace_cost.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    L = _lib.lib()
    job = bench.Job(bench.CONFIGS[3], args.envs, dev, 0, seed=0)
    info = bench.preroll(job, L, _lib, 600, 1, None, dev, 150)
    env = job.env
    gen = torch.Generator().manual_seed(5)
    arms = {"none": None, f"traced_{args.traced}": torch.randperm(args.envs, generator=gen)[:args.traced].sort().values,
            "traced_all": torch.arange(args.envs)}
    names = list(arms)
    times = {k: [] for k in names}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep in range(args.repeats):
        for k in names[rep % 3:] + names[:rep % 3]:
            env.set_substep_trace(arms[k])
            for _ in range(args.warmup):
                job.step(job.next_input())
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                job.step(job.next_input())
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / args.steps)
    env.set_substep_trace(None)
    res = {k: {"step_ms_median": statistics.median(v), "step_ms_min": min(v), "step_ms_max": max(v), "repeats": v}
           for k, v in times.items()}
    print(json.dumps({"config": bench.CONFIGS[3]["name"], "envs": args.envs, "steps_per_repeat": args.steps,
                      "device": torch.cuda.get_device_name(dev), "power_limit": power_limit(dev.index or 0),
                      "preroll": info, "arms": res}))


if __name__ == "__main__":
    main()
