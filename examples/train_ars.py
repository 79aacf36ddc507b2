"""Train an ARS policy on the GPU, save it as an rl-baselines3-zoo directory and replay it with load_model.replay.

Every iteration evaluates all 2 * n_delta candidate policies at once, one candidate per group of n_eval_episodes envs.

    python examples/train_ars.py [log_dir] [iterations] [LinearPolicy|MlpPolicy]"""
import os
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import quadruped_springs_b200 as qs
from quadruped_springs_b200 import load_model

ENV_KWARGS = dict(task_env="JUMPING_IN_PLACE_PPO", observation_space_mode="ARS_BASIC", action_space_mode="SYMMETRIC",
                  enable_springs=True, motor_control_mode="PD")


def main(log_dir=None, iterations=10, policy="LinearPolicy"):
    log_dir = log_dir or tempfile.mkdtemp(prefix="ars_")
    model = qs.BatchedARS(policy, ENV_KWARGS, n_delta=8, n_eval_episodes=256, seed=0, verbose=1)   # 4096 envs
    print("zero policy:", float(model.evaluate(256).mean()))
    model.learn(total_timesteps=10**12, callback=lambda m, rec: rec["iteration"] < iterations)
    print("trained:    ", float(model.evaluate(256).mean()))
    model.save(log_dir)
    ret = load_model.replay(log_dir, ENV_KWARGS["task_env"], algo="ars", n_envs=256, go_to_rest_wrapper=False, seed=0)
    print(f"replayed from {log_dir}:", float(ret.mean()))


if __name__ == "__main__":
    a = sys.argv[1:]
    main(a[0] if a else None, int(a[1]) if len(a) > 1 else 10, a[2] if len(a) > 2 else "LinearPolicy")
