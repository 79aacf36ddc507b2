"""Train a PPO policy on the GPU, save it as an rl-baselines3-zoo directory and replay it with load_model.replay.

The rollout buffer holds n_steps x num_envs samples: every control step of every env is a sample, so at 65536 envs a
small n_steps (here 16: 1 M samples per iteration) plays the part of SB3's 2048 steps of a handful of envs.

    python examples/train_ppo.py [log_dir] [iterations] [num_envs]"""
import os
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import quadruped_springs_b200 as qs
from quadruped_springs_b200 import load_model

ENV_KWARGS = dict(task_env="JUMPING_IN_PLACE_PPO", observation_space_mode="PPO_BASIC", action_space_mode="SYMMETRIC",
                  enable_springs=True, motor_control_mode="PD")


def main(log_dir=None, iterations=10, num_envs=65536):
    log_dir = log_dir or tempfile.mkdtemp(prefix="ppo_")
    n_steps = 16
    model = qs.BatchedPPO("MlpPolicy", ENV_KWARGS, num_envs=num_envs, n_steps=n_steps, batch_size=num_envs * n_steps // 8,
                          n_epochs=5, seed=0, verbose=1)
    print("initial policy:", float(model.evaluate(256).mean()))
    model.learn(total_timesteps=iterations * num_envs * n_steps)
    print("trained:       ", float(model.evaluate(256).mean()))
    model.save(log_dir)
    ret = load_model.replay(log_dir, ENV_KWARGS["task_env"], algo="ppo", n_envs=256, go_to_rest_wrapper=False, seed=0)
    print(f"replayed from {log_dir}:", float(ret.mean()))


if __name__ == "__main__":
    a = sys.argv[1:]
    main(a[0] if a else None, int(a[1]) if len(a) > 1 else 10, int(a[2]) if len(a) > 2 else 65536)
