#!/usr/bin/env python
"""Train the policy on the door with PPO on the GPU, save it, and let the saved policy drive the reference's gym.Env
(needs a CUDA device; run from the repository root).

    python examples/train_and_drive.py [checkpoint.pt]

Without an argument it trains for 10 iterations of 4096 environments x 100 steps (about 4 M env-steps, a few seconds
on a B200) and writes /tmp/paintrl_door_ppo.pt; with one it loads that checkpoint instead.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from paintrl_b200 import ppo, train
from paintrl_b200.config import DEFAULT_EXTRA_CONFIG
from PaintRLEnv.robot_gym_env import PaintGymEnv

device = torch.device('cuda:0')
if len(sys.argv) > 1:
    path = sys.argv[1]
else:
    path = '/tmp/paintrl_door_ppo.pt'
    tr = train.Trainer(0, 4096, 100, seed=0, device=device, config=ppo.PPOConfig(lr=1e-3))
    for it in range(10):
        r = tr.iteration()
        print('iteration %d: %d env-steps, coverage %.3f, length ratio %.3f' % (it, r['env_steps'], r['coverage'], r['length_ratio']))
    tr.save(path)
    tr.close()

policy = train.load_policy(path, device)
env = PaintGymEnv('', with_robot=False, renders=False, rollout=True, extra_config=dict(DEFAULT_EXTRA_CONFIG))
obs, done, total, steps = env.reset(), False, 0.0, 0
while not done:
    logits, _ = policy.forward(torch.as_tensor(obs, device=device)[None])
    obs, reward, done, info = env.step(int(logits.argmax()))          # greedy action
    total += reward
    steps += 1
print('gym.Env episode with the trained policy: %d steps, return %.2f, last info %s' % (steps, total, info))
env.close()
