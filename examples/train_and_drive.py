#!/usr/bin/env python
"""Train the policy on the door with PPO on the GPU, save it, and let the saved policy drive the reference's gym.Env
(needs a CUDA device; run from the repository root).

    python examples/train_and_drive.py [checkpoint.pt]

Without an argument it trains for 10 iterations of 4096 environments x 100 steps (about 4 M env-steps, a few seconds
on a B200) and writes /tmp/paintrl_door_ppo.pt; with one it loads that checkpoint instead, PPO or DQN
(`python -m paintrl_b200.train --algo dqn ...`): for a DQN policy the argmax of the head's first n_out columns is the
greedy Q action, up to the tie rule.  A continuous checkpoint (`--action-mode continuous`) drives with its mean action;
the gym.Env is set to the spaces the checkpoint records.
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
spaces = train.checkpoint_spaces(torch.load(path, map_location='cpu', weights_only=False))
PaintGymEnv.change_obs_mode(spaces['obs_mode'], spaces['obs_grad'])
PaintGymEnv.change_action_mode(spaces['action_shape'], spaces['action_mode'], spaces['granularity'])
env = PaintGymEnv('', with_robot=False, renders=False, rollout=True, extra_config=dict(DEFAULT_EXTRA_CONFIG))
obs, done, total, steps = env.reset(), False, 0.0, 0
while not done:
    out, _ = policy.forward(torch.as_tensor(obs, device=device)[None])
    if policy.discrete:
        action = int(out.argmax())                                    # greedy action
    elif policy.dist == 'diag_gaussian':
        action = out[0, :policy.action_dim].double().cpu().numpy()   # mean action
    else:
        action = torch.tanh(out[0]).double().cpu().numpy()
    obs, reward, done, info = env.step(action)
    total += reward
    steps += 1
print('gym.Env episode with the trained policy: %d steps, return %.2f, last info %s' % (steps, total, info))
env.close()
