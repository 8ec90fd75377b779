"""PPO with continuous actions on the door panel: the diagonal-Gaussian head (learned log-std) against the fixed
N(tanh mu, I) head, with C2's settings except continuous-2 actions.

    python profiles/ppo_continuous_door.py --out ppo_continuous_door_b200.json [--samples 20000000]

- act kernel: one `policy_act_kernel` launch for 65536 environments, the diagonal-Gaussian instantiation
  (paintrl_policy_act_diag_gaussian, n_out 4) against the existing continuous one (paintrl_policy_act, n_out 2),
  alternated in rounds of 200 launches each, CUDA events around each round.
- learner: one `PPOLearner.update` of 4096 x 100 samples x 16 epochs (minibatch 4096), diagonal-Gaussian and
  categorical (discrete-4, the learner of profiles/ppo_door.py) alternated, host clock around a call that ends in a
  device synchronisation.
- learning curves from seed 0 up to --samples env-steps, 4096 environments x 100 steps, lr 1e-3 (the train script's
  PPO default): coverage ratio, length ratio (length / 235) and, for the diagonal-Gaussian head, the mean sigma of the
  sampled fragment per iteration.  The discrete-4 curve to compare with is profiles/ppo_door_b200.json.

The GPU's name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ppo_door import gpu_info  # noqa: E402

SPACES = dict(action_mode='continuous', action_shape=2)


def act_kernel(device, envs=65536, rounds=10, launches=200):
    from paintrl_b200.rollout import MlpPolicy
    obs = torch.rand(envs, 6, dtype=torch.float64, device=device)
    arms = {}
    for dist in ('diag_gaussian', 'tanh_gaussian'):
        pol = MlpPolicy(6, 2, device=device, seed=0, discrete=False, dist=dist)
        assert pol.enable_native(envs)
        act = torch.zeros(envs, 2, dtype=torch.float64, device=device)
        logp, value = torch.zeros(envs, device=device), torch.zeros(envs, device=device)
        if dist == 'diag_gaussian':
            call = lambda p=pol, a=act, l=logp, v=value: p.native.act_diag_gaussian_into(obs, a, l, v)
        else:
            call = lambda p=pol, a=act, l=logp, v=value: p.native.act_into(obs, a, l, v)
        for _ in range(20):
            call()
        arms[dist] = (pol, call, [])
    torch.cuda.synchronize(device)
    for _ in range(rounds):
        for dist, (pol, call, times) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                call()
            e1.record()
            torch.cuda.synchronize(device)
            times.append(e0.elapsed_time(e1) * 1e3 / launches)
    out = {'envs': envs, 'launches_per_round': launches}
    for dist, (pol, call, times) in arms.items():
        out[dist + '_us'] = sorted(times)
        out[dist + '_median_us'] = sorted(times)[len(times) // 2]
        pol.native.close()
    return out


def learner_update(device, rounds=3):
    from paintrl_b200 import ppo
    from paintrl_b200.rollout import MlpPolicy, RolloutFragment
    T, B = 100, 4096
    arms = {}
    for dist in ('diag_gaussian', 'categorical'):
        discrete = dist == 'categorical'
        pol = MlpPolicy(6, 2 if not discrete else 4, device=device, seed=0, discrete=discrete, dist=dist)
        f = RolloutFragment(T, B, 6, () if discrete else (2,), device, logits_dim=pol.n_out + 1)
        g = torch.Generator(device=device).manual_seed(1)
        f.obs.copy_(torch.rand(f.obs.shape, generator=g, device=device, dtype=torch.float64))
        if discrete:
            f.actions.copy_(torch.randint(0, 4, f.actions.shape, generator=g, device=device))
        else:
            f.actions.copy_(torch.randn(f.actions.shape, generator=g, device=device, dtype=torch.float64).float().double())
        f.actual.copy_(torch.rand(f.actual.shape, generator=g, device=device, dtype=torch.float64))
        f.done.copy_((torch.rand(f.done.shape, generator=g, device=device) < 0.01).to(torch.uint8))
        f.logits.copy_(0.1 * torch.randn(f.logits.shape, generator=g, device=device))
        f.logp.copy_(-2.0 + 0.1 * torch.randn(f.logp.shape, generator=g, device=device))
        L = ppo.PPOLearner(pol, ppo.PPOConfig(lr=1e-3))
        L.update(f)
        arms[dist] = (L, f, [])
    for _ in range(rounds):
        for dist, (L, f, times) in arms.items():
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            L.update(f)                       # ends in the read of its statistics
            times.append(time.perf_counter() - t0)
    out = {'samples_per_update': T * B, 'epochs': 16, 'minibatch': 4096}
    for dist, (L, f, times) in arms.items():
        out[dist + '_update_s'] = times
        L.close()
    return out


def curve(device, dist, samples, seed=0):
    from paintrl_b200 import ppo
    from paintrl_b200.train import Trainer
    tr = Trainer(0, 4096, 100, seed=seed, device=device, config=ppo.PPOConfig(seed=seed, lr=1e-3), spaces=SPACES, dist=dist)
    A = tr.policy.action_dim
    its = []
    t0 = time.perf_counter()
    while tr.env_steps < samples:
        r = tr.iteration()
        row = {k: r[k] for k in ('env_steps', 'episodes', 'mean_return', 'coverage', 'length_ratio', 'collect_s', 'learn_s')}
        row.update({k: r['learner'][k] for k in ('policy_loss', 'vf_loss', 'kl', 'entropy', 'mean_ratio', 'kl_coeff')})
        row['wall_s'] = time.perf_counter() - t0
        if dist == 'diag_gaussian':
            # mean sigma over the fragment just collected (its log-std columns, before this iteration's update)
            row['mean_sigma'] = float(torch.exp(tr.worker.frag.logits[..., A:2 * A]).mean())
        its.append(row)
    tr.close()
    return its


def at(its, n):
    """The iteration that reaches n env-steps: coverage and length ratio there and averaged over the last 5."""
    k = next(i for i, r in enumerate(its) if r['env_steps'] >= n)
    last = its[max(0, k - 4):k + 1]
    mean = lambda key: sum(r[key] for r in last if r[key] is not None) / max(1, sum(r[key] is not None for r in last))
    return {'env_steps': its[k]['env_steps'], 'coverage': its[k]['coverage'], 'length_ratio': its[k]['length_ratio'],
            'coverage_last5': mean('coverage'), 'length_ratio_last5': mean('length_ratio'),
            'mean_sigma': its[k].get('mean_sigma')}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='ppo_continuous_door_b200.json')
    ap.add_argument('--samples', type=int, default=20000000)
    args = ap.parse_args()
    device = torch.device('cuda:0')
    res = {'gpu': gpu_info(), 'torch': torch.__version__,
           'settings': 'door (Part_NO 0), C2 settings except continuous-2 actions: RGB, section-4 observation, late termination, '
                       'anchor starts, auto-reset; 4096 environments x 100 steps, PPOConfig defaults with lr 1e-3, seed 0'}
    res['act_kernel'] = act_kernel(device)
    print(json.dumps(res['act_kernel']), flush=True)
    res['learner'] = learner_update(device)
    print(json.dumps(res['learner']), flush=True)
    res['curves'] = {}
    for dist in ('diag_gaussian', 'tanh_gaussian'):
        its = curve(device, dist, args.samples)
        res['curves'][dist] = {'iterations': its, 'at_2M': at(its, 2000000), 'at_end': at(its, args.samples)}
        print(dist, json.dumps(res['curves'][dist]['at_2M']), json.dumps(res['curves'][dist]['at_end']), flush=True)
    res['gpu_after'] = gpu_info()
    with open(args.out, 'w') as fh:
        json.dump(res, fh)


if __name__ == '__main__':
    main()
