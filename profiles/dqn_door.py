"""Double DQN on the door panel (C2 settings) with the on-GPU learner: the learning curve to 2 M and 20 M env-steps
next to PPO's (profiles/ppo_door_b200.json), and the learner's throughput against a torch autograd learner on the same
schedule.

    python profiles/dqn_door.py --out dqn_door_b200.json

Curve: coverage ratio (episode `reward` total x 100 / max points) and episode-length ratio (length / 235) of the
episodes that ended in each iteration, with epsilon and the learner's statistics, against env-steps and wall-clock.

Learner throughput: gradient steps / s and replayed samples / s of `DQNLearner.update` on a full fragment (host clock
around the call, which ends in a device synchronisation), and the same schedule -- same minibatch size, uniform replay
indices, double-Q dueling Huber loss, clip_grad_norm_, torch.optim.Adam, target sync -- in torch autograd (FP32),
timed the same way.  The GPU's name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import math
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ppo_door import gpu_info                                     # noqa: E402  (profiles/ is on sys.path when run as a script)

PPO_JSON = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'ppo_door_b200.json')


def torch_steps(learner, n_steps):
    """n_steps gradient steps of the same schedule in torch autograd (FP32): returns the final parameters."""
    cfg, buf = learner.cfg, learner.replay
    obs_dim, n_out = learner.obs_dim, learner.n_out
    p = learner.params.detach().clone().requires_grad_(True)
    target = learner.target.detach().clone()
    opt = torch.optim.Adam([p], lr=cfg.lr, betas=(cfg.adam_beta1, cfg.adam_beta2), eps=cfg.adam_eps)
    sizes = [obs_dim * 256, 256, 256 * 128, 128, 128 * (n_out + 1), n_out + 1]
    gen = torch.Generator(device=p.device).manual_seed(123)

    def q_values(params, x):
        w1, b1, w2, b2, w3, b3 = torch.split(params, sizes)
        h = torch.tanh(x @ w1.view(obs_dim, 256) + b1)
        h = torch.tanh(h @ w2.view(256, 128) + b2)
        out = h @ w3.view(128, n_out + 1) + b3
        A = out[:, :n_out]
        return out[:, n_out:] + A - A.mean(1, keepdim=True)

    for step in range(1, n_steps + 1):
        i = buf.sample(cfg.minibatch_size, gen).long()
        with torch.no_grad():
            nx = buf.next_obs[i].float()
            an = q_values(p, nx).argmax(1, keepdim=True)
            y = buf.reward[i] + cfg.gamma * (1.0 - buf.done[i].float()) * q_values(target, nx).gather(1, an)[:, 0]
        qsa = q_values(p, buf.obs[i].float()).gather(1, buf.actions[i][:, None])[:, 0]
        loss = torch.nn.functional.huber_loss(qsa, y, delta=1.0)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_([p], cfg.grad_clip)
        opt.step()
        if step % cfg.target_update_freq == 0:
            target.copy_(p.detach())
    return p.detach()


def throughput(args, device):
    from paintrl_b200 import dqn
    from paintrl_b200.train import Trainer
    cfg = dqn.DQNConfig(seed=0)
    tr = Trainer(0, args.envs, args.fragment, seed=0, device=device, config=cfg, algo='dqn', total_samples=args.samples)
    tr.iteration()                                  # fills past learning_starts; warm-up of graph capture and first launches
    tr.iteration()
    frag, _ = tr.worker.collect()
    L = tr.learner
    res = {}
    for rep in range(3):
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        st = L.update(frag)
        res.setdefault('ours_s', []).append(time.perf_counter() - t0)
    steps = st['grad_steps']
    torch.backends.cuda.matmul.allow_tf32 = False
    torch_steps(L, 5)                               # warm-up
    for rep in range(2):
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        torch_steps(L, steps)
        torch.cuda.synchronize(device)
        res.setdefault('torch_s', []).append(time.perf_counter() - t0)
    tr.close()
    ours, ref = min(res['ours_s']), min(res['torch_s'])
    return {'samples_per_update': frag.T * frag.B, 'grad_steps_per_update': steps, 'minibatch': cfg.minibatch_size,
            'ours_update_s': res['ours_s'], 'torch_autograd_update_s': res['torch_s'],
            'ours_grad_steps_per_s': steps / ours, 'ours_replayed_samples_per_s': steps * cfg.minibatch_size / ours,
            'torch_grad_steps_per_s': steps / ref, 'torch_replayed_samples_per_s': steps * cfg.minibatch_size / ref,
            'speedup': ref / ours}


def curve(args, device):
    from paintrl_b200 import dqn
    from paintrl_b200.train import Trainer
    cfg = dqn.DQNConfig(seed=args.seed)
    tr = Trainer(0, args.envs, args.fragment, seed=args.seed, device=device, config=cfg, algo='dqn', total_samples=args.samples)
    iters = int(math.ceil(args.samples / float(args.envs * args.fragment)))
    t0 = time.perf_counter()
    out = []
    for it in range(iters):
        r = tr.iteration()
        r['wall_s'] = time.perf_counter() - t0
        r.update({k: v for k, v in r.pop('learner').items() if k != 'samples'})
        out.append(r)
        print(json.dumps(r), flush=True)
    tr.close()
    return {'config': cfg.to_dict(), 'iterations': out}


def at_steps(iterations, steps):
    """The first iteration at or past `steps` env-steps: coverage and length ratio."""
    for r in iterations:
        if r['env_steps'] >= steps:
            return {'env_steps': r['env_steps'], 'coverage': r['coverage'], 'length_ratio': r['length_ratio']}
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--fragment', type=int, default=100)
    ap.add_argument('--samples', type=int, default=20000000)
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--no-throughput', action='store_true')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('dqn_door.py measures on a CUDA device; none is visible')
    device = torch.device('cuda:0')
    from paintrl_b200 import build
    build.build()
    res = {'gpu': gpu_info(), 'torch': torch.__version__, 'settings': 'door (Part_NO 0), C2: RGB, section-4 observation, '
           'discrete-4 actions, late termination, anchor starts, auto-reset', 'envs': args.envs, 'fragment': args.fragment,
           'reference_at_2M_samples': {'coverage': 0.95, 'length_ratio': 1.0}}
    if not args.no_throughput:
        res['learner_throughput'] = throughput(args, device)
        print(json.dumps(res['learner_throughput']), flush=True)
    res['curve'] = curve(args, device)
    its = res['curve']['iterations']
    res['summary'] = {'dqn': {'2M': at_steps(its, 2000000), '20M': at_steps(its, 20000000)}}
    if os.path.isfile(PPO_JSON):
        with open(PPO_JSON) as f:
            ppo_res = json.load(f)
        for c in ppo_res['curves']:
            res['summary']['ppo_lr_%g' % c['lr']] = {'2M': at_steps(c['iterations'], 2000000), '20M': at_steps(c['iterations'], 20000000)}
    res['gpu_after'] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f)
    print(json.dumps({'gpu': res['gpu'], 'learner_throughput': res.get('learner_throughput'), 'summary': res['summary']}))


if __name__ == '__main__':
    main()
