"""PPO on the door panel (C2 settings) with the on-GPU learner: the learning curve up to and past the reference's
2 M-sample point, and the learner's throughput against a torch autograd learner on the same fragment.

    python profiles/ppo_door.py --out ppo_door_b200.json

Curve: coverage ratio (episode `reward` total x 100 / max points) and episode-length ratio (length / 235) of the
episodes that ended in each iteration, against env-steps and wall-clock, for each learning rate given.  The
reference's published values at 2 M samples are about 0.95 coverage and 1.0 length ratio on the door.

Learner throughput: samples x epochs / s of `PPOLearner.update` (host clock around the call, which ends in a device
synchronisation), and the same schedule -- same fragment, same minibatches, same Adam -- run through torch autograd
(FP32 matmuls, torch.optim.Adam), timed the same way.  The GPU's name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        line = subprocess.run(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader', '-i', '0'], stdout=subprocess.PIPE,
                              text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(','), [s.strip() for s in line.split(',')]))
    except Exception as exc:       # noqa: BLE001 - keep the measurement, say why the query is missing
        return {'error': str(exc)}


def torch_update(params, rows, bounds, perms, cfg, kl_coeff, obs_dim, n_out):
    """The same PPO schedule in torch autograd (FP32): forward, loss, backward and Adam per minibatch."""
    p = params.detach().clone().requires_grad_(True)
    opt = torch.optim.Adam([p], lr=cfg.lr, betas=(cfg.adam_beta1, cfg.adam_beta2), eps=cfg.adam_eps)
    sizes = [obs_dim * 256, 256, 256 * 128, 128, 128 * (n_out + 1), n_out + 1]
    for perm in perms:
        for s, n in bounds:
            i = perm[s:s + n].long()
            w1, b1, w2, b2, w3, b3 = torch.split(p, sizes)
            x = rows['obs'][i].float()
            h = torch.tanh(x @ w1.view(obs_dim, 256) + b1)
            h = torch.tanh(h @ w2.view(256, 128) + b2)
            out = h @ w3.view(128, n_out + 1) + b3
            lp_all = torch.log_softmax(out[:, :n_out], 1)
            v = out[:, n_out]
            logp = lp_all.gather(1, rows['actions'][i][:, None])[:, 0]
            lpo = torch.log_softmax(rows['logits'][i][:, :n_out], 1)
            kl = (lpo.exp() * (lpo - lp_all)).sum(1)
            ent = -(lp_all.exp() * lp_all).sum(1)
            A, R, vold = rows['adv'][i], rows['vtarg'][i], rows['value'][i]
            r = torch.exp(logp - rows['logp'][i])
            surr = torch.min(A * r, A * torch.clamp(r, 1 - cfg.clip_param, 1 + cfg.clip_param))
            vf = torch.max((v - R) ** 2, (vold + torch.clamp(v - vold, -cfg.vf_clip_param, cfg.vf_clip_param) - R) ** 2)
            loss = (-surr + kl_coeff * kl + cfg.vf_loss_coeff * vf - cfg.entropy_coeff * ent).mean()
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
    return p.detach()


def throughput(args, device):
    from paintrl_b200 import ppo
    from paintrl_b200.train import Trainer
    cfg = ppo.PPOConfig(minibatch_size=args.minibatch, num_sgd_iter=args.sgd_iters, lr=args.lrs[0], seed=0)
    tr = Trainer(0, args.envs, args.fragment, seed=0, device=device, config=cfg)
    tr.iteration()                                       # warm-up: graph capture, first launches
    frag, _ = tr.worker.collect()
    L = tr.learner
    rows = L.flatten(frag)
    bounds = ppo.minibatches(rows['n'], cfg.minibatch_size)
    res = {}
    for rep in range(2):
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        L.update(frag)
        res.setdefault('ours_s', []).append(time.perf_counter() - t0)
    perms = [torch.randperm(rows['n'], device=device).to(torch.int32) for _ in range(cfg.num_sgd_iter)]
    torch.backends.cuda.matmul.allow_tf32 = False
    torch_update(L.params, rows, bounds[:2], perms[:1], cfg, L.kl_coeff, L.obs_dim, L.n_out)      # warm-up
    for rep in range(2):
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        torch_update(L.params, rows, bounds, perms, cfg, L.kl_coeff, L.obs_dim, L.n_out)
        torch.cuda.synchronize(device)
        res.setdefault('torch_s', []).append(time.perf_counter() - t0)
    work = rows['n'] * cfg.num_sgd_iter
    tr.close()
    return {'samples_per_update': rows['n'], 'epochs': cfg.num_sgd_iter, 'minibatch': cfg.minibatch_size,
            'minibatches_per_update': len(bounds) * cfg.num_sgd_iter,
            'ours_update_s': res['ours_s'], 'torch_autograd_update_s': res['torch_s'],
            'ours_samples_x_epochs_per_s': work / min(res['ours_s']),
            'torch_samples_x_epochs_per_s': work / min(res['torch_s']),
            'speedup': min(res['torch_s']) / min(res['ours_s'])}


def curve(args, lr, device):
    from paintrl_b200 import ppo
    from paintrl_b200.train import Trainer
    cfg = ppo.PPOConfig(minibatch_size=args.minibatch, num_sgd_iter=args.sgd_iters, lr=lr, seed=args.seed)
    tr = Trainer(0, args.envs, args.fragment, seed=args.seed, device=device, config=cfg)
    iters = int(math.ceil(args.samples / float(args.envs * args.fragment)))
    t0 = time.perf_counter()
    out = []
    for it in range(iters):
        r = tr.iteration()
        r['wall_s'] = time.perf_counter() - t0
        ls = r.pop('learner')
        r.update({k: ls[k] for k in ('policy_loss', 'vf_loss', 'kl_last_epoch', 'entropy', 'clip_fraction', 'kl_coeff')})
        out.append(r)
        print(json.dumps(dict(lr=lr, **r)), flush=True)
    tr.close()
    return {'lr': lr, 'config': cfg.to_dict(), 'iterations': out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--fragment', type=int, default=100)
    ap.add_argument('--samples', type=int, default=8000000)
    ap.add_argument('--minibatch', type=int, default=4096)
    ap.add_argument('--sgd-iters', type=int, default=16)
    ap.add_argument('--lrs', type=float, nargs='+', default=[5e-5, 1e-3])
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--no-throughput', action='store_true')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('ppo_door.py measures on a CUDA device; none is visible')
    device = torch.device('cuda:0')
    from paintrl_b200 import build
    build.build()
    res = {'gpu': gpu_info(), 'torch': torch.__version__, 'settings': 'door (Part_NO 0), C2: RGB, section-4 observation, '
           'discrete-4 actions, late termination, anchor starts, auto-reset', 'envs': args.envs, 'fragment': args.fragment,
           'reference_at_2M_samples': {'coverage': 0.95, 'length_ratio': 1.0}}
    if not args.no_throughput:
        res['learner_throughput'] = throughput(args, device)
        print(json.dumps(res['learner_throughput']), flush=True)
    res['curves'] = [curve(args, lr, device) for lr in args.lrs]
    res['gpu_after'] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f)
    print(json.dumps({'gpu': res['gpu'], 'learner_throughput': res.get('learner_throughput')}))


if __name__ == '__main__':
    main()
