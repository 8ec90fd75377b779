"""Prioritized replay with 3-step returns against uniform 1-step replay, for double DQN on the door panel (C2 settings):
learner throughput, the priority-tree kernels' times, and the learning curves to 2 M and 20 M env-steps.

    python profiles/dqn_per_door.py --out dqn_per_door_b200.json

Throughput: gradient steps / s of `DQNLearner.update` on one full fragment (4096 environments x 100 steps, 800 gradient
steps of minibatch 4096, replay capacity 2^21), host clock around the call (it ends in a device synchronisation), the
two configurations alternated in one run.  The prioritized update also pays the fragment's insertion into the trees.

Kernel times: CUDA events around many back-to-back launches of `paintrl_prio_sample` (n = 4096), `paintrl_prio_update`
(n = 4096, with its full rebuild of both trees) and `paintrl_prio_fill` (one fragment, 409,600 rows, with its rebuild), at
capacity 2^21 (L = 2^21: 16 MB of leaves read, 32 MB of internal nodes written per rebuild), and an update of one row,
which is the rebuild alone.

Curves: the ended episodes' coverage ratio and episode-length ratio per iteration for both configurations from the same
seed.  The GPU's name, power limit and SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import math
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ppo_door import gpu_info                                     # noqa: E402  (profiles/ is on sys.path when run as a script)
from dqn_door import at_steps                                     # noqa: E402

CONFIGS = {'uniform_1step': {}, 'prioritized_3step': {'prioritized_replay': True, 'n_step': 3}}


def _cfg(name, seed):
    from paintrl_b200 import dqn
    return dqn.DQNConfig(seed=seed, **CONFIGS[name])


def throughput(args, device, reps=3):
    from paintrl_b200.train import Trainer
    trainers, frags = {}, {}
    for name in CONFIGS:
        tr = Trainer(0, args.envs, args.fragment, seed=0, device=device, config=_cfg(name, 0), algo='dqn', total_samples=args.samples)
        tr.iteration()                              # fills past learning_starts; warms graph capture and first launches
        tr.iteration()
        frags[name], _ = tr.worker.collect()
        trainers[name] = tr
    times = {name: [] for name in CONFIGS}
    steps = {}
    for rep in range(reps):
        for name, tr in trainers.items():
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            st = tr.learner.update(frags[name])
            times[name].append(time.perf_counter() - t0)
            steps[name] = st['grad_steps']
    out = {}
    for name, tr in trainers.items():
        best = min(times[name])
        out[name] = {'update_s': times[name], 'grad_steps_per_update': steps[name], 'grad_steps_per_s': steps[name] / best,
                     'ms_per_grad_step': 1e3 * best / steps[name]}
        tr.close()
    out['prioritized_over_uniform_time'] = min(times['prioritized_3step']) / min(times['uniform_1step'])
    return out


def kernel_times(device, capacity=1 << 21, n=4096, fill_rows=409600, iters=200):
    from paintrl_b200 import _capi, dqn
    lib = _capi.lib()
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    L = dqn.tree_leaves(capacity)
    sum_t = torch.zeros(2 * L, dtype=torch.float64, device=device)
    min_t = torch.full((2 * L,), math.inf, dtype=torch.float64, device=device)
    maxp = torch.ones(1, dtype=torch.float64, device=device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    g = torch.Generator(device=device).manual_seed(0)
    _capi.check(lib.paintrl_prio_fill(P(sum_t), P(min_t), L, capacity, 0, capacity, P(maxp), 0.6, stream))
    all_rows = torch.arange(capacity, dtype=torch.int32, device=device)
    _capi.check(lib.paintrl_prio_update(P(sum_t), P(min_t), L, capacity, P(all_rows), P(torch.randn(capacity, generator=g, device=device)),
                                        capacity, P(maxp), 0.6, 1e-6, stream))
    u = torch.rand(n, generator=g, dtype=torch.float64, device=device)
    idx = torch.empty(n, dtype=torch.int32, device=device)
    w = torch.empty(n, dtype=torch.float32, device=device)
    td = torch.randn(n, generator=g, device=device)
    calls = {
        'prio_sample_n4096': lambda: lib.paintrl_prio_sample(P(sum_t), P(min_t), L, capacity, capacity, P(u), n, 0.4, P(idx), P(w), stream),
        'prio_update_n4096_with_rebuild': lambda: lib.paintrl_prio_update(P(sum_t), P(min_t), L, capacity, P(idx), P(td), n, P(maxp), 0.6,
                                                                          1e-6, stream),
        'prio_update_n1_rebuild_alone': lambda: lib.paintrl_prio_update(P(sum_t), P(min_t), L, capacity, P(idx), P(td), 1, P(maxp), 0.6,
                                                                        1e-6, stream),
        'prio_fill_409600_rows_with_rebuild': lambda: lib.paintrl_prio_fill(P(sum_t), P(min_t), L, capacity, 12345, fill_rows, P(maxp), 0.6,
                                                                            stream),
    }
    out = {'capacity': capacity, 'tree_leaves': L, 'iters': iters}
    for name, fn in calls.items():
        for _ in range(10):
            _capi.check(fn())
        res = []
        for rep in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                _capi.check(fn())
            e1.record()
            e1.synchronize()
            res.append(1e3 * e0.elapsed_time(e1) / iters)
        out[name + '_us'] = res
    return out


def curve(name, args, device):
    from paintrl_b200.train import Trainer
    cfg = _cfg(name, args.seed)
    tr = Trainer(0, args.envs, args.fragment, seed=args.seed, device=device, config=cfg, algo='dqn', total_samples=args.samples)
    iters = int(math.ceil(args.samples / float(args.envs * args.fragment)))
    t0 = time.perf_counter()
    out = []
    for it in range(iters):
        r = tr.iteration()
        r['wall_s'] = time.perf_counter() - t0
        r.update({k: v for k, v in r.pop('learner').items() if k != 'samples'})
        out.append(r)
        print(json.dumps(dict(r, config=name)), flush=True)
    tr.close()
    return {'config': cfg.to_dict(), 'iterations': out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--fragment', type=int, default=100)
    ap.add_argument('--samples', type=int, default=20000000)
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('dqn_per_door.py measures on a CUDA device; none is visible')
    device = torch.device('cuda:0')
    from paintrl_b200 import build
    build.build()
    res = {'gpu': gpu_info(), 'torch': torch.__version__, 'settings': 'door (Part_NO 0), C2: RGB, section-4 observation, '
           'discrete-4 actions, late termination, anchor starts, auto-reset', 'envs': args.envs, 'fragment': args.fragment,
           'configs': CONFIGS}
    res['learner_throughput'] = throughput(args, device)
    print(json.dumps(res['learner_throughput']), flush=True)
    res['kernel_times'] = kernel_times(device)
    print(json.dumps(res['kernel_times']), flush=True)
    res['curves'] = {name: curve(name, args, device) for name in CONFIGS}
    res['summary'] = {name: {'2M': at_steps(c['iterations'], 2000000), '20M': at_steps(c['iterations'], 20000000)}
                      for name, c in res['curves'].items()}
    res['gpu_after'] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f)
    print(json.dumps({'gpu': res['gpu'], 'learner_throughput': res['learner_throughput'], 'kernel_times': res['kernel_times'],
                      'summary': res['summary']}))


if __name__ == '__main__':
    main()
