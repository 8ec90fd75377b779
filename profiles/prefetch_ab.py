#!/usr/bin/env python
"""A/B of the step's start order on one build: PAINTRL_START_ORDER=1 (the default: the one-kernel step loads the record
before the L2 sweep of the tables and copies the bit-plane in after the move phase) against 0 (sweep, copy, record).
The switch is read at handle creation.

    python profiles/prefetch_ab.py [--workloads c2,c3_late,c5,c4] [--rounds 6] [--steps 40] [--out FILE]

Per workload one handle per setting, all created from bench.py's seeded inputs (same seed, starts and actions).  The
settings step in turn, step by step, in a rotating order (ABCD, BCDA, ...), with bench.py's method: a 512 MiB write
flushes the L2 between steps and one CUDA event pair brackets each step.  Every step's outputs and, at the end of each
round, the status planes are compared with the first setting's: the switch must not change a bit.  Prints per
setting the median and the spread of us/step and the GPU's name, power limit and SM clock, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from paintrl_b200.batched_env import BatchedPaintEnv
from paintrl_b200.config import EnvConfig

SETTINGS = {
    'off': {'PAINTRL_START_ORDER': '0'},
    'on': {'PAINTRL_START_ORDER': '1'},
}
OUTS = ('obs', 'reward', 'penalty', 'actual', 'done', 'next_obs')


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader', '-i', '0'],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        return dict(zip(q.split(','), [v.strip() for v in r.stdout.strip().split(',')]))
    except (OSError, subprocess.SubprocessError):
        return {'name': torch.cuda.get_device_name(0)}


def make(key, names, device):
    w = bench.WORKLOADS[key]
    n_env, _ = bench.envs_of(w, 0, 1)
    cfg = EnvConfig(w['extra'], auto_reset=True, seed=1234, **w['kw'])
    envs = []
    for nm in names:
        saved = {k: os.environ.get(k) for k in SETTINGS[nm]}
        os.environ.update(SETTINGS[nm])
        try:
            envs.append(BatchedPaintEnv(n_env, cfg, device=device, texture_size=w.get('texture', (240, 240))))
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    return cfg, envs


def run(key, names, rounds, steps, warmup, device):
    cfg, envs = make(key, names, device)
    actions, start, _ = bench.seeded_inputs(envs[0], cfg, 0, device, rounds * steps, warmup, False)
    n_env_all = envs[0].num_envs
    for e in envs:
        e.reset(start)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=device)
    for i in range(warmup):
        for e in envs:
            flush.fill_(i & 0xff)
            e.step(actions[i])
    torch.cuda.synchronize(device)
    ev = {nm: [] for nm in names}
    per_round = {nm: [] for nm in names}
    mismatches = []
    t = warmup
    for r in range(rounds):
        marks = {nm: len(ev[nm]) for nm in names}
        for _ in range(steps):
            order = [(t + j) % len(names) for j in range(len(names))]
            outs = {}
            for j in order:
                e, nm = envs[j], names[j]
                flush.fill_(t & 0xff)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                e.step(actions[t])
                b.record()
                ev[nm].append((a, b))
                outs[nm] = {k: getattr(e, k).clone() for k in OUTS}
            for nm in names[1:]:
                for k in OUTS:
                    if not torch.equal(outs[names[0]][k], outs[nm][k]):
                        mismatches.append((t, nm, k))
            t += 1
        torch.cuda.synchronize(device)
        ids = torch.arange(min(n_env_all, 8192), dtype=torch.int32, device=device)
        st0 = envs[0].get_state(env_ids=ids)['status']
        for e, nm in zip(envs[1:], names[1:]):
            if not torch.equal(st0, e.get_state(env_ids=ids)['status']):
                mismatches.append((t, nm, 'status'))
        for nm in names:
            us = [a.elapsed_time(b) * 1e3 for a, b in ev[nm][marks[nm]:]]
            per_round[nm].append(float(np.median(us)))
    res = {}
    for nm in names:
        us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev[nm]])
        res[nm] = {'median_us': round(float(np.median(us)), 2), 'p10_us': round(float(np.percentile(us, 10)), 2),
                   'p90_us': round(float(np.percentile(us, 90)), 2),
                   'round_medians_us': [round(v, 2) for v in per_round[nm]],
                   'round_median_range_us': [round(min(per_round[nm]), 2), round(max(per_round[nm]), 2)]}
    for e in envs:
        e.close()
    assert not mismatches, 'settings disagree: %s' % mismatches[:10]
    return {'envs': n_env_all, 'steps_per_setting': rounds * steps, 'bit_identical': True, 'settings': res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='c2,c3_late,c5,c4')
    ap.add_argument('--settings', default=','.join(SETTINGS))
    ap.add_argument('--rounds', type=int, default=6)
    ap.add_argument('--steps', type=int, default=40, help='steps per setting per round')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('prefetch_ab.py needs a CUDA device')
    device = torch.device('cuda', 0)
    names = args.settings.split(',')
    doc = {'gpu_before': gpu_info(), 'method': 'settings interleaved step by step in rotating order; 512 MiB L2 flush '
           'before every step; one CUDA event pair per step', 'settings': {nm: SETTINGS[nm] for nm in names},
           'workloads': {}}
    for key in args.workloads.split(','):
        rounds, steps = (max(5, args.rounds // 2), max(5, args.steps // 4)) if key == 'c4' else (args.rounds, args.steps)
        r = run(key, names, rounds, steps, args.warmup, device)
        doc['workloads'][key] = r
        base = r['settings'][names[0]]['median_us']
        print('%-8s %6d envs' % (key, r['envs']), flush=True)
        for nm in names:
            s = r['settings'][nm]
            print('   %-6s median %8.2f us  (%+6.2f %%)  p10 %8.2f  p90 %8.2f  round medians %s' % (
                nm, s['median_us'], 100.0 * (s['median_us'] / base - 1.0), s['p10_us'], s['p90_us'],
                ' '.join('%.1f' % v for v in s['round_medians_us'])), flush=True)
    doc['gpu_after'] = gpu_info()
    print(json.dumps({'gpu': doc['gpu_before'], 'gpu_after': doc['gpu_after']}))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(doc, f, indent=1)


if __name__ == '__main__':
    main()
