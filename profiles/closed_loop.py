#!/usr/bin/env python
"""Closed-loop host stepping: a policy that picks action t + 1 from observation t, as zigzag.py / spiral.py and
RLlib's sampler drive PaintRL, through the host-buffer entry points on one GPU.

    python profiles/closed_loop.py [--out FILE]

Configuration: door panel, C2 settings (bench.py WORKLOADS['c2']), auto-reset on.  Policy: deterministic and
obs-dependent, vectorised NumPy -- the discrete action is the argmax of the four section values.  Two schedules on
the same seeds:
  * sync:      `step_host` on the whole batch, then act on its next_obs (the step cannot be submitted before the
               previous observation is back, so copies, the host's wake-up and the policy add to the device time);
  * ping-pong: the batch as two range groups on host slots 0 / 1 (`step_host_submit(subset=...)`): wait for group g,
               compute its actions, resubmit it, go on with the other group -- one group's copies and policy run
               while the other group's kernels do.
Sizes: 8192 environments (2 x 4096, one-kernel groups) and 65536 (2 x 32768, two-kernel groups); a group has to
fill a wave of the GPU, smaller groups are latency-bound and gain nothing from the overlap.

Prints ONE JSON line: env-steps/s per schedule (median of 5 timed repeats, wall clock of the whole loop ending in
a device synchronisation), where each schedule's host time per step goes (one extra run: policy, blocked in
step_host / step_host_wait, submit), the device time of one step of the whole batch and of each group (CUDA events,
device buffers, no host in the loop), a trajectory checksum per schedule (sha256 over obs, reward and done of every step of a
first, untimed run from fresh engines; equal checksums = the schedules computed the same trajectories), the GPU's
name, power limit and SM clock read in the same run."""
import argparse
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SIZES = ((8192, 1000), (65536, 300))     # (environments, steps per repeat): timed windows of a few hundred ms
REPEATS = 5


def greedy(obs):
    """argmax of the four section values (obs[:, 0:4]) as the discrete action."""
    return np.argmax(obs[:, :4], axis=1)


class Checksum(object):
    """sha256 per group over (obs, reward, done) of every step, in step order; the digest of the digests."""

    def __init__(self, groups):
        self.h = [hashlib.sha256() for _ in range(groups)]

    def add(self, g, obs, reward, done):
        for a in (obs, reward, done):
            self.h[g].update(np.ascontiguousarray(a).tobytes())

    def digest(self):
        return hashlib.sha256(b''.join(h.digest() for h in self.h)).hexdigest()


def run_sync(env, start, steps, check=None, split=None):
    """`split` (a dict): also sum the host time spent in the policy and inside step_host (blocked on the GPU)."""
    import torch
    half = env.num_envs // 2
    out = env.host_buffers()
    obs = env.reset(start).cpu().numpy()
    torch.cuda.synchronize(env.device)
    t0 = time.perf_counter()
    for _ in range(steps):
        if split is None:
            out = env.step_host(greedy(obs), out)
        else:
            ta = time.perf_counter()
            act = greedy(obs)
            tb = time.perf_counter()
            out = env.step_host(act, out)
            split['policy_s'] = split.get('policy_s', 0.0) + tb - ta
            split['step_host_s'] = split.get('step_host_s', 0.0) + time.perf_counter() - tb
        if check is not None:
            for g in range(2):
                rows = slice(g * half, (g + 1) * half)
                check.add(g, out['obs'][rows], out['reward'][rows], out['done'][rows])
        obs = out['next_obs']
    return env.num_envs * steps / (time.perf_counter() - t0)


def run_ping_pong(env, start, steps, check=None, split=None):
    """`split` (a dict): also sum the host time blocked in step_host_wait, in the policy and in step_host_submit."""
    import torch
    n = env.num_envs
    half = n // 2
    groups = [env.subset(range(0, half)), env.subset(range(half, n))]
    bufs = [env.host_buffers(n=half) for _ in range(2)]
    acts = [torch.zeros(half, dtype=torch.int64).pin_memory().numpy() for _ in range(2)]
    obs = env.reset(start).cpu().numpy()
    torch.cuda.synchronize(env.device)
    t0 = time.perf_counter()
    for g in range(2):
        acts[g][:] = greedy(obs[g * half:(g + 1) * half])
        env.step_host_submit(acts[g], bufs[g], slot=g, subset=groups[g])
    for t in range(steps):
        for g in range(2):
            ta = time.perf_counter()
            res = env.step_host_wait(g)
            tb = time.perf_counter()
            if check is not None:
                check.add(g, res['obs'], res['reward'], res['done'])
            if t + 1 < steps:
                acts[g][:] = greedy(res['next_obs'])
                tc = time.perf_counter()
                env.step_host_submit(acts[g], bufs[g], slot=g, subset=groups[g])
                if split is not None:
                    split['policy_s'] = split.get('policy_s', 0.0) + tc - tb
                    split['submit_s'] = split.get('submit_s', 0.0) + time.perf_counter() - tc
            if split is not None:
                split['wait_s'] = split.get('wait_s', 0.0) + tb - ta
    return n * steps / (time.perf_counter() - t0)


def device_us_per_step(env, subsets, steps=50):
    """Device time of one step of each of `subsets` (None = the whole batch), CUDA events around `steps` back-to-back
    device-buffer steps with fixed random actions: what the GPU needs, with no copy and no host in the loop."""
    import torch
    out = []
    rng = np.random.default_rng(1)
    for sub in subsets:
        n = env.num_envs if sub is None else sub.n
        acts = torch.as_tensor(rng.integers(0, 4, size=n), device=env.device)
        env.step(acts, subset=sub)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            env.step(acts, subset=sub)
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) * 1000.0 / steps)
    return out


def gpu_info(index):
    import torch
    info = {'gpu': torch.cuda.get_device_name(index)}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        info['power_limit_w'] = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
        info['sm_max_mhz'] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as exc:        # pragma: no cover - depends on the machine
        info['nvml_error'] = repr(exc)
    return info


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out', help='also write the JSON line to this file')
    args = ap.parse_args()
    import torch
    from bench import WORKLOADS, ClockSampler, physical_gpu_index
    from paintrl_b200.batched_env import BatchedPaintEnv
    from paintrl_b200.config import EnvConfig
    from paintrl_b200.partpack import PartPack

    if not torch.cuda.is_available():
        raise SystemExit('closed_loop.py measures on a CUDA device; there is none')
    device = torch.device('cuda:0')
    wl = WORKLOADS['c2']
    cfg = EnvConfig(dict(wl['extra']), auto_reset=True, **wl['kw'])
    pack = PartPack.for_part(cfg.part_no)
    line = dict(gpu_info(physical_gpu_index(0)), workload='closed loop, ' + wl['name'] + ', greedy section policy',
                repeats=REPEATS, timing='wall clock of the whole loop, median of the repeats', results=[])
    sampler = ClockSampler(physical_gpu_index(0))
    sampler.start()
    for n, steps in SIZES:
        start = np.random.default_rng(0).integers(0, pack.start_points(cfg.start_point_mode).shape[0], size=n).astype(np.int32)
        row = {'envs': n, 'groups': '2 x %d' % (n // 2), 'steps': steps}
        for name, run in (('sync', run_sync), ('ping_pong', run_ping_pong)):
            env = BatchedPaintEnv(n, cfg, device=device, pack=pack)
            check = Checksum(2)
            run(env, start, steps, check)                   # fresh engine: the checksum run, also the warm-up
            rates = [run(env, start, steps) for _ in range(REPEATS)]
            split = {}
            run(env, start, steps, None, split)          # one more run with the host-side split (not in the median)
            row[name + '_host_us_per_step'] = {k[:-2]: round(v * 1e6 / steps, 1) for k, v in sorted(split.items())}
            if name == 'sync':
                whole, g0, g1 = device_us_per_step(env, [None, env.subset(range(0, n // 2)), env.subset(range(n // 2, n))])
                row['device_us_per_step'] = {'whole': round(whole, 1), 'group0': round(g0, 1), 'group1': round(g1, 1)}
            row[name + '_env_steps_per_s'] = float(np.median(rates))
            row[name + '_spread'] = [float(min(rates)), float(max(rates))]
            row[name + '_checksum'] = check.digest()
            env.close()
            del env
        row['checksums_equal'] = row['sync_checksum'] == row['ping_pong_checksum']
        row['ping_pong_over_sync'] = row['ping_pong_env_steps_per_s'] / row['sync_env_steps_per_s']
        line['results'].append(row)
    line['clocks'] = sampler.stop()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
