#!/usr/bin/env python
"""Benchmark of the batched paint-simulation step (BASELINE.json metric: batched env steps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c3_late|c4|c5] [--impl reference]
                    [--dump-outputs DIR]

One process per GPU (torchrun for N > 1), environments sharded by index, no collective on the
step path.  A "step" is one `paintrl_step` over the whole per-GPU batch with random actions that
are already resident in HBM; `value` = env-steps of all ranks / max-over-ranks device time.
Prints ONE JSON line on rank 0 (see the driver contract in the task statement).

Timing: W >= 3 warm-up steps; each timed step is bracketed by CUDA events on the launch stream
and the L2 is flushed (a 512 MiB write) between timed steps, outside the event brackets, so every
step starts with its status planes in HBM, not in the 126 MB L2; `ms_per_step` is the mean
bracketed duration, max over ranks.

What the line carries besides the contract's keys:
  * `parity_check`: a sample of the environments of the TIMED run (rank 0), logged on the device outside the
    event brackets and replayed through the C oracle after the timed loop (oracle/replay.py) -- the oracle is
    the checker here, never the thing measured;
  * `roofline`: the HBM model of SURVEY.md section 8(d) (`achieved`, `frac`) next to what the kernels are
    actually bound by: `issue_frac` (warp instructions / issue slots of the timed duration) and
    `dram_gbs_measured`, from the ncu counters committed under profiles/ for this kernel source
    (`counters_source_sha` says whether they belong to the build that ran);
  * `extra.configs`: the other BASELINE configurations measured the same way with fewer steps (C3 sheet HSI
    hybrid, its steady-state variant with late termination, C4 2048x2048, C5 65536 environments sharded over
    the GPUs), each with its own p_reset / clocks / parity sample.
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASE = {'RENDER_HEIGHT': 720, 'RENDER_WIDTH': 960, 'Part_NO': 0, 'Expected_Episode_Length': 245,
        'EPISODE_MAX_LENGTH': 245, 'TERMINATION_MODE': 'late', 'SWITCH_THRESHOLD': 0.9,
        'START_POINT_MODE': 'anchor', 'TURNING_PENALTY': False, 'OVERLAP_PENALTY': False,
        'COLOR_MODE': 'RGB'}
_C3 = dict(BASE, Part_NO=1, COLOR_MODE='HSI', TURNING_PENALTY=True, OVERLAP_PENALTY=True, TERMINATION_MODE='hybrid')

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    'c2': dict(name='C2 door panel x4096 envs/GPU, RGB, START_POINT_MODE=anchor, random discrete-4 actions, '
                    'OBS_MODE=section-4, late termination, auto-reset',
               extra=dict(BASE), kw={}, envs_per_gpu=4096, scaling='weak'),
    # configs[2].  Under random actions hybrid termination ends every episode at its first step (p_reset = 1):
    # this line measures reset + one stamp; c3_late is the same batch in steady state.
    'c3': dict(name='C3 quadratic sheet x16384 envs/GPU, HSI, turning+overlap penalties, hybrid termination',
               extra=dict(_C3), kw={}, envs_per_gpu=16384, scaling='weak'),
    'c3_late': dict(name='C3 steady state: quadratic sheet x16384 envs/GPU, HSI, turning+overlap penalties, LATE termination '
                         '(episodes last: the HSI stamp / thickness path every step)',
                    extra=dict(_C3, TERMINATION_MODE='late'), kw={}, envs_per_gpu=16384, scaling='weak'),
    # configs[3]: continuous 2-D actions, grid observation, every start point, 2048x2048 synthetic texture
    'c4': dict(name='C4 door panel 2048x2048 synthetic texture x8192 envs/GPU, RGB, continuous ACTION_SHAPE=2, OBS_MODE=grid-4, '
                    'START_POINT_MODE=all, late termination, auto-reset',
               extra=dict(BASE, START_POINT_MODE='all'),
               kw=dict(action_mode='continuous', action_shape=2, obs_mode='grid', obs_grad=4),
               texture=(2048, 2048), envs_per_gpu=8192, scaling='weak'),
    # SURVEY 8(f) row f3: Robot.PAINT_METHOD = 'normal' -- a fan of 124 rays per shot instead of the ball query
    'c2_normal': dict(name='C2 settings with the normal paint method (robot.py:172, 414-417: 124-ray beam fan per shot, nearest texel per hit), '
                           'door panel x4096 envs/GPU',
                      extra=dict(BASE), kw=dict(paint_method='normal'), envs_per_gpu=4096, scaling='weak'),
    # configs[4] env side: 65536 envs sharded over the GPUs (strong scaling)
    'c5': dict(name='C5 door panel, 65536 envs sharded over N GPUs, C2 settings',
               extra=dict(BASE), kw={}, envs_total=65536, scaling='strong'),
}

METRIC = 'batched env steps/sec'
UNIT = 'env-steps/s'
N_SMS = 148
DUMP_BYTES = 60 << 20      # --dump-outputs: the .npy files stay under 64 MB, headers included


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def kernel_source_sha():
    """Hash of the CUDA sources + ABI header: ties committed ncu counters to the build they were captured from."""
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, 'paintrl_b200', 'csrc')
    for p in sorted(os.listdir(csrc)) + [os.path.join(ROOT, 'include', 'paintrl.h')]:
        path = p if os.path.isabs(p) else os.path.join(csrc, p)
        with open(path, 'rb') as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def captured_counters(workload_key):
    """Per-step ncu counters of this workload (profiles/kernel_counters.json, written by profiles/capture_counters.py
    from an `ncu` pass of this very command): DRAM bytes read + written and warp instructions executed, both
    kernels of the step summed.  Returns (dict or None, sha of the source they were captured from)."""
    path = os.path.join(ROOT, 'profiles', 'kernel_counters.json')
    try:
        with open(path) as f:
            doc = json.load(f)
        return doc.get('workloads', {}).get(workload_key), doc.get('source_sha')
    except (OSError, ValueError):
        return None, None


def algorithmic_bytes(status_bytes, n_front, obs_dim, act_dim, scan, u_mean, p_reset):
    """SURVEY.md section 8(d): B_alg per env-step."""
    return (status_bytes * n_front * (1 if scan else 0) + 2 * status_bytes * u_mean + 8 * obs_dim + 8 * act_dim
            + 40 + 2 * 160 + p_reset * status_bytes * n_front)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""
    REASONS = {0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown'}

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.error = index, [], set(), None, None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self._stop_evt.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.002)
        except Exception as exc:      # pragma: no cover - depends on the box
            self.error = repr(exc)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        out = {'sm_mhz': float(np.median(self.samples)) if self.samples else None, 'sm_max_mhz': self.max_mhz,
               'reasons': sorted(self.reasons), 'samples': len(self.samples)}
        if self.error:
            out['error'] = self.error
        return out


def physical_gpu_index(local_index):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES')
    if vis:
        try:
            return int(vis.split(',')[local_index])
        except (ValueError, IndexError):
            return local_index
    return local_index


def pin_to_gpu_numa_node(index):
    """Keep this rank's host thread on the CPUs NVML reports as local to its GPU (the e2e leg is a host loop per rank:
    eight of them on one box should not wander across sockets).  Returns the number of CPUs in the mask, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        return None
    return None


def dump_outputs(out_dir, arrays, env_axis=0):
    """--dump-outputs: `arrays` (name -> device tensor, environments along `env_axis`) as out_dir/<name>.npy, float32
    tensors and flags in float32, everything else in float64, and the environments written as env_ids.npy.  Above
    DUMP_BYTES in all, a fixed seeded sample of the environments is written, the same one in every run."""
    import torch
    n_env = next(iter(arrays.values())).shape[env_axis]
    as_f32 = {k: t.dtype in (torch.float32, torch.uint8, torch.bool) for k, t in arrays.items()}
    per_env = 8 + sum((4 if as_f32[k] else 8) * (t.numel() // n_env) for k, t in arrays.items())
    keep = min(n_env, DUMP_BYTES // per_env)
    ids = np.arange(n_env) if keep == n_env else np.sort(np.random.default_rng(0).choice(n_env, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'env_ids.npy'), ids.astype(np.float64))
    for k, t in arrays.items():
        rows = t.index_select(env_axis, torch.as_tensor(ids, device=t.device)).cpu().numpy()
        np.save(os.path.join(out_dir, k + '.npy'), rows.astype(np.float32 if as_f32[k] else np.float64))


def workload_pack(workload, cfg, rasterizer='oracle'):
    """The part pack of a workload for the CPU legs (texels of synthetic textures from the oracle's own rasteriser)."""
    from paintrl_b200.partpack import PartPack
    pack = PartPack.for_part(cfg.part_no)
    if 'texture' in workload:
        from oracle.oracle import retextured_pack
        pack = retextured_pack(pack, *workload['texture'])
    return pack


def workload_config(workload, cfg, n_front, n_env, total_envs, world_size):
    """`config` of the JSON line: what was run, identical for both arms (`--impl reference` prints the same keys
    and values; its own, bounded environment sample is stated in `cpu_baseline`)."""
    return {'workload': workload['name'], 'envs_per_gpu': int(n_env), 'envs_total': int(total_envs),
            'n_front_texels': int(n_front), 'status_bytes_per_texel': 1 if cfg.color_mode == 'RGB' else 2,
            'obs_dim': int(cfg.obs_dim), 'parallelism': 'env-sharded x%d, no step-path collective' % world_size}


def envs_of(workload, rank, world_size, override=None):
    from paintrl_b200 import sharding
    if override:
        return int(override), int(override) * world_size
    if 'envs_total' in workload:
        lo, hi = sharding.shard_range(workload['envs_total'], rank, world_size)
        return hi - lo, workload['envs_total']
    return workload['envs_per_gpu'], workload['envs_per_gpu'] * world_size


def cpu_baseline_sample(workload, seconds=12.0, threads=None):
    """The oracle's C restatement (kind "port") on the host cores: a bounded sample of the same
    workload (same part, config, start mode, random discrete actions, reset on done)."""
    from oracle.oracle import OracleBatch
    from paintrl_b200.config import EnvConfig
    threads = threads or os.cpu_count() or 1
    cfg = EnvConfig(workload['extra'], **workload['kw'])
    pack = workload_pack(workload, cfg)
    n_env = (16 if 'texture' not in workload else 1) * threads
    ora = OracleBatch(pack, cfg, n_env, threads=threads)
    rng = np.random.default_rng(1234)
    n_starts = pack.start_points(cfg.start_point_mode).shape[0]
    ora.reset(rng.integers(0, n_starts, size=n_env))
    steps = 0
    t0 = time.perf_counter()
    while True:
        if cfg.action_mode == 'discrete':
            acts = rng.integers(0, cfg.discrete_granularity, size=n_env)
        else:
            acts = rng.uniform(-1, 1, size=(n_env, cfg.action_dim))
        _, _, _, _, done = ora.step(acts)
        ids = np.flatnonzero(done)
        if len(ids):
            ora.reset(rng.integers(0, n_starts, size=len(ids)), env_ids=list(ids))
        steps += n_env
        dt = time.perf_counter() - t0
        if dt >= seconds:
            break
    ora.close()
    return {'value': steps / dt, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'envs': n_env, 'n_front_texels': int(pack.n_texels),
            'sample': '%d envs x %d steps of the same workload (C restatement oracle/paint_oracle.c, OpenMP, '
                      '%.1f s); the Python reference itself runs ~44 env-steps/s/core (BASELINE.md)'
                      % (n_env, steps // n_env, dt)}


def run_reference(args, workload, rank, world_size):
    """--impl reference: the reference path's CPU implementation on the host cores (the oracle
    port: the Python reference cannot travel to the GPU box), same config / metric / unit."""
    if rank != 0:
        return
    from paintrl_b200.config import EnvConfig
    per_step = max(2.0, min(20.0, 60.0 / max(1, args.steps + args.warmup)))
    per_step = float(os.environ.get('PAINTRL_BENCH_REFERENCE_SECONDS', per_step))     # tests shorten the sample
    for _ in range(min(args.warmup, 1)):
        cpu_baseline_sample(workload, seconds=0.5)
    samples = [cpu_baseline_sample(workload, seconds=per_step) for _ in range(max(1, min(args.steps, 5)))]
    value = float(np.mean([s['value'] for s in samples]))
    base = dict(samples[-1], value=value)
    cfg = EnvConfig(workload['extra'], **workload['kw'])
    n_env, total = envs_of(workload, 0, args.gpus, args.envs)
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': None, 'higher_is_better': True,
            'scaling': workload['scaling'], 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(workload, cfg, base['n_front_texels'], n_env, total, args.gpus), 'cpu_baseline': base,
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def run_rollout(args, workload, env, cfg, rank, world_size, device, warmup, dump_dir=None):
    """--rollout: fragments of 100 steps collected by paintrl_b200.rollout (policy obs->256->128->{logits, value}
    evaluated and sampled on the GPU, paint_ppo.py:179-190), one all-reduce of rollout statistics per fragment."""
    import torch
    import torch.distributed as dist
    from paintrl_b200 import rollout
    T = 100
    n_out = cfg.discrete_granularity if cfg.action_mode == 'discrete' else cfg.action_dim
    policy = rollout.MlpPolicy(env.obs_dim, n_out, device=device, seed=rank, discrete=cfg.action_mode == 'discrete')
    worker = rollout.RolloutWorker(env, policy, fragment_length=T, use_cuda_graph=not args.no_graph)
    worker.start()
    for _ in range(max(2, min(warmup, 3))):      # the first fragment runs eagerly, the second captures the CUDA graph
        worker.collect(); worker.advance()
    torch.cuda.synchronize(device)
    if world_size > 1:
        dist.barrier()
    sampler = ClockSampler(physical_gpu_index(int(os.environ.get('LOCAL_RANK', 0))))
    sampler.start()
    s0 = env.stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total = {}
    e0.record()
    for _ in range(args.steps):
        _, st = worker.collect()
        worker.advance()
        red = rollout.iteration_stats(st, device=device)
        for k, v in red.items():
            total[k] = max(total.get(k, 0.0), v) if k.startswith('max') else total.get(k, 0.0) + v
    e1.record()
    torch.cuda.synchronize(device)
    if world_size > 1:
        dist.barrier()
    clocks = sampler.stop()
    if dump_dir and rank == 0:
        f = worker.frag
        dump_outputs(dump_dir, {k: getattr(f, k) for k in ('obs', 'term_obs', 'actions', 'reward', 'penalty', 'actual', 'done',
                                                          'new_texels', 'logp', 'value')}, env_axis=1)
    s1 = env.stats()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    if rank == 0:
        print(json.dumps({
            'metric': METRIC, 'value': total['env_steps'] / (ms * 1e-3), 'unit': UNIT, 'n_gpus': world_size, 'steps': args.steps,
            'warmup': warmup, 'ms_per_step': ms / (args.steps * T), 'higher_is_better': True, 'scaling': workload['scaling'],
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': workload['name'] + '; rollout fragments of %d steps with the on-GPU MLP policy '
                       '(obs->256->128->logits+value, %s, random init), one stats all-reduce per fragment; %s' % (
                           T, policy.describe() if hasattr(policy, 'describe') else 'FP32',
                           'whole fragment replayed from one CUDA graph' if worker._graph is not None else 'eager launches (%s)' % (worker.graph_error or 'graph off')),
                       'envs_per_gpu': env.num_envs, 'l2': 'not flushed (policy and fragment traffic between steps)',
                       'timing': 'CUDA events around all fragments, max over ranks',
                       'parallelism': 'env-sharded x%d, no step-path collective' % world_size},
            'clocks': clocks, 'gpu_launches': s1['kernel_launches'] - s0['kernel_launches'], 'rollout_stats': total}), flush=True)
    env.close()
    if world_size > 1:
        dist.barrier()
        dist.destroy_process_group()


def seeded_inputs(env, cfg, rank, device, steps, warmup, e2e):
    """The step benchmark's inputs, seeded by rank: random actions [rows, n_env(, action_dim)] for the warm-up, timed
    and e2e steps, and one start index per environment.  Returns (actions, start, e2e_steps)."""
    import torch
    n_env = env.num_envs
    gen = torch.Generator(device=device)
    gen.manual_seed(1234 + rank)
    e2e_steps = max(10, min(steps, 200)) if e2e else 0
    total = warmup + max(steps, e2e_steps)
    if cfg.action_mode == 'discrete':
        actions = torch.randint(0, cfg.discrete_granularity, (total, n_env), generator=gen, device=device,
                                dtype=torch.int64)
    else:
        actions = torch.rand((total, n_env, cfg.action_dim), generator=gen, device=device, dtype=torch.float64) * 2 - 1
    gs = torch.Generator(device=device)
    gs.manual_seed(rank)
    start = torch.randint(0, env.n_starts, (n_env,), generator=gs, device=device, dtype=torch.int32)
    return actions, start, e2e_steps


def measure(key, args, rank, local_rank, world_size, device, steps, warmup, e2e=True, parity_envs=128, rollout=False,
            dump_dir=None):
    """One workload on this rank's GPU: W warm-up steps, `steps` timed steps (CUDA events per step, L2 flushed in
    between), the host-buffer (e2e) leg, the oracle replay of a sample of the timed run.  Every rank returns the
    same reduced numbers; rank 0 also the roofline / parity details, and writes what the last timed step returned
    to `dump_dir` when one is given."""
    import torch
    import torch.distributed as dist
    from paintrl_b200 import sharding
    from paintrl_b200.batched_env import BatchedPaintEnv
    from paintrl_b200.config import EnvConfig
    workload = WORKLOADS[key]
    n_env, _ = envs_of(workload, rank, world_size, args.envs if key == args.workload else None)
    cfg = EnvConfig(workload['extra'], auto_reset=True, seed=1234 + rank, **workload['kw'])
    t_create = time.perf_counter()
    env = BatchedPaintEnv(n_env, cfg, device=device, texture_size=workload.get('texture', (240, 240)))
    torch.cuda.synchronize(device)
    create_s = time.perf_counter() - t_create
    if rollout:
        run_rollout(args, workload, env, cfg, rank, world_size, device, warmup, dump_dir=dump_dir)
        return None
    actions, start, e2e_steps = seeded_inputs(env, cfg, rank, device, steps, warmup, e2e)
    env.reset(start)
    flush = None if args.no_flush else torch.empty(512 << 20, dtype=torch.uint8, device=device)
    drain = torch.empty(256 << 20, dtype=torch.uint8, device=device) if (flush is not None and args.flush_mode == 'write+read') else None

    def flush_l2(i):
        """Evict the environments' state from the 126 MB L2: write a 512 MiB buffer.  'write+read' then reads another
        256 MiB buffer so that the L2 is left holding CLEAN foreign lines (the write alone leaves it full of dirty
        lines, whose write-backs the timed step would pay for on every miss)."""
        if flush is not None:
            flush.fill_(i & 0xff)
            if drain is not None:
                drain_sink.add_(drain.view(torch.int64)[::8].sum())
    drain_sink = torch.zeros((), dtype=torch.int64, device=device)

    # the parity sample of the timed run (rank 0): logged on the device between the event brackets
    rec = None
    if parity_envs and rank == 0:
        from oracle.replay import SubsetRecorder, sample_env_ids
        ids = sample_env_ids(n_env, parity_envs, seed=11)
        rec = SubsetRecorder(env, ids, warmup + steps)

    def barrier():
        torch.cuda.synchronize(device)
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for i in range(warmup):
        flush_l2(i)
        env.step(actions[i])
        if rec is not None:
            rec.record(actions[i])
    barrier()
    s0 = env.stats()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    acc = torch.zeros(4, dtype=torch.float64, device=device)   # rollout statistics, accumulated outside the timed event pairs
    t_wall = time.perf_counter()
    for i in range(steps):
        flush_l2(i)
        starts[i].record()
        env.step(actions[warmup + i])
        stops[i].record()
        acc += torch.stack([env.reward.sum(), env.penalty.sum(), env.actual.sum(), env.new_texels.sum().to(torch.float64)])
        if rec is not None:
            rec.record(actions[warmup + i], status=(i == steps - 1))
    barrier()
    wall_s = time.perf_counter() - t_wall
    clocks = sampler.stop()
    if dump_dir and rank == 0:        # before the legs below step the same environments again
        dump_outputs(dump_dir, {'obs': env.obs, 'reward': env.reward, 'penalty': env.penalty, 'actual': env.actual,
                                'done': env.done, 'new_texels': env.new_texels, 'next_obs': env.next_obs})
    s1 = env.stats()
    step_ms = np.array([a.elapsed_time(b) for a, b in zip(starts, stops)])
    dev_ms = float(step_ms.sum())
    # informational: the same steps back to back under ONE event pair (warm L2, no flush, no per-step events)
    b2b = min(steps, 100)
    eb0, eb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eb0.record()
    for i in range(b2b):
        env.step(actions[warmup + i])
    eb1.record()
    torch.cuda.synchronize(device)
    b2b_us = eb0.elapsed_time(eb1) * 1e3 / b2b

    # ---- end-to-end through the host-buffer API (pinned host actions in, results out, every step)
    e2e_s, act_bytes, d2h_bytes, e2e_api = 0.0, 0, 0, None
    if e2e:
        host_out = [env.host_buffers(pinned=True), env.host_buffers(pinned=True)]
        host_actions = actions[warmup:warmup + e2e_steps].cpu().pin_memory().numpy()
        pipelined = hasattr(env, 'step_host_submit') and not args.e2e_sync
        e2e_api = ('BatchedPaintEnv.step_host_submit / step_host_wait -> paintrl_step_host_submit / _wait (two slots: step t+1 is '
                   'submitted before step t is waited for)') if pipelined else 'BatchedPaintEnv.step_host -> paintrl_step_host'

        def e2e_pass(n):
            cs = 0.0
            if not pipelined:
                for i in range(n):
                    env.step_host(host_actions[i], host_out[0])
                    cs += float(host_out[0]['actual'][0])
                return cs
            env.step_host_submit(host_actions[0], host_out[0], slot=0)
            for i in range(n):
                if i + 1 < n:
                    env.step_host_submit(host_actions[i + 1], host_out[(i + 1) & 1], slot=(i + 1) & 1)
                env.step_host_wait(slot=i & 1)
                cs += float(host_out[i & 1]['actual'][0])
            return cs
        e2e_pass(3)
        barrier()
        e2e_runs = []
        checksum = 0.0
        for rep in range(5):                      # median of 5 repeats: the host side of this leg is noisy
            t0 = time.perf_counter()
            checksum += e2e_pass(e2e_steps)
            torch.cuda.synchronize(device)
            e2e_runs.append(time.perf_counter() - t0)
        e2e_s = float(np.median(e2e_runs))
        act_bytes = int(host_actions[0].nbytes)
        d2h_bytes = int(sum(host_out[0][k].nbytes for k in ('obs', 'reward', 'penalty', 'actual', 'next_obs', 'done')))

    # ---- reduce over ranks: max time, summed work
    t = torch.tensor([dev_ms, e2e_s], dtype=torch.float64, device=device)
    w = torch.tensor([float(n_env)], dtype=torch.float64, device=device)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
    dev_ms_max, e2e_s_max = float(t[0]), float(t[1])
    total_envs = int(w[0])
    rollout_stats = sharding.allreduce_stats({
        'env_steps': s1['env_steps'] - s0['env_steps'], 'episodes': s1['episodes_ended'] - s0['episodes_ended'],
        'sum_reward': float(acc[0]), 'sum_penalty': float(acc[1]), 'sum_return': float(acc[2]), 'new_texels': float(acc[3]),
        'max_step_ms': float(step_ms.max())}, device=device)

    res = {'key': key, 'workload': workload, 'cfg': cfg, 'n_env': n_env, 'total_envs': total_envs, 'steps': steps, 'warmup': warmup,
           'value': total_envs * steps / (dev_ms_max * 1e-3), 'ms_per_step': dev_ms_max / steps, 'clocks': clocks,
           'rollout_stats': rollout_stats, 'wall_s': wall_s, 'create_s': create_s, 'n_front': env.n_texels,
           'gpu_launches': s1['kernel_launches'] - s0['kernel_launches'],
           'step_us': {'mean': float(step_ms.mean() * 1e3), 'median': float(np.median(step_ms) * 1e3), 'p10': float(np.percentile(step_ms, 10) * 1e3),
                       'p90': float(np.percentile(step_ms, 90) * 1e3), 'max': float(step_ms.max() * 1e3),
                       'back_to_back_warm_l2': b2b_us}}
    if e2e:
        res['e2e'] = {'value': total_envs * e2e_steps / e2e_s_max, 'unit': UNIT, 'h2d_bytes_per_step': act_bytes,
                      'd2h_bytes_per_step': d2h_bytes, 'steps': e2e_steps, 'repeats': 5, 'statistic': 'median repeat', 'api': e2e_api}
    if rank == 0:
        steps_done = s1['env_steps'] - s0['env_steps']
        u_mean = (s1['footprint_texels'] - s0['footprint_texels']) / max(1, steps_done)
        p_reset = (s1['episodes_ended'] - s0['episodes_ended']) / max(1, steps_done)
        status_bytes = 1 if cfg.color_mode == 'RGB' else 2
        b_alg = algorithmic_bytes(status_bytes, env.n_texels, env.obs_dim, cfg.action_dim,
                                  cfg.obs_mode != 'simple', u_mean, p_reset)
        kernel_ms = dev_ms / steps                      # rank 0's own mean launch duration
        achieved = b_alg * n_env / (kernel_ms * 1e-3) / 1e9
        peak, peak_src = measured_peaks()
        counters, counters_sha = captured_counters(key)
        sha = kernel_source_sha()
        sm_hz = (clocks.get('sm_mhz') or 1965.0) * 1e6
        per_step_launches = (s1['kernel_launches'] - s0['kernel_launches']) / float(max(1, steps))
        if cfg.paint_method == 'normal':
            kernel_desc = 'paintrl::move_kernel + paintrl::paint_normal_kernel (beam-fan paint method: two launches per step)'
        elif per_step_launches < 1.5:
            kernel_desc = ('paintrl::step_fused_kernel (one launch per step: a warp runs the move and the paint phase of its environment; '
                           'batches below 16384 environments per GPU)')
        else:
            kernel_desc = ('paintrl::move_fast_kernel + paintrl::paint_kernel (two launches per step; the paint grid is a programmatic '
                           'dependent launch whose warps acquire per-environment flags)')
        roof = {'bound': 'hbm', 'model_bound': 'hbm (SURVEY 8d algorithmic-bytes model: achieved / peak / frac are on that model)',
                'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': None, 'traffic_unit': 'bytes per step (ncu capture, profiles/kernel_counters.json)',
                'peak_source': peak_src,
                'kernel': kernel_desc,
                'kernel_ms': kernel_ms, 'algorithmic_bytes_per_env_step': b_alg,
                'footprint_union_texels_mean': u_mean, 'p_reset': p_reset,
                'ray_full_scans_per_env_step': (s1['ray_full_scans'] - s0['ray_full_scans']) / max(1, steps_done),
                'move_bailouts_per_env_step': (s1['move_bailouts'] - s0['move_bailouts']) / max(1, steps_done),
                'bound_measured': None, 'issue_frac': None, 'dram_gbs_measured': None, 'dram_frac_measured': None,
                'kernel_source_sha': sha, 'counters_source_sha': counters_sha,
                'counters_current': bool(counters is not None and counters_sha == sha)}
        if counters:
            scale = n_env / float(counters.get('envs_per_gpu', n_env))      # counters are per step of the captured batch size
            dram = counters['dram_bytes_per_step'] * scale
            insts = counters['warp_insts_per_step'] * scale
            roof['traffic'] = dram
            roof['dram_gbs_measured'] = dram / (kernel_ms * 1e-3) / 1e9
            roof['dram_frac_measured'] = roof['dram_gbs_measured'] / peak
            roof['warp_insts_per_env_step'] = insts / n_env
            roof['issue_frac'] = insts / (N_SMS * 4 * sm_hz * kernel_ms * 1e-3)
            # what the step is bound by, read off the two measured fractions: neither reaches its roof when
            # both are low -- the remainder is dependent latency (FP64 chains, table lookups) per environment
            roof['serialized_kernel_us'] = {k: v['us'] for k, v in counters.get('kernels', {}).items()}
            if roof['dram_frac_measured'] >= 0.6:
                roof['bound_measured'] = 'hbm'
            elif roof['issue_frac'] >= 0.6:
                roof['bound_measured'] = 'instruction issue'
                roof['bound'] = 'issue'
            else:
                roof['bound'] = 'latency'
                roof['bound_measured'] = ('latency (dependent FP64 / lookup chains per environment; issue slots %.0f %% busy, '
                                          'DRAM %.1f %% of peak -- NOT hbm-bound; `frac` is the algorithmic-bytes model of SURVEY 8d)'
                                          % (100 * roof['issue_frac'], 100 * roof['dram_frac_measured']))
        res['roofline'] = roof
        res['state'] = {'state_bytes_per_gpu': env.state_bytes_per_env * n_env,
                        'state_fits_l2': bool(env.state_bytes_per_env * n_env < 126e6)}
        if rec is not None:
            from oracle.replay import replay_subset
            t0 = time.perf_counter()
            pack = workload_pack(workload, cfg) if 'texture' in workload else env.pack
            chk = replay_subset(pack, cfg, rec.env_ids, start.cpu().numpy()[rec.env_ids], rec.host(), status=rec.status)
            chk['seconds'] = time.perf_counter() - t0
            chk['what'] = ('%d environments of the timed run (warm-up + timed steps, rank 0) replayed through the C oracle: done / obs / '
                           'reward / penalty / next_obs every step, status planes after the last step' % chk['envs'])
            res['parity_check'] = chk
    env.close()
    del env, actions, flush, drain
    torch.cuda.empty_cache()
    return res


def compact(res):
    """Sub-result of an extra configuration for `extra.configs`."""
    out = {'workload': res['workload']['name'], 'value': res['value'], 'unit': UNIT, 'ms_per_step': res['ms_per_step'],
           'steps': res['steps'], 'warmup': res['warmup'], 'envs_per_gpu': res['n_env'], 'envs_total': res['total_envs'],
           'scaling': res['workload']['scaling'], 'clocks': res['clocks'], 'gpu_launches': res['gpu_launches'],
           'create_s': res['create_s']}
    if 'e2e' in res:
        out['e2e'] = res['e2e']
    roof = res.get('roofline')
    if roof:
        out['roofline'] = {k: roof[k] for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic', 'kernel_ms', 'p_reset',
                                                'footprint_union_texels_mean', 'algorithmic_bytes_per_env_step', 'move_bailouts_per_env_step', 'bound_measured',
                                                'issue_frac', 'dram_gbs_measured', 'counters_current')}
    if 'parity_check' in res:
        out['parity_check'] = {k: res['parity_check'][k] for k in ('envs', 'steps', 'ok', 'exact', 'episodes', 'mismatch')}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=500)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS))
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--envs', type=int, default=None, help='override environments per GPU')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-flush', action='store_true', help='keep the L2 warm between steps (not the headline)')
    ap.add_argument('--flush-mode', default='write', choices=['write', 'write+read'],
                    help="how the L2 is flushed between timed steps: a 512 MiB write, or that write followed by a 256 MiB read")
    ap.add_argument('--no-graph', action='store_true', help='--rollout: keep the eager per-step launch loop (no CUDA graph)')
    ap.add_argument('--no-extra', action='store_true', help='skip the other BASELINE configurations (extra.configs)')
    ap.add_argument('--no-parity', action='store_true', help='skip the oracle replay of the timed run')
    ap.add_argument('--e2e-sync', action='store_true', help='e2e leg through the synchronous paintrl_step_host only')
    ap.add_argument('--rollout', action='store_true',
                    help='time whole rollout fragments (on-GPU MLP policy + env step, paintrl_b200.rollout) instead of bare steps; '
                         '--steps counts fragments of 100 steps (BASELINE config C5 / paint_ppo.py sample_batch_size)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="after the timed steps, write what the last one returned (rank 0's environments; with --rollout the "
                         'last fragment) as DIR/<name>.npy, under 64 MB: compares two builds run with the same arguments')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU path; --impl reference has none')
    workload = WORKLOADS[args.workload]

    from paintrl_b200 import sharding
    rank, local_rank, world_size = sharding.world()
    if args.impl == 'reference':
        run_reference(args, workload, rank, world_size)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    warmup = max(args.warmup, 3)
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    sharding.init_process_group()
    numa_cpus = pin_to_gpu_numa_node(physical_gpu_index(local_rank)) if world_size > 1 else None

    parity_envs = 0 if args.no_parity else 128
    res = measure(args.workload, args, rank, local_rank, world_size, device, args.steps, warmup, e2e=True,
                  parity_envs=parity_envs, rollout=args.rollout, dump_dir=args.dump_outputs)
    if res is None:
        return

    # ---- the other BASELINE configurations, fewer steps each (N > 1: only the strong-scaling C5)
    extras = {}
    if not args.no_extra and args.workload == 'c2' and args.envs is None:
        keys = ['c3', 'c3_late', 'c4', 'c5', 'c2_normal'] if world_size == 1 else ['c5']
        xsteps = max(10, min(args.steps, 60))
        for k in keys:
            try:
                r = measure(k, args, rank, local_rank, world_size, device, xsteps if k != 'c4' else max(5, xsteps // 3),
                            3, e2e=(k != 'c4'), parity_envs=0 if args.no_parity else (16 if k == 'c4' else 64))
                if rank == 0:
                    extras[k] = compact(r)
            except Exception as exc:            # an extra must never take the headline line down with it
                if rank == 0:
                    extras[k] = {'error': repr(exc)}
                if world_size > 1:
                    raise

    if rank == 0:
        cfg = res['cfg']
        config = workload_config(workload, cfg, res['n_front'], res['n_env'], res['total_envs'], world_size)
        line = {
            'metric': METRIC, 'value': res['value'], 'unit': UNIT, 'n_gpus': world_size, 'steps': args.steps,
            'warmup': warmup, 'ms_per_step': res['ms_per_step'], 'higher_is_better': True,
            'scaling': workload['scaling'], 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': config,
            'timing': dict(res['state'], l2='warm (no flush)' if args.no_flush else ('flushed with a 512 MiB write between timed steps' + (' followed by a 256 MiB read (L2 left clean)' if args.flush_mode == 'write+read' else '')),
                           method='CUDA events per step on the launch stream, summed; max over ranks'),
            'clocks': res['clocks'], 'e2e': dict(res['e2e'], host_thread_cpus=numa_cpus), 'gpu_launches': res['gpu_launches'], 'roofline': res['roofline'],
            'rollout_stats': res['rollout_stats'], 'wall_s_timed_region': res['wall_s'], 'step_us': res['step_us'],
        }
        if 'parity_check' in res:
            line['parity_check'] = res['parity_check']
        if extras:
            line['extra'] = {'configs': extras}
        if world_size == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline_sample(workload)
            one = cpu_baseline_sample(workload, seconds=3.0, threads=1)      # BASELINE.md section 3: one core beside all cores
            line['cpu_baseline']['single_core'] = {'value': one['value'], 'unit': UNIT, 'cores': 1, 'sample': one['sample']}
        print(json.dumps(line), flush=True)
    if world_size > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
