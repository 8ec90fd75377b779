"""bench.py --dump-outputs on the GPU: the step path's dump is what the last timed step returned (replayed here with the
benchmark's own seeded inputs), and the --rollout dump is the last fragment."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir, *args):
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--envs', '512', '--no-extra', '--no-cpu-baseline', '--no-parity',
           '--no-flush', '--dump-outputs', str(out_dir)] + list(args)
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return {f[:-4]: np.load(str(out_dir / f)) for f in os.listdir(str(out_dir))}


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path, cuda_device):
    sys.path.insert(0, ROOT)
    import bench
    from paintrl_b200.batched_env import BatchedPaintEnv
    from paintrl_b200.config import EnvConfig
    steps, warmup = 5, 3
    got = _bench_dump(tmp_path / 'a', '--steps', str(steps), '--warmup', str(warmup))
    assert np.array_equal(got['env_ids'], np.arange(512))
    w = bench.WORKLOADS['c2']
    cfg = EnvConfig(w['extra'], auto_reset=True, seed=1234, **w['kw'])
    env = BatchedPaintEnv(512, cfg, device=cuda_device)
    actions, start, _ = bench.seeded_inputs(env, cfg, 0, cuda_device, steps, warmup, True)
    env.reset(start)
    for i in range(warmup + steps):
        env.step(actions[i])
    want = {'obs': env.obs, 'reward': env.reward, 'penalty': env.penalty, 'actual': env.actual, 'done': env.done,
            'new_texels': env.new_texels, 'next_obs': env.next_obs}
    assert sorted(got) == sorted(list(want) + ['env_ids'])
    for k, t in want.items():
        assert np.array_equal(got[k], t.cpu().numpy().astype(got[k].dtype)), k
    env.step(actions[warmup + steps])            # one step further is not what was dumped
    assert not np.array_equal(got['obs'], env.obs.cpu().numpy())
    env.close()


@pytest.mark.gpu
def test_rollout_dump_is_the_last_fragment(tmp_path, cuda_device):
    got = _bench_dump(tmp_path / 'r', '--workload', 'c5', '--rollout', '--steps', '1', '--warmup', '3')
    assert got['obs'].shape == (101, 512, 6) and got['term_obs'].shape == (100, 512, 6)
    for k in ('actions', 'reward', 'penalty', 'actual', 'done', 'new_texels', 'logp'):
        assert got[k].shape == (100, 512), k
    assert got['value'].shape == (101, 512) and got['logp'].dtype == np.float32 and got['obs'].dtype == np.float64
    # one fragment, step after step: where no episode ended, the next step starts from what this one returned
    going = got['done'] == 0
    assert going.any() and np.array_equal(got['obs'][1:][going], got['term_obs'][going])
