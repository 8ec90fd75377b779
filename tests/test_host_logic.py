"""CPU checks of the host-side mirror: configuration parsing (robot_gym_env.py:126-157, 240-252),
the discrete-action direction table (robot_gym_env.py:342-347, robot.py:151-160, 352-358), the
algorithmic-bytes model of bench.py, and index sharding including a world_size-2 gloo run."""
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_extra_config_keys_are_all_required():
    from paintrl_b200.config import DEFAULT_EXTRA_CONFIG, EnvConfig
    EnvConfig(dict(DEFAULT_EXTRA_CONFIG))
    for key in DEFAULT_EXTRA_CONFIG:
        cfg = dict(DEFAULT_EXTRA_CONFIG)
        del cfg[key]
        with pytest.raises(KeyError):          # the reference reads every key with [] (:240-252)
            EnvConfig(cfg)


def test_obs_dim_follows_the_reference_spaces():
    from paintrl_b200.config import obs_dim
    assert obs_dim('section', 4) == 6 and obs_dim('section', 8) == 10      # :166-167
    assert obs_dim('grid', 4) == 16 and obs_dim('grid', 10) == 100         # :168-169
    assert obs_dim('simple', 4) == 2                                       # :170-171
    assert obs_dim('discrete', 4) == 5                                     # :172-173


def test_discrete_table_carries_the_reference_residues():
    from paintrl_b200.config import STEP_SIZE, discrete_table
    t = discrete_table(4)
    # a = 0..3 -> act = -1, -.5, 0, .5 -> phi = 0, pi/2, pi, 3pi/2 (robot.py:153)
    for a, act in enumerate((-1.0, -0.5, 0.0, 0.5)):
        phi = (act + 1) * np.pi
        assert t[a, 0] == np.cos(phi) and t[a, 1] == np.sin(phi)
        d1, d2 = t[a, 0] * STEP_SIZE, t[a, 1] * STEP_SIZE
        assert t[a, 2] == (math.atan(abs(d2 / d1)) if d1 != 0 else math.pi / 2)
    assert t[0, 0] == 1.0 and t[0, 1] == 0.0
    assert abs(t[1, 0]) < 1e-15 and t[1, 0] != 0.0 and t[1, 1] == 1.0      # the 6e-17 residue is kept
    assert t[2, 0] == -1.0 and abs(t[2, 1]) < 1e-15 and t[2, 1] != 0.0
    # row n: every action >= n is clipped to +1 (robot.py:390-393) -> phi = 2 pi
    assert t.shape == (5, 3) and t[4, 0] == np.cos(2 * np.pi) and t[4, 1] == np.sin(2 * np.pi)


def test_algorithmic_bytes_matches_survey_8d():
    sys.path.insert(0, ROOT)
    import bench
    # SURVEY.md 8(d): C2 floor with U = 200, p_reset = 0
    assert bench.algorithmic_bytes(1, 9663, 6, 1, True, 200, 0.0) == 9663 + 400 + 48 + 8 + 40 + 320
    assert bench.algorithmic_bytes(2, 14482, 6, 1, True, 150, 0.0) == 28964 + 600 + 48 + 8 + 40 + 320
    assert bench.algorithmic_bytes(1, 9663, 2, 1, False, 0, 0.0) == 16 + 8 + 40 + 320


def test_bench_dump_outputs_writes_a_fixed_sample_within_the_limit(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every environment while the arrays fit the limit, a seeded sample (the same one in
    every run) once they do not; flags and float32 tensors in float32, the rest in float64."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    arrays = {'obs': torch.arange(600, dtype=torch.float64).reshape(100, 6), 'done': torch.ones(100, dtype=torch.uint8),
              'new_texels': torch.arange(100, dtype=torch.int32), 'value': torch.zeros(100, dtype=torch.float32)}
    bench.dump_outputs(str(tmp_path / 'all'), arrays)
    got = {k: np.load(str(tmp_path / 'all' / (k + '.npy'))) for k in list(arrays) + ['env_ids']}
    assert np.array_equal(got['env_ids'], np.arange(100)) and np.array_equal(got['obs'], arrays['obs'].numpy())
    assert got['obs'].dtype == np.float64 and got['new_texels'].dtype == np.float64
    assert got['done'].dtype == np.float32 and got['value'].dtype == np.float32
    monkeypatch.setattr(bench, 'DUMP_BYTES', 10 * (8 + 48 + 1 * 4 + 8 + 4))
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), arrays)
    ids = np.load(str(tmp_path / 'a' / 'env_ids.npy'))
    assert len(ids) == 10 and np.all(np.diff(ids) > 0)
    assert np.array_equal(ids, np.load(str(tmp_path / 'b' / 'env_ids.npy')))
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'obs.npy')), arrays['obs'].numpy()[ids.astype(np.int64)])
    total = sum(os.path.getsize(str(tmp_path / 'a' / (k + '.npy'))) - 128 for k in list(arrays) + ['env_ids'])
    assert total <= bench.DUMP_BYTES


def test_shard_range_partitions_every_env_exactly_once():
    from paintrl_b200.sharding import shard_range
    for total in (0, 1, 7, 4096, 65536, 65537):
        for world in (1, 2, 3, 4, 8):
            seen = []
            for r in range(world):
                lo, hi = shard_range(total, r, world)
                assert 0 <= lo <= hi <= total
                seen.extend(range(lo, hi))
            assert seen == list(range(total))
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


_GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, %r)
import torch, torch.distributed as dist
from paintrl_b200 import sharding
rank, local_rank, world = sharding.init_process_group(backend='gloo')
assert world == 2 and dist.get_backend() == 'gloo'
lo, hi = sharding.shard_range(65536, rank, world)
stats = {'env_steps': hi - lo, 'episodes': 10 * (rank + 1), 'sum_reward': 1.5 * (rank + 1),
         'max_episode_len': 100 + rank, 'max_step_ms': 2.0 - rank}
out = sharding.allreduce_stats(stats)
assert out['env_steps'] == 65536 and out['episodes'] == 30 and abs(out['sum_reward'] - 4.5) < 1e-12
assert out['max_episode_len'] == 101 and out['max_step_ms'] == 2.0
dist.barrier()
dist.destroy_process_group()
print('rank %%d ok' %% rank)
'''


def test_world_size_2_gloo_statistics_allreduce(tmp_path):
    """The only exchange of the multi-GPU path (rollout statistics) on the gloo backend."""
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    script = tmp_path / 'worker.py'
    script.write_text(_GLOO_WORKER % ROOT)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE='2', MASTER_ADDR='127.0.0.1',
                   MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES='')
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for rank, p in enumerate(procs):
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out
        assert 'rank %d ok' % rank in out


@pytest.mark.parametrize('name,part_no,mode', [('door_rgb', 0, 'RGB'), ('sheet_hsi', 1, 'HSI')])
def test_compose_texture_rebuilds_the_reference_texels(name, part_no, mode):
    """Part.texels of the verbatim reference after 25 steps (oracle/make_texture_golden.py) from its front-texel
    status plane alone."""
    from paintrl_b200.partpack import PartPack
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 't_texture.npz'))
    pack = PartPack.for_part(part_no)
    tex = pack.compose_texture(g[name + '/status'], mode)
    assert np.array_equal(tex, g[name + '/texels'])
    img = pack.texture_image(g[name + '/status'], mode)
    assert img.shape == (240, 240, 3) and img.dtype == np.uint8
    assert np.array_equal(img.reshape(-1), (g[name + '/texels'] & 0xff).astype(np.uint8))
    # computed offsets equal the stored ones
    stored = pack.arrays['texel_off']
    bare = PartPack(pack.meta, {k: v for k, v in pack.arrays.items() if k != 'texel_off'})
    assert np.array_equal(bare.texel_offsets(), stored)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line with the contract's keys,
    produced by the oracle port on the host cores; non-zero ranks print nothing."""
    import json
    env = dict(os.environ, PAINTRL_BENCH_REFERENCE_SECONDS='0.3')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['metric'] == 'batched env steps/sec' and line['unit'] == 'env-steps/s'
    assert line['value'] > 0 and line['higher_is_better'] is True and line['n_gpus'] == 1
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1 and line['cpu_baseline']['value'] == line['value']
    assert line['e2e'] == {'value': line['value'], 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert line['config']['workload'].startswith('C2 door panel')
    other = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300,
                           env=dict(env, RANK='1', LOCAL_RANK='1', WORLD_SIZE='2'))
    assert other.returncode == 0 and other.stdout.strip() == ''
