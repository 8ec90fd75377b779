"""GPU tests of the step's start-order switch (PAINTRL_START_ORDER, read at handle creation): it only moves the L2
sweep of the tables, the bit-plane copy and its wait, so both settings must give the same outputs and the same state,
bit for bit, on every kernel shape it touches."""
import os

import numpy as np
import pytest
import torch

from paintrl_b200.config import EnvConfig
from paintrl_b200.partpack import PartPack

pytestmark = pytest.mark.gpu

BASE = {'RENDER_HEIGHT': 720, 'RENDER_WIDTH': 960, 'Part_NO': 0, 'Expected_Episode_Length': 25,
        'EPISODE_MAX_LENGTH': 25, 'TERMINATION_MODE': 'late', 'SWITCH_THRESHOLD': 0.9,
        'START_POINT_MODE': 'anchor', 'TURNING_PENALTY': False, 'OVERLAP_PENALTY': False,
        'COLOR_MODE': 'RGB'}
C3_LATE = dict(BASE, Part_NO=1, COLOR_MODE='HSI', TURNING_PENALTY=True, OVERLAP_PENALTY=True)

# PAINTRL_START_ORDER; the first is the reference (the step's earlier order), None = the default
SETTINGS = ['0', '1', None]

CASES = {
    'c2_one_kernel': (dict(BASE), {}, 192, False),
    'c3_steady_two_kernel': (dict(C3_LATE), {'PAINTRL_FUSED': '0'}, 160, False),
    'c3_steady_one_kernel': (dict(C3_LATE), {'PAINTRL_FUSED': '1'}, 160, False),
    'subset_one_kernel': (dict(BASE), {}, 192, True),
    'bail_one_kernel': (dict(BASE, START_POINT_MODE='edge'), {'PAINTRL_DEBUG_BAIL_MOD': '3'}, 96, False),
    'bail_two_kernel': (dict(BASE, START_POINT_MODE='edge'), {'PAINTRL_DEBUG_BAIL_MOD': '3', 'PAINTRL_FUSED': '0',
                                                              'PAINTRL_MOVE_LANES': '8'}, 96, False),
}
OUTS = ('obs', 'actual', 'reward', 'penalty', 'done', 'new_texels', 'next_obs')


def _engine(cfg, n, env_vars, pack):
    from paintrl_b200.batched_env import BatchedPaintEnv
    saved = {k: os.environ.get(k) for k in env_vars}
    for k, v in env_vars.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
    try:
        return BatchedPaintEnv(n, cfg, device=torch.device('cuda:0'), pack=pack)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _outputs(obs, actual, done, info):
    return {'obs': obs, 'actual': actual, 'done': done, 'reward': info['reward'], 'penalty': info['penalty'],
            'new_texels': info['new_texels'], 'next_obs': info['next_obs']}


@pytest.mark.parametrize('case', sorted(CASES))
def test_switch_settings_are_bit_identical(case):
    """One engine per setting, same configuration, seed, starts and actions; 40 steps with auto-reset.  Every output
    of every step and the full state (status planes included) equal the reference setting's."""
    extra, env_vars, n, use_subsets = CASES[case]
    cfg = EnvConfig(extra, auto_reset=True, seed=7)
    pack = PartPack.for_part(cfg.part_no)
    engines = [_engine(cfg, n, dict(env_vars, PAINTRL_START_ORDER=so), pack) for so in SETTINGS]
    rng = np.random.default_rng(sum(map(ord, case)))
    start = rng.integers(0, engines[0].n_starts, size=n).astype(np.int32)
    for e in engines:
        e.reset(start)
    parts = [range(0, n // 3), rng.permutation(np.arange(n // 3, n)).tolist()] if use_subsets else None
    subsets = [[e.subset(p) for p in parts] for e in engines] if use_subsets else None
    episodes = 0
    for t in range(40):
        acts = rng.integers(0, cfg.discrete_granularity + 1, size=n)
        ref = None
        for i, e in enumerate(engines):
            if use_subsets:
                got = {}
                for p, s in zip(parts, subsets[i]):
                    ids = np.asarray(list(p))
                    out = _outputs(*e.step(acts[ids], subset=s))
                    for k, v in out.items():
                        if k not in got:
                            got[k] = torch.zeros((n,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)
                        got[k][torch.as_tensor(ids, device=v.device).long()] = v
            else:
                got = {k: v.clone() for k, v in _outputs(*e.step(acts)).items()}
            if ref is None:
                ref = got
                episodes += int(ref['done'].sum())
                continue
            for k in OUTS:
                assert torch.equal(ref[k], got[k]), (case, SETTINGS[i], t, k)
        if t % 8 == 7 or t == 39:
            s0 = engines[0].get_state()
            for i, e in enumerate(engines[1:], 1):
                si = e.get_state()
                for key in ('status', 'pose', 'quat', 'scalars'):
                    assert torch.equal(s0[key], si[key]), (case, SETTINGS[i], t, key)
    assert episodes > 0, 'no auto-reset exercised'
    for e in engines:
        e.close()
