"""GPU parity of the kernel variants the default configuration does not reach at small batches: the
two-kernel step with 8- and 32-lane move groups (8 lanes are chosen from 16384 environments per GPU on),
the hand-over of a bailed move to the paint warp, the paint kernel with the flip-bit plane in global
memory (textures whose plane exceeds the shared-memory stage), and state export / import.
Each case replays a seeded batch against the C oracle, bit-exact (RGB / discrete)."""
import os

import numpy as np
import pytest
import torch

from paintrl_b200.config import EnvConfig
from paintrl_b200.partpack import PartPack

pytestmark = pytest.mark.gpu

BASE = {'RENDER_HEIGHT': 720, 'RENDER_WIDTH': 960, 'Part_NO': 0, 'Expected_Episode_Length': 245,
        'EPISODE_MAX_LENGTH': 245, 'TERMINATION_MODE': 'late', 'SWITCH_THRESHOLD': 0.9,
        'START_POINT_MODE': 'anchor', 'TURNING_PENALTY': False, 'OVERLAP_PENALTY': False,
        'COLOR_MODE': 'RGB'}


def _replay(extra, kw, num_envs, steps, env_vars):
    from oracle.oracle import OracleBatch
    from paintrl_b200.batched_env import BatchedPaintEnv
    saved = {k: os.environ.get(k) for k in env_vars}
    os.environ.update(env_vars)
    try:
        cfg = EnvConfig(extra, auto_reset=True, **kw)
        pack = PartPack.for_part(cfg.part_no)
        env = BatchedPaintEnv(num_envs, cfg, device=torch.device('cuda:0'), pack=pack)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    ora = OracleBatch(pack, cfg, num_envs)
    rng = np.random.default_rng(7)
    start = rng.integers(0, env.n_starts, size=num_envs).astype(np.int32)
    assert np.array_equal(env.reset(start).cpu().numpy(), ora.reset(start))
    exact = cfg.color_mode == 'RGB' and cfg.action_mode == 'discrete'
    for t in range(steps):
        if cfg.action_mode == 'discrete':
            acts = rng.integers(0, cfg.discrete_granularity, size=num_envs)
        else:
            acts = rng.uniform(-1, 1, size=(num_envs, cfg.action_dim))
        nxt = rng.integers(0, env.n_starts, size=num_envs).astype(np.int32)
        obs, actual, done, info = env.step(acts, reset_start_index=nxt)
        o_obs, o_rew, o_pen, o_act, o_done = ora.step(acts)
        assert np.array_equal(done.cpu().numpy(), o_done), t
        if exact:
            assert np.array_equal(obs.cpu().numpy(), o_obs), t
            assert np.array_equal(actual.cpu().numpy(), o_act), t
        else:
            assert np.allclose(obs.cpu().numpy(), o_obs, rtol=1e-5, atol=1e-12), t
            assert np.allclose(actual.cpu().numpy(), o_act, rtol=1e-5, atol=1e-12), t
        if t % 9 == 0 or t == steps - 1:
            status = env.get_state()['status'].cpu().numpy()
            for e in range(num_envs):
                if not o_done[e]:
                    assert np.array_equal(status[e], ora.status(e)), (t, e)
        ids = np.flatnonzero(o_done)
        if len(ids):
            ora.reset(nxt[ids], env_ids=list(ids))
    env.close()
    ora.close()


@pytest.mark.parametrize('lanes', [8, 32])
def test_move_kernel_lane_groups(lanes):
    _replay(dict(BASE), {}, 96, 60, {'PAINTRL_MOVE_LANES': str(lanes), 'PAINTRL_FUSED': '0'})


@pytest.mark.parametrize('fused', ['0', '1'])
@pytest.mark.parametrize('kw', [dict(), dict(action_mode='continuous', action_shape=2, obs_mode='grid', obs_grad=4),
                                dict(action_mode='continuous', action_shape=1, obs_mode='section', obs_grad=8)])
def test_one_kernel_and_two_kernel_steps(fused, kw):
    """The step as one launch (a warp runs the move and the paint phase of its environment back to back; default
    below 16384 environments) and as two launches (move grid + paint grid with per-environment hand-off flags),
    forced either way on the same small batch."""
    _replay(dict(BASE, START_POINT_MODE='all', OVERLAP_PENALTY=True), kw, 80, 50, {'PAINTRL_FUSED': fused})


def test_one_kernel_step_unstaged_hsi():
    _replay(dict(BASE, Part_NO=1, COLOR_MODE='HSI', OVERLAP_PENALTY=True), {}, 64, 40, {'PAINTRL_FUSED': '1', 'PAINTRL_FORCE_UNSTAGED': '1'})


@pytest.mark.parametrize('lanes', ['8', '32', 'fused'])
@pytest.mark.parametrize('color', ['RGB', 'HSI'])
def test_fast_move_kernel_hands_over_to_the_paint_warp(lanes, color):
    """Every third environment is forced off the fast move kernel: its paint warp runs the generic move itself
    (the path rays take that their move cell cannot decide).  Results stay bit-exact."""
    extra = dict(BASE, COLOR_MODE=color, START_POINT_MODE='edge', OVERLAP_PENALTY=True)
    env_vars = {'PAINTRL_DEBUG_BAIL_MOD': '3', 'PAINTRL_FUSED': '1'} if lanes == 'fused' else {
        'PAINTRL_DEBUG_BAIL_MOD': '3', 'PAINTRL_MOVE_LANES': lanes, 'PAINTRL_FUSED': '0'}
    _replay(extra, {}, 100, 50, env_vars)


@pytest.mark.parametrize('color', ['RGB', 'HSI'])
def test_paint_kernel_unstaged_plane(color):
    extra = dict(BASE, Part_NO=1, COLOR_MODE=color, OVERLAP_PENALTY=True)
    _replay(extra, {}, 64, 50, {'PAINTRL_FORCE_UNSTAGED': '1'})


def test_unstaged_grid_and_discrete_observations():
    _replay(dict(BASE, START_POINT_MODE='edge'), dict(obs_mode='discrete', obs_grad=4, discrete_granularity=8), 48, 40,
            {'PAINTRL_FORCE_UNSTAGED': '1', 'PAINTRL_MOVE_LANES': '8'})


def test_state_round_trip():
    """Exact mid-episode checkpoint (ABI v2): get_state -> set_state into ANOTHER engine reproduces the future
    bit for bit, OVERLAP_PENALTY included -- the scalars carry the overlap reference
    (Part._last_painted_pixels, bullet_paint_wrapper.py:483, 575-576, as the last shot's centre), so the source
    engine does not have to re-import its own state."""
    from paintrl_b200.batched_env import BatchedPaintEnv
    for color in ('RGB', 'HSI'):
        cfg = EnvConfig(dict(BASE, OVERLAP_PENALTY=True, TURNING_PENALTY=True, COLOR_MODE=color, START_POINT_MODE='edge'), auto_reset=False)
        dev = torch.device('cuda:0')
        a = BatchedPaintEnv(32, cfg, device=dev)
        b = BatchedPaintEnv(40, cfg, device=dev)
        rng = np.random.default_rng(11)
        a.reset(rng.integers(0, a.n_starts, size=32).astype(np.int32))
        b.reset(np.zeros(40, dtype=np.int32))
        for _ in range(15):
            a.step(rng.integers(0, 4, size=32))
        st = a.get_state()
        assert st['scalars'].shape == (32, 12) and bool(st['has_overlap_reference'].all())
        ids = np.arange(32, dtype=np.int32) + 8           # into other slots of another engine
        b.set_state(env_ids=ids, status=st['status'], pose=st['pose'], quat=st['quat'], scalars=st['scalars'])
        st_b = b.get_state(env_ids=ids)
        assert torch.equal(st['status'], st_b['status'])
        assert torch.equal(st['pose'], st_b['pose']) and torch.equal(st['scalars'], st_b['scalars'])
        assert torch.equal(a.job_status(), b.job_status()[8:])
        saw_overlap = False
        for _ in range(10):
            acts = rng.integers(0, 4, size=32)
            oa, ra, da, ia = a.step(acts)
            ob, rb, db, ib = b.step(np.concatenate([np.zeros(8, dtype=np.int64), acts]))
            assert torch.equal(oa, ob[8:]) and torch.equal(ra, rb[8:]) and torch.equal(da, db[8:])
            assert torch.equal(ia['penalty'], ib['penalty'][8:])
            saw_overlap = saw_overlap or bool((ia['penalty'] > 0.2).any())
        assert saw_overlap
        assert torch.equal(a.get_state()['status'], b.get_state(env_ids=ids)['status'])
        # a status plane WITHOUT scalars clears the overlap reference (reset_part, bullet_paint_wrapper.py:708)
        b.set_state(env_ids=ids, status=st['status'])
        assert not bool(b.get_state(env_ids=ids)['has_overlap_reference'].any())
        a.close()
        b.close()


def test_env_ids_are_validated():
    """Out-of-range, duplicate and empty id lists are refused on the host (the kernels index state with them);
    a short reset_start_index is refused too."""
    from paintrl_b200.batched_env import BatchedPaintEnv
    env = BatchedPaintEnv(16, dict(BASE), device=torch.device('cuda:0'), auto_reset=True)
    env.reset(0)
    for bad, exc in (([16], IndexError), ([-1], IndexError), ([3, 3], ValueError), ([], ValueError),
                     (torch.tensor([2, 99], device='cuda:0'), IndexError), (torch.tensor([5, 5], device='cuda:0'), ValueError)):
        with pytest.raises(exc):
            env.reset(0, env_ids=bad)
        with pytest.raises(exc):
            env.get_state(env_ids=bad)
    with pytest.raises(ValueError):
        env.step(np.zeros(16, dtype=np.int64), reset_start_index=np.zeros(8, dtype=np.int32))
    assert env.reset(1, env_ids=torch.tensor([15, 0], device='cuda:0')).shape == (2, env.obs_dim)
    env.close()


def test_step_rejects_bad_buffers():
    """paintrl_step refuses null and misaligned I/O buffers with PAINTRL_E_INVALID instead of launching."""
    import ctypes
    import torch
    from paintrl_b200 import _capi
    from paintrl_b200.batched_env import BatchedPaintEnv
    env = BatchedPaintEnv(8, dict(BASE), device=torch.device('cuda:0'))
    env.reset(0)
    lib = _capi.lib()
    acts = torch.zeros(8, dtype=torch.int64, device='cuda:0')
    raw = torch.zeros(8 * 6 * 8 + 16, dtype=torch.uint8, device='cuda:0')
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    good = [p(acts), p(env.obs), p(env.reward), p(env.penalty), p(env.actual), p(env.done), None, None, None, None]
    assert lib.paintrl_step(env._h, *good) == 0
    bad = list(good)
    bad[1] = ctypes.c_void_p(raw.data_ptr() + 4)              # observation buffer off by 4 bytes
    assert lib.paintrl_step(env._h, *bad) == -1               # PAINTRL_E_INVALID
    assert b'misaligned' in lib.paintrl_last_error()
    bad = list(good)
    bad[2] = None
    assert lib.paintrl_step(env._h, *bad) < 0 and b'null' in lib.paintrl_last_error()
    torch.cuda.synchronize()
    env.close()
