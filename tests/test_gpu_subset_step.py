"""GPU tests of stepping a subset of a handle's environments (paintrl_step_subset / paintrl_step_host_submit_range):
a subset step does to its environments exactly what the whole-batch step does and leaves the others alone, bit for
bit, across every kernel variant; it is pinned to the C oracle directly; the two-slot host pipeline runs a
closed-loop policy on two groups; a fixed subset step replays from a CUDA graph."""
import ctypes
import os

import numpy as np
import pytest
import torch

from paintrl_b200.config import EnvConfig
from paintrl_b200.partpack import PartPack

pytestmark = pytest.mark.gpu

BASE = {'RENDER_HEIGHT': 720, 'RENDER_WIDTH': 960, 'Part_NO': 0, 'Expected_Episode_Length': 25,
        'EPISODE_MAX_LENGTH': 25, 'TERMINATION_MODE': 'late', 'SWITCH_THRESHOLD': 0.9,
        'START_POINT_MODE': 'anchor', 'TURNING_PENALTY': True, 'OVERLAP_PENALTY': True,
        'COLOR_MODE': 'RGB'}
OUTS = ('obs', 'actual', 'reward', 'penalty', 'done', 'new_texels', 'next_obs')


def _make(cfg, num_envs, env_vars, pack=None, copies=2):
    """`copies` engines of the same configuration and seed, created under `env_vars` (read at creation)."""
    from paintrl_b200.batched_env import BatchedPaintEnv
    saved = {k: os.environ.get(k) for k in env_vars}
    os.environ.update(env_vars)
    try:
        pack = pack if pack is not None else PartPack.for_part(cfg.part_no)
        return [BatchedPaintEnv(num_envs, cfg, device=torch.device('cuda:0'), pack=pack) for _ in range(copies)]
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _partition(rng, n):
    """2-5 subsets covering 0..n-1: some contiguous ranges, the rest id lists with ids from anywhere, shuffled."""
    k = int(rng.integers(2, 6))
    cuts = np.sort(rng.choice(np.arange(1, n), k - 1, replace=False))
    chunks = np.split(np.arange(n), cuts)
    as_range = rng.random(k) < 0.5
    as_range[0], as_range[-1] = True, False        # at least one of each kind
    parts = [range(int(c[0]), int(c[-1]) + 1) for c, r in zip(chunks, as_range) if r]
    pool = rng.permutation(np.concatenate([c for c, r in zip(chunks, as_range) if not r]))
    n_lists = int(rng.integers(1, min(3, len(pool)) + 1))
    for j, ids in enumerate(np.array_split(pool, n_lists)):
        parts.append(torch.as_tensor(ids, device='cuda:0') if j % 2 else ids.tolist())
    return parts


def _actions(rng, cfg, n):
    if cfg.action_mode == 'discrete':
        return rng.integers(0, cfg.discrete_granularity + 1, size=n)
    return rng.uniform(-1.2, 1.2, size=(n, cfg.action_dim))


def _full_outputs(obs, actual, done, info):
    return {'obs': obs, 'actual': actual, 'done': done, 'reward': info['reward'], 'penalty': info['penalty'],
            'new_texels': info['new_texels'], 'next_obs': info['next_obs']}


def _assert_same_state(a, b, ctx):
    sa, sb = a.get_state(), b.get_state()
    for key in ('status', 'pose', 'quat', 'scalars'):
        assert torch.equal(sa[key], sb[key]), (ctx, key)


CASES = {
    'one_kernel': (dict(BASE), {}, {}, 96),
    'two_kernel_8_lanes': (dict(BASE), {}, {'PAINTRL_FUSED': '0', 'PAINTRL_MOVE_LANES': '8'}, 96),
    'two_kernel_32_lanes': (dict(BASE), {}, {'PAINTRL_FUSED': '0', 'PAINTRL_MOVE_LANES': '32'}, 96),
    'hsi_sheet_unstaged': (dict(BASE, Part_NO=1, COLOR_MODE='HSI'), {}, {'PAINTRL_FORCE_UNSTAGED': '1'}, 64),
    'continuous2_grid4': (dict(BASE, START_POINT_MODE='all'),
                          dict(action_mode='continuous', action_shape=2, obs_mode='grid', obs_grad=4), {}, 80),
    'generic_axes': (dict(BASE, START_POINT_MODE='all'), {}, {}, 80),
    'normal_paint': (dict(BASE, START_POINT_MODE='edge'), dict(paint_method='normal'), {}, 24),
    'cold_move_bail_one_kernel': (dict(BASE, START_POINT_MODE='edge'), {}, {'PAINTRL_DEBUG_BAIL_MOD': '3'}, 96),
    'cold_move_bail_two_kernel': (dict(BASE, START_POINT_MODE='edge'), {},
                                  {'PAINTRL_DEBUG_BAIL_MOD': '3', 'PAINTRL_FUSED': '0', 'PAINTRL_MOVE_LANES': '8'}, 96),
}


@pytest.mark.parametrize('case', sorted(CASES))
def test_partition_equals_whole_batch(case):
    """Engine A steps the whole batch; engine B (same configuration and seed) steps the same actions through a
    partition into ranges and id lists, in a new order every step.  Auto-reset alternates between the seeded
    stream and explicit start indices.  Every output row (gathered by id) and the full state are bit-identical."""
    extra, kw, env_vars, n = CASES[case]
    cfg = EnvConfig(extra, auto_reset=True, seed=5, **kw)
    pack = None
    if case == 'generic_axes':
        from pack_util import permuted_pack
        pack = permuted_pack(PartPack.for_part(0), 'axes02')
    a, b = _make(cfg, n, env_vars, pack=pack)
    rng = np.random.default_rng(sum(map(ord, case)))
    start = rng.integers(0, a.n_starts, size=n).astype(np.int32)
    assert torch.equal(a.reset(start), b.reset(start))
    subsets = [b.subset(p) for p in _partition(rng, n)]
    host_ids = [s.env_ids.cpu().numpy() for s in subsets]
    assert np.array_equal(np.sort(np.concatenate(host_ids)), np.arange(n))
    episodes = 0
    for t in range(64):
        acts = _actions(rng, cfg, n)
        nxt = rng.integers(0, a.n_starts, size=n).astype(np.int32) if t % 2 else None
        full = {k: v.clone() for k, v in _full_outputs(*a.step(acts, reset_start_index=nxt)).items()}
        got = {k: torch.zeros_like(v) for k, v in full.items()}
        for j in rng.permutation(len(subsets)):
            s, ids = subsets[j], host_ids[j]
            obs, actual, done, info = b.step(acts[ids], reset_start_index=None if nxt is None else nxt[ids], subset=s)
            assert torch.equal(info['env_ids'], s.env_ids)
            for k, v in _full_outputs(obs, actual, done, info).items():
                got[k][torch.as_tensor(ids, device=v.device).long()] = v
        for k in OUTS:
            assert torch.equal(full[k], got[k]), (case, t, k)
        episodes += int(full['done'].sum())
        if t % 10 == 9:
            _assert_same_state(a, b, (case, t))
    assert episodes > 0, 'no auto-reset exercised'
    assert a.stats()['env_steps'] == b.stats()['env_steps'] == 64 * n
    a.close()
    b.close()


def test_other_environments_are_untouched():
    """A subset step changes nothing of the environments outside it; env_steps grows by n."""
    cfg = EnvConfig(dict(BASE), auto_reset=True, seed=2)
    env, = _make(cfg, 64, {}, copies=1)
    rng = np.random.default_rng(3)
    env.reset(rng.integers(0, env.n_starts, size=64).astype(np.int32))
    for _ in range(5):
        env.step(rng.integers(0, 4, size=64))
    for spec in (np.array([3, 60, 17, 40, 8, 33]), range(20, 29)):
        sub = env.subset(spec)
        members = sub.env_ids.cpu().numpy()
        others = np.setdiff1d(np.arange(64), members)
        before = env.get_state(env_ids=others)
        steps0 = env.stats()['env_steps']
        env.step(rng.integers(0, 4, size=len(members)), subset=sub)
        after = env.get_state(env_ids=others)
        for key in ('status', 'pose', 'quat', 'scalars'):
            assert torch.equal(before[key], after[key]), key
        assert env.stats()['env_steps'] == steps0 + len(members)
    env.close()


def test_kernel_shape_follows_the_subset_size():
    """16384 environments stepped as four 4096-ranges (one-kernel step each) equal the same batch stepped whole
    (two-kernel step), bit for bit (RGB, discrete)."""
    n = 16384
    cfg = EnvConfig(dict(BASE), auto_reset=True, seed=9)
    a, b = _make(cfg, n, {})
    rng = np.random.default_rng(4)
    start = rng.integers(0, a.n_starts, size=n).astype(np.int32)
    a.reset(start)
    b.reset(start)
    subs = [b.subset(range(q * 4096, (q + 1) * 4096)) for q in range(4)]
    steps0 = a.stats()['kernel_launches'], b.stats()['kernel_launches']
    for t in range(30):
        acts = rng.integers(0, 4, size=n)
        full = {k: v.clone() for k, v in _full_outputs(*a.step(acts)).items()}
        for q, s in enumerate(subs):
            part = _full_outputs(*b.step(acts[q * 4096:(q + 1) * 4096], subset=s))
            for k in OUTS:
                assert torch.equal(full[k][q * 4096:(q + 1) * 4096], part[k]), (t, q, k)
    launches = a.stats()['kernel_launches'] - steps0[0], b.stats()['kernel_launches'] - steps0[1]
    assert launches == (2 * 30, 4 * 30)          # two kernels per whole step, one per 4096-subset step
    _assert_same_state(a, b, 'end')
    a.close()
    b.close()


def _oracle_step_subset(ora, ids, acts):
    """OracleBatch.step for the environments `ids` only (the oracle steps any list of its environments)."""
    from oracle.oracle import action_directions
    dirs = np.ascontiguousarray(action_directions(ora.cfg, acts))
    n = len(ids)
    arr = (ctypes.c_void_p * n)(*[ora.envs[i] for i in ids])
    obs = np.zeros((n, ora.obs_dim))
    reward, penalty, actual = np.zeros(n), np.zeros(n), np.zeros(n)
    done = np.zeros(n, dtype=np.uint8)
    ora._h.oracle_step_batch(arr, n, dirs.ctypes.data, obs.ctypes.data, reward.ctypes.data, penalty.ctypes.data,
                             actual.ctypes.data, done.ctypes.data, ora.threads)
    return obs, reward, penalty, actual, done


def test_shuffled_subsets_match_the_oracle():
    """One shuffled-subset schedule replayed against the C oracle stepping the same subsets (RGB, discrete:
    bit-exact), explicit auto-reset start indices."""
    from oracle.oracle import OracleBatch
    n = 72
    cfg = EnvConfig(dict(BASE, START_POINT_MODE='edge'), auto_reset=True)
    env, = _make(cfg, n, {}, copies=1)
    ora = OracleBatch(env.pack, cfg, n)
    rng = np.random.default_rng(21)
    start = rng.integers(0, env.n_starts, size=n).astype(np.int32)
    assert np.array_equal(env.reset(start).cpu().numpy(), ora.reset(start))
    for t in range(40):
        parts = _partition(rng, n)
        for p in rng.permutation(len(parts)):
            sub = env.subset(parts[p])
            ids = sub.env_ids.cpu().numpy()
            acts = rng.integers(0, 4, size=len(ids))
            nxt = rng.integers(0, env.n_starts, size=len(ids)).astype(np.int32)
            obs, actual, done, info = env.step(acts, reset_start_index=nxt, subset=sub)
            o_obs, o_rew, o_pen, o_act, o_done = _oracle_step_subset(ora, ids.tolist(), acts)
            assert np.array_equal(obs.cpu().numpy(), o_obs), (t, p)
            assert np.array_equal(actual.cpu().numpy(), o_act), (t, p)
            assert np.array_equal(info['reward'].cpu().numpy(), o_rew), (t, p)
            assert np.array_equal(info['penalty'].cpu().numpy(), o_pen), (t, p)
            assert np.array_equal(done.cpu().numpy(), o_done), (t, p)
            ended = np.flatnonzero(o_done)
            if len(ended):
                ora.reset(nxt[ended], env_ids=[int(ids[k]) for k in ended])
    status = env.get_state()['status'].cpu().numpy()
    assert np.array_equal(status, ora.status())
    env.close()
    ora.close()


def _greedy(obs):
    """The closed-loop policy of profiles/closed_loop.py: the discrete action = argmax of the four section values."""
    return np.argmax(obs[:, :4], axis=1).astype(np.int64)


def test_host_ping_pong_equals_synchronous_loop():
    """A closed-loop greedy policy driven through two range groups on slots 0 / 1 (wait for one group, act on its
    observation, resubmit it, go on with the other) equals the synchronous whole-batch step_host loop."""
    n, half, T = 256, 128, 50
    cfg = EnvConfig(dict(BASE), auto_reset=True, seed=13)
    a, b = _make(cfg, n, {})
    start = np.random.default_rng(8).integers(0, a.n_starts, size=n).astype(np.int32)
    obs = a.reset(start).cpu().numpy()
    b_obs = b.reset(start).cpu().numpy()
    assert np.array_equal(obs, b_obs)
    ref = []
    out = a.host_buffers()
    for _ in range(T):
        out = a.step_host(_greedy(obs), out)
        ref.append((out['obs'].copy(), out['reward'].copy(), out['done'].copy()))
        obs = out['next_obs'].copy()
    groups = [b.subset(range(0, half)), b.subset(range(half, n))]
    bufs = [b.host_buffers(n=half), b.host_buffers(n=half)]
    acts = [torch.zeros(half, dtype=torch.int64).pin_memory().numpy() for _ in range(2)]
    for g in range(2):
        acts[g][:] = _greedy(b_obs[g * half:(g + 1) * half])
        b.step_host_submit(acts[g], bufs[g], slot=g, subset=groups[g])
    for t in range(T):
        for g in range(2):
            res = b.step_host_wait(g)
            rows = slice(g * half, (g + 1) * half)
            assert np.array_equal(res['obs'], ref[t][0][rows]), (g, t)
            assert np.array_equal(res['reward'], ref[t][1][rows]), (g, t)
            assert np.array_equal(res['done'], ref[t][2][rows]), (g, t)
            if t + 1 < T:
                acts[g][:] = _greedy(res['next_obs'])
                b.step_host_submit(acts[g], bufs[g], slot=g, subset=groups[g])
    assert sum(int(r[2].sum()) for r in ref) > 0, 'no auto-reset exercised'
    with pytest.raises(ValueError):
        b.step_host_submit(acts[0], bufs[0], slot=0, subset=b.subset([0, 1]))      # id lists: device steps only
    a.close()
    b.close()


def test_subset_steps_replay_from_a_cuda_graph():
    """Two subset steps (a range and an id list) captured once and replayed 10 times equal an eager twin."""
    n = 64
    cfg = EnvConfig(dict(BASE), auto_reset=True, seed=17)
    g_env, e_env = _make(cfg, n, {})
    rng = np.random.default_rng(12)
    start = rng.integers(0, g_env.n_starts, size=n).astype(np.int32)
    g_env.reset(start)
    e_env.reset(start)
    ids = rng.permutation(np.arange(20, n))[:30]
    specs = (range(0, 20), ids)
    g_subs = [g_env.subset(s) for s in specs]
    e_subs = [e_env.subset(s) for s in specs]
    acts = [torch.zeros(len(s), dtype=torch.int64, device='cuda:0') for s in g_subs]
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for s, act in zip(g_subs, acts):
            g_env.step(act, subset=s)
    torch.cuda.synchronize()
    for t in range(10):
        host = [rng.integers(0, 4, size=len(s)) for s in g_subs]
        for act, h in zip(acts, host):
            act.copy_(torch.as_tensor(h))
        graph.replay()
        for s_g, s_e, h in zip(g_subs, e_subs, host):
            e_env.step(h, subset=s_e)
            for k in ('obs', 'actual', 'done', 'next_obs', 'reward', 'penalty', 'new_texels'):
                assert torch.equal(getattr(s_g, k), getattr(s_e, k)), (t, k)
    _assert_same_state(g_env, e_env, 'end')
    del graph
    g_env.close()
    e_env.close()
