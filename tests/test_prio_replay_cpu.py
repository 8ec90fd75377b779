"""CPU checks of prioritized replay and n-step returns (paintrl_b200.dqn) that need no device:

- n-step insertion of `ReplayBuffer.add` on CPU tensors against a plain per-transition loop (tests/prio_replica.py):
  episodes shorter than n, an episode end at every offset of the window, carries across two and three fragments, a
  fragment larger than the ring, wrap-around;
- n_step = 1 writes the ring bytes the uniform 1-step insertion always wrote;
- the learner handle's discount is fl32(gamma^n);
- the new DQNConfig fields: validation, and a config dict from before them loading with their defaults;
- the NumPy tree, descent and weight replicas that the GPU tests compare the kernels with, on hand-made cases."""
import types

import numpy as np
import pytest
import torch

import prio_replica as pr
from paintrl_b200 import dqn


def _frag(T, B, D, g, p_done=0.3):
    return types.SimpleNamespace(
        T=T, B=B,
        obs=torch.rand(T + 1, B, D, generator=g, dtype=torch.float64),
        term_obs=torch.rand(T, B, D, generator=g, dtype=torch.float64),
        actions=torch.randint(0, 4, (T, B), generator=g),
        actual=torch.randn(T, B, generator=g, dtype=torch.float64) * 3.0,
        done=(torch.rand(T, B, generator=g) < p_done).to(torch.uint8))


def _ring(buf):
    return (buf.obs.numpy(), buf.next_obs.numpy(), buf.actions.numpy(), buf.reward.numpy(), buf.done.numpy())


def _assert_ring_equal(got, ref):
    for name, a, b in zip(('obs', 'next_obs', 'actions', 'reward', 'done'), got, ref):
        assert a.dtype == b.dtype and a.tobytes() == b.tobytes(), name


@pytest.mark.parametrize('n,T_list,B,capacity', [
    (3, [10, 10, 10], 5, 4096),        # carries across fragments, no wrap
    (3, [1, 1, 1, 1, 6], 4, 4096),     # fragments shorter than the carry: one window spans three fragments
    (5, [2, 3, 7], 3, 4096),           # n larger than whole fragments
    (2, [9, 9, 9, 9], 7, 50),          # wrap-around, several times
    (4, [30, 5], 6, 64),               # a fragment larger than the ring (only its last rows stay)
    (3, [4], 2, 4096),                 # a single fragment: only T - n + 1 steps complete
])
def test_nstep_insertion_matches_a_plain_loop(n, T_list, B, capacity):
    g = torch.Generator().manual_seed(n * 100 + B)
    D, gamma = 3, 0.97
    buf = dqn.ReplayBuffer(capacity, D, 'cpu', n_step=n, gamma=gamma)
    frags = [_frag(T, B, D, g, p_done=0.35) for T in T_list]
    for f in frags:
        start, count = buf.add(f)
        assert 0 <= start < capacity and 0 <= count <= capacity
    ring, q, cut_at = pr.nstep_ring(frags, n, gamma, capacity)
    assert buf.size == min(capacity, q) and buf.pos == q % capacity
    _assert_ring_equal(_ring(buf), ring)
    if sum(T_list) * B >= 100:
        assert (cut_at > 0).all(), cut_at          # an episode ends at every offset of the window somewhere


def test_nstep_done_at_every_offset_and_short_episodes():
    """One environment per offset: done only at step j of the first window (episodes of length j + 1 <= n), then a
    run without dones, so the windows that reach the end of the data bootstrap with gamma^n."""
    n, D, T = 4, 2, 12
    g = torch.Generator().manual_seed(7)
    f = _frag(T, n, D, g, p_done=0.0)
    for j in range(n):
        f.done[j, j] = 1
    f.done[1, 0] = 1                               # env 0: two episodes of length 1 and 1 (shorter than n)
    buf = dqn.ReplayBuffer(256, D, 'cpu', n_step=n, gamma=0.9)
    buf.add(f)
    ring, q, cut_at = pr.nstep_ring([f], n, 0.9, 256)
    _assert_ring_equal(_ring(buf), ring)
    assert (cut_at > 0).all()
    # transition (t = 0, env j) ends at step j: s' = term_obs[j], done = 1, return sum_{k <= j} 0.9^k r[k]
    for j in range(n):
        R = 0.0
        for k in range(j + 1):
            R += 0.9 ** k * float(f.actual[k, j])
        assert buf.done[j] == 1 and torch.equal(buf.next_obs[j], f.term_obs[j, j]) and buf.reward[j] == np.float32(R)


def _legacy_add(buf, frag):
    """ReplayBuffer.add as it was before n-step returns (uniform 1-step insertion)."""
    T, B = frag.T, frag.B
    N = T * B
    src = (frag.obs[:T].reshape(N, -1), frag.term_obs.reshape(N, -1), frag.actions.reshape(N), frag.actual.reshape(N),
           frag.done.reshape(N))
    dst = (buf.obs, buf.next_obs, buf.actions, buf.reward, buf.done)
    skip = max(0, N - buf.capacity)
    start = (buf.pos + skip) % buf.capacity
    n = N - skip
    first = min(n, buf.capacity - start)
    for s, d in zip(src, dst):
        d[start:start + first].copy_(s[skip:skip + first])
        if n > first:
            d[:n - first].copy_(s[skip + first:])
    buf.pos = (buf.pos + N) % buf.capacity
    buf.size = min(buf.capacity, buf.size + N)


def test_one_step_insertion_is_byte_identical_to_the_uniform_buffer():
    g = torch.Generator().manual_seed(3)
    new = dqn.ReplayBuffer(100, 4, 'cpu', n_step=1, gamma=0.5)
    old = dqn.ReplayBuffer(100, 4, 'cpu')
    for T in (3, 20, 1, 40):                       # the 40 x 7 fragment is larger than the ring
        f = _frag(T, 7, 4, g)
        new.add(f)
        _legacy_add(old, f)
        _assert_ring_equal(_ring(new), _ring(old))
        assert (new.pos, new.size) == (old.pos, old.size)


def test_nstep_rejects_a_change_of_batch():
    g = torch.Generator().manual_seed(0)
    buf = dqn.ReplayBuffer(64, 2, 'cpu', n_step=3, gamma=0.9)
    buf.add(_frag(5, 4, 2, g))
    with pytest.raises(ValueError, match='environments'):
        buf.add(_frag(5, 3, 2, g))


@pytest.mark.parametrize('n', [1, 2, 3, 5])
def test_handle_discount_is_gamma_to_the_n_in_float32(n):
    cfg = dqn.DQNConfig(n_step=n, gamma=0.99, minibatch_size=128)
    c = dqn.DQNLearner._c_config(types.SimpleNamespace(obs_dim=6, n_out=4, cfg=cfg))
    assert c.gamma == float(np.float32(0.99 ** n))
    if n == 1:
        assert c.gamma == float(np.float32(0.99))


def test_config_fields_validation_and_old_dicts():
    c = dqn.DQNConfig()
    assert (c.prioritized_replay, c.prioritized_replay_alpha, c.prioritized_replay_beta, c.prioritized_replay_eps, c.n_step) == \
        (False, 0.6, 0.4, 1e-6, 1)
    for bad in (dict(n_step=0), dict(prioritized_replay_alpha=-0.1), dict(prioritized_replay_alpha=float('inf')),
                dict(prioritized_replay_beta=1.5), dict(prioritized_replay_beta=-0.01), dict(prioritized_replay_eps=0.0),
                dict(prioritized_replay_alpha=float('nan'))):
        with pytest.raises(ValueError):
            dqn.DQNConfig(**bad)
    ok = dqn.DQNConfig(prioritized_replay=True, n_step=3, prioritized_replay_alpha=0.0, prioritized_replay_beta=1.0)
    assert ok.prioritized_replay is True and ok.n_step == 3
    old = {k: v for k, v in dqn.DQNConfig(lr=1e-3).to_dict().items()
           if not k.startswith('prioritized_replay') and k != 'n_step'}
    loaded = dqn.DQNConfig.from_dict(old)
    assert loaded.lr == 1e-3 and loaded.to_dict() == dqn.DQNConfig(lr=1e-3).to_dict()
    assert dqn.DQNConfig.from_dict(ok.to_dict()).to_dict() == ok.to_dict()


def test_tree_leaves():
    assert [dqn.tree_leaves(c) for c in (1, 2, 3, 5, 1024, 1025, 1 << 21)] == [1, 2, 4, 8, 1024, 2048, 1 << 21]


def test_replica_tree_is_the_pairwise_rebuild():
    leaves = np.array([0.5, 0.0, 2.0, 0.25, 1.0])
    s, m = pr.tree_from_leaves(leaves, 8)
    assert s[1] == 3.75 and m[1] == 0.25
    assert s[2] == 0.5 + 0.0 + 2.0 + 0.25 and s[3] == 1.0 and m[3] == 1.0 and np.isinf(m[7])
    for i in range(1, 8):
        assert s[i] == s[2 * i] + s[2 * i + 1] and m[i] == min(m[2 * i], m[2 * i + 1])


def test_replica_descent_hand_cases():
    top = 1.0 - 2.0 ** -53                         # the largest double below 1: u * root may round up to the root
    # all mass in the first leaf
    s, _ = pr.tree_from_leaves([1.0, 0, 0, 0, 0, 0, 0, 0], 8)
    assert (pr.descend(s, 8, [0.0, 0.5, top]) == 0).all()
    # all mass in the last leaf: the descent must go right past empty left subtrees
    s, _ = pr.tree_from_leaves([0, 0, 0, 0, 0, 0, 0, 3.0], 8)
    assert (pr.descend(s, 8, [0.0, 0.5, top]) == 7).all()
    # zero leaves between filled ones, non-power-of-two capacity 5 (L = 8, rows 5..7 unfilled)
    s, m = pr.tree_from_leaves([3.0, 0.0, 0.0, 2.0, 0.0], 8)
    assert list(pr.descend(s, 8, [0.0, 0.59, 0.6, 0.99, top])) == [0, 0, 3, 3, 3]
    # u * root rounding to the root is clamped below it; the leaf is the last positive one, never an unfilled row
    s, _ = pr.tree_from_leaves([0.1, 0.2, 0.7], 4)
    assert pr.descend(s, 4, [top])[0] == 2
    # rounding in the subtraction: a mass past the left sum never lands on a zero leaf
    leaves = np.array([0.1] * 7 + [0.0])
    s, _ = pr.tree_from_leaves(leaves, 8)
    idx = pr.descend(s, 8, np.linspace(0.0, top, 10001))
    assert (leaves[idx] > 0).all() and idx.max() == 6
    assert (np.diff(idx) >= 0).all()               # the descent is monotone in u


def test_replica_weights():
    s, m = pr.tree_from_leaves([4.0, 1.0, 0.0, 2.0], 4)
    w = pr.weights(s, m, 4, np.array([0, 1, 3]), 0.4)
    assert w[1] == 1.0 and np.allclose(w, [4.0 ** -0.4, 1.0, 2.0 ** -0.4], rtol=0, atol=1e-15) and (w <= 1.0).all()
    assert (pr.weights(s, m, 4, np.array([0, 1, 3]), 0.0) == 1.0).all()
