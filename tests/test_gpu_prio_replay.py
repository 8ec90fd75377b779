"""GPU: prioritized replay and n-step returns (csrc/paintrl_replay.cuh, the kLossDqnPer stage of csrc/paintrl_learn.cuh,
paintrl_b200.dqn).

- the trees: leaves (|td| + eps)^alpha within CUDA's double pow bound, every internal node equal to a NumPy rebuild from
  the kernel's own leaves bit for bit, max_priority exact, duplicate rows, prio_fill across the ring's wrap;
- sampling: rows equal to the NumPy descent (tests/prio_replica.py) on the kernel's tree with the same uniforms, edge
  uniforms included; never a zero-priority row or one at or beyond size; a chi-square test of 10^6 draws; the weights
  against the FP64 formula; weight exactly 1 on the minimum-priority row and for alpha = 0 or beta = 0;
- the weighted loss at one shape per <MO, MX> instantiation: all-ones weights give paintrl_dqn_grad's gradient and
  statistics bit for bit, w = 2^k scales a one-sample gradient by exactly 2^k, td_out is Q(s, a) - y of the one-sample
  statistics, duplicate rows get identical td, and mixed weights match torch autograd;
- end to end: reproducible prioritized 3-step learners, the weighted loss falling on a fixed buffer, the train script.

CUDA's double-precision pow has a maximum error of 2 ulp over its full range (CUDA C++ Programming Guide, "Mathematical
Functions", double-precision table), so leaves and weights are compared with that bound; everything built from them by
additions, fmin and comparisons is compared exactly."""
import ctypes
import json

import numpy as np
import pytest
import torch

import prio_replica as pr
from test_gpu_dqn import GRAD_COS, GRAD_RTOL, _errors, _Forward, _policy, _q_greedy, _split, _transitions

pytestmark = pytest.mark.gpu

POW_ULP = 2                                      # CUDA double pow, full range (Programming Guide)
P = lambda t: ctypes.c_void_p(t.data_ptr())


def _lib():
    from paintrl_b200 import _capi
    return _capi


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _trees(L, device):
    return (torch.zeros(2 * L, dtype=torch.float64, device=device),
            torch.full((2 * L,), float('inf'), dtype=torch.float64, device=device))


def _fill(sum_t, min_t, L, capacity, start, count, maxp, alpha):
    c = _lib()
    c.check(c.lib().paintrl_prio_fill(P(sum_t), P(min_t), L, capacity, start, count, P(maxp), alpha, _stream()))


def _update(sum_t, min_t, L, capacity, idx, td, maxp, alpha, eps):
    c = _lib()
    c.check(c.lib().paintrl_prio_update(P(sum_t), P(min_t), L, capacity, P(idx), P(td), idx.numel(), P(maxp), alpha, eps, _stream()))


def _sample(sum_t, min_t, L, capacity, size, u, beta):
    c = _lib()
    idx = torch.empty(u.numel(), dtype=torch.int32, device=u.device)
    w = torch.empty(u.numel(), dtype=torch.float32, device=u.device)
    c.check(c.lib().paintrl_prio_sample(P(sum_t), P(min_t), L, capacity, size, P(u), u.numel(), beta, P(idx), P(w), _stream()))
    return idx.cpu().numpy(), w.cpu().numpy()


def _ulps(a, b):
    """Distance in FP64 ulps (both positive and finite)."""
    return np.abs(np.asarray(a, np.float64).view(np.int64) - np.asarray(b, np.float64).view(np.int64))


def _assert_nodes_rebuilt(sum_t, min_t, L):
    """Every internal node equals the NumPy pairwise rebuild from the kernel's own leaves, bit for bit."""
    s, m = sum_t.cpu().numpy(), min_t.cpu().numpy()
    rs, rm = s.copy(), m.copy()
    pr.rebuild(rs, rm, L)
    assert s[1:L].tobytes() == rs[1:L].tobytes()
    assert m[1:L].tobytes() == rm[1:L].tobytes()
    return s, m


@pytest.mark.parametrize('capacity', [5, 3000, 1 << 21])
def test_update_writes_leaves_nodes_and_max_priority(cuda_device, capacity):
    alpha, eps, n = 0.6, 1e-6, 4096
    L = 1 << (capacity - 1).bit_length()
    sum_t, min_t = _trees(L, cuda_device)
    maxp = torch.ones(1, dtype=torch.float64, device=cuda_device)
    _fill(sum_t, min_t, L, capacity, 0, capacity, maxp, alpha)
    g = torch.Generator(device=cuda_device).manual_seed(capacity)
    idx = torch.randint(0, capacity, (n,), generator=g, device=cuda_device, dtype=torch.int32)
    idx[n // 2:n // 2 + 64] = idx[:64]                               # duplicates, with identical td as in a minibatch
    table = torch.randn(capacity, generator=g, device=cuda_device) * 2.0
    table[:3] = torch.tensor([0.0, -0.0, 1e-30], device=cuda_device)
    idx[:3] = torch.arange(3, dtype=torch.int32, device=cuda_device) % capacity
    td = table[idx.long()]
    _update(sum_t, min_t, L, capacity, idx, td, maxp, alpha, eps)
    torch.cuda.synchronize()
    s, m = _assert_nodes_rebuilt(sum_t, min_t, L)
    i, t = idx.cpu().numpy(), td.cpu().numpy()
    p = np.abs(t.astype(np.float64)) + eps
    assert float(maxp) == max(1.0, float(p.max()))                    # exact: the max of the same FP64 values
    ref = np.ones(capacity)                                           # rows not in the minibatch keep 1^alpha = 1
    ref[i] = p ** alpha
    assert _ulps(s[L:L + capacity], ref).max() <= POW_ULP
    assert np.array_equal(s[L:L + capacity], m[L:L + capacity])
    assert (s[L + capacity:] == 0).all() and np.isinf(m[L + capacity:]).all()


def test_fill_across_the_wrap(cuda_device):
    capacity, L, alpha = 1000, 1024, 0.6
    sum_t, min_t = _trees(L, cuda_device)
    maxp = torch.full((1,), 2.5, dtype=torch.float64, device=cuda_device)
    _fill(sum_t, min_t, L, capacity, 900, 250, maxp, alpha)           # rows 900..999 and 0..149
    torch.cuda.synchronize()
    s, m = _assert_nodes_rebuilt(sum_t, min_t, L)
    rows = np.r_[900:1000, 0:150]
    other = np.setdiff1d(np.arange(L), rows)
    leaf = s[L + rows]
    assert (leaf == leaf[0]).all() and _ulps(leaf[0], 2.5 ** alpha) <= POW_ULP
    assert np.array_equal(m[L + rows], leaf)
    assert (s[L + other] == 0).all() and np.isinf(m[L + other]).all()
    with pytest.raises(Exception, match='count'):
        _fill(sum_t, min_t, L, capacity, 0, capacity + 1, maxp, alpha)
    with pytest.raises(Exception, match='power of two'):
        _fill(sum_t, min_t, 1000, capacity, 0, 10, maxp, alpha)


def _random_tree(cuda_device, capacity, size, seed):
    """Trees whose rows [0, size) were filled, then given priorities |td| + 1e-6 (td = randn^3, so they span decades)
    through prio_update; rows [size, capacity) stay unfilled."""
    L = 1 << (capacity - 1).bit_length()
    sum_t, min_t = _trees(L, cuda_device)
    maxp = torch.ones(1, dtype=torch.float64, device=cuda_device)
    _fill(sum_t, min_t, L, capacity, 0, size, maxp, 0.6)
    g = torch.Generator(device=cuda_device).manual_seed(seed)
    idx = torch.arange(size, dtype=torch.int32, device=cuda_device)
    td = torch.randn(size, generator=g, device=cuda_device) ** 3
    _update(sum_t, min_t, L, capacity, idx, td, maxp, 0.6, 1e-6)
    return L, sum_t, min_t


def test_sampling_matches_the_descent_replica(cuda_device):
    capacity, size, n = 5000, 4000, 4096
    L, sum_t, min_t = _random_tree(cuda_device, capacity, size, 3)
    s, m = sum_t.cpu().numpy(), min_t.cpu().numpy()
    leaves = s[L:]
    g = torch.Generator(device=cuda_device).manual_seed(9)
    u = torch.rand(n, generator=g, dtype=torch.float64, device=cuda_device)
    # edge uniforms: 0, the largest double below 1, and the prefix-sum boundaries of some rows and their neighbours
    prefix = np.cumsum(leaves[:size]) / s[1]
    edge = [0.0, 1.0 - 2.0 ** -53, 2.0 ** -60]
    for k in (0, 1, 17, size // 2, size - 2, size - 1):
        b = min(prefix[k], 1.0 - 2.0 ** -53)
        edge += [b, np.nextafter(b, 0.0), np.nextafter(b, 1.0) if b < 1.0 - 2.0 ** -53 else b]
    u[:len(edge)] = torch.tensor(edge, dtype=torch.float64, device=cuda_device)
    idx, w = _sample(sum_t, min_t, L, capacity, size, u, 0.4)
    ref = pr.descend(s, L, u.cpu().numpy())
    assert np.array_equal(idx, ref)
    assert (idx >= 0).all() and (idx < size).all() and (leaves[idx] > 0).all()
    # weights: (p_i / p_min)^-beta in FP64 (pow within 2 ulp), rounded to FP32: within one FP32 ulp of the FP64 formula
    wref = pr.weights(s, m, L, idx, 0.4)
    assert (np.abs(w.astype(np.float64) - wref) <= np.spacing(wref.astype(np.float32)).astype(np.float64)).all()
    assert (w <= 1.0).all()
    # the minimum-priority row gets exactly 1
    rmin = int(np.argmin(np.where(leaves[:size] > 0, leaves[:size], np.inf)))
    lo = (prefix[rmin - 1] if rmin else 0.0)
    u1 = torch.tensor([lo + 0.5 * (prefix[rmin] - lo)], dtype=torch.float64, device=cuda_device)
    i1, w1 = _sample(sum_t, min_t, L, capacity, size, u1, 0.4)
    assert i1[0] == rmin and w1[0] == 1.0


def test_sampling_guards_with_empty_rows_and_rounding(cuda_device):
    """Zero-priority rows between filled ones, all mass on the first or last filled row, and uniforms at 1 - 2^-53."""
    top = 1.0 - 2.0 ** -53
    for capacity, rows in ((8, [7]), (8, [0]), (1000, [3, 500, 999]), (77, list(range(0, 77, 5)))):
        L = 1 << (capacity - 1).bit_length()
        leaves = np.zeros(capacity)                                    # the kernels never write a zero leaf: set them here
        leaves[rows] = np.linspace(1.0, 3.0, len(rows))
        s, m = pr.tree_from_leaves(leaves, L)
        sum_t, min_t = torch.from_numpy(s).to(cuda_device), torch.from_numpy(m).to(cuda_device)
        u = torch.tensor([0.0, 0.25, 0.5, 0.999, top] + list(np.linspace(0.0, top, 2000)), dtype=torch.float64, device=cuda_device)
        idx, w = _sample(sum_t, min_t, L, capacity, capacity, u, 1.0)
        assert np.array_equal(idx, pr.descend(s, L, u.cpu().numpy()))
        assert set(idx.tolist()) <= set(rows) and (w <= 1.0).all()
        assert idx[0] == rows[0] and idx[4] == rows[-1]


def test_sampling_distribution_chi_square(cuda_device):
    from scipy import stats
    capacity, size, N = 64, 50, 10 ** 6
    L, sum_t, min_t = _random_tree(cuda_device, capacity, size, 5)
    s = sum_t.cpu().numpy()
    p = s[L:L + size] / s[1]
    g = torch.Generator(device=cuda_device).manual_seed(2024)
    u = torch.rand(N, generator=g, dtype=torch.float64, device=cuda_device)
    idx, _ = _sample(sum_t, min_t, L, capacity, size, u, 0.4)
    counts = np.bincount(idx, minlength=capacity)
    assert counts[size:].sum() == 0
    chi2 = float((((counts[:size] - N * p) ** 2) / (N * p)).sum())
    df = size - 1
    threshold = stats.chi2.ppf(1.0 - 1e-4, df)                      # p-value 1e-4: a correct sampler fails 1 seed in 10^4
    pval = float(stats.chi2.sf(chi2, df))
    print('chi-square of %d draws over %d rows: %.2f (threshold %.2f at p = 1e-4), p-value %.3f' % (N, size, chi2, threshold, pval))
    assert chi2 < threshold, (chi2, threshold, pval)


def test_alpha_or_beta_zero_gives_unit_weights(cuda_device):
    capacity, size = 300, 300
    L = 512
    g = torch.Generator(device=cuda_device).manual_seed(1)
    u = torch.rand(1000, generator=g, dtype=torch.float64, device=cuda_device)
    # alpha = 0: every leaf is (|td| + eps)^0 = 1
    sum_t, min_t = _trees(L, cuda_device)
    maxp = torch.ones(1, dtype=torch.float64, device=cuda_device)
    _fill(sum_t, min_t, L, capacity, 0, capacity, maxp, 0.0)
    idx = torch.arange(capacity, dtype=torch.int32, device=cuda_device)
    _update(sum_t, min_t, L, capacity, idx, torch.randn(capacity, generator=g, device=cuda_device), maxp, 0.0, 1e-6)
    assert (sum_t[L:L + capacity] == 1.0).all()
    _, w = _sample(sum_t, min_t, L, capacity, size, u, 0.4)
    assert (w == 1.0).all()
    # beta = 0 on a non-uniform tree
    L, sum_t, min_t = _random_tree(cuda_device, capacity, size, 8)
    _, w = _sample(sum_t, min_t, L, capacity, size, u, 0.0)
    assert (w == 1.0).all()


def _per_learner(cuda_device, obs_dim, n_out, minibatch=1024):
    from paintrl_b200 import dqn
    pol = _policy(obs_dim, n_out, cuda_device)
    return pol, dqn.DQNLearner(pol, dqn.DQNConfig(minibatch_size=minibatch, gamma=0.99, replay_capacity=128))


SHAPES = [(6, 4), (9, 7), (8, 15), (32, 15)]       # <8, 8>, <32, 8>, <8, 16>, <32, 16>


@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_unit_weights_equal_the_unweighted_loss(cuda_device, obs_dim, n_out):
    from paintrl_b200 import ppo
    pol, learner = _per_learner(cuda_device, obs_dim, n_out)
    target = ppo.flat_params(_policy(obs_dim, n_out, cuda_device, seed=11))
    buf = _transitions(1500, obs_dim, n_out, cuda_device, seed=obs_dim + n_out, reward_scale=1.5)
    g = torch.Generator(device=cuda_device).manual_seed(1)
    idx = torch.randint(0, 1500, (1000,), generator=g, device=cuda_device, dtype=torch.int32)
    idx[500:520] = idx[:20]                                            # duplicate rows
    ones = torch.ones(1000, device=cuda_device)
    g0, g1 = torch.zeros_like(learner.params), torch.zeros_like(learner.params)
    s0, s1 = torch.zeros(8, device=cuda_device), torch.zeros(8, device=cuda_device)
    td = torch.zeros(1000, device=cuda_device)
    learner.grad_into(buf, idx, g0, s0, target=target)
    learner.grad_weighted_into(buf, idx, ones, td, g1, s1, target=target)
    assert torch.equal(g0, g1)
    assert torch.equal(s0[:4], s1[:4])
    assert abs(float(s1[4]) - 1.0) <= 1e-6
    t = td.cpu().numpy()
    assert t[500:520].tobytes() == t[:20].tobytes()                   # duplicates carry bit-identical td
    learner.close()


@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_one_sample_power_of_two_weights_and_td_out(cuda_device, obs_dim, n_out):
    from paintrl_b200 import ppo
    pol, learner = _per_learner(cuda_device, obs_dim, n_out, minibatch=128)
    target = ppo.flat_params(_policy(obs_dim, n_out, cuda_device, seed=11))
    buf = _transitions(40, obs_dim, n_out, cuda_device, seed=3, reward_scale=1.5)
    td = torch.zeros(1, device=cuda_device)
    big = 0
    for r in range(40):
        idx = torch.tensor([r], dtype=torch.int32, device=cuda_device)
        g_ref, s_ref = torch.zeros_like(learner.params), torch.zeros(8, device=cuda_device)
        learner.grad_weighted_into(buf, idx, torch.ones(1, device=cuda_device), td, g_ref, s_ref, target=target)
        st = s_ref.cpu().numpy()
        assert td.cpu().numpy()[0] == np.float32(st[2] - st[3])        # td = Q(s, a) - y, from the one-sample statistics
        big += abs(float(td)) > 1.0
        for k in (-3, 1, 5):
            w = torch.full((1,), 2.0 ** k, device=cuda_device)
            g_w, s_w = torch.zeros_like(learner.params), torch.zeros(8, device=cuda_device)
            learner.grad_weighted_into(buf, idx, w, td, g_w, s_w, target=target)
            assert torch.equal(g_w, g_ref * 2.0 ** k), (r, k)
            assert float(s_w[0]) == float(s_ref[0]) * 2.0 ** k and float(s_w[4]) == 2.0 ** k
            assert torch.equal(s_w[1:4], s_ref[1:4])
    assert 0 < big < 40                                                # |td| on both sides of the Huber knee
    learner.close()


def _weighted_reference_grad(params, target, buf, idx, w, gamma, obs_dim, n_out, fwd):
    """mean_k w_k Huber(Q(s_k, a_k) - y_k) in torch autograd (layer-2 operands rounded to BF16 straight-through)."""
    torch.backends.cuda.matmul.allow_tf32 = False
    i = idx.long()
    _, an = _q_greedy(fwd(params, buf.next_obs, idx).cpu().numpy(), n_out)
    qt, _ = _q_greedy(fwd(target, buf.next_obs, idx).cpu().numpy(), n_out)
    y = buf.reward[i] + gamma * (1.0 - buf.done[i].float()) * torch.from_numpy(qt[np.arange(len(an)), an]).to(params.device)
    p = params.detach().clone().requires_grad_(True)
    w1, b1, w2, b2, w3, b3 = _split(p, obs_dim, n_out)
    bf = lambda t: t + (t.to(torch.bfloat16).float() - t).detach()
    h2 = torch.tanh(bf(torch.tanh(buf.obs[i].float() @ w1 + b1)) @ bf(w2) + b2)
    out = h2 @ w3 + b3
    A, V = out[:, :n_out], out[:, n_out:]
    qsa = (V + A - A.mean(1, keepdim=True)).gather(1, buf.actions[i][:, None])[:, 0]
    loss = (w * torch.nn.functional.huber_loss(qsa, y, delta=1.0, reduction='none')).mean()
    loss.backward()
    return p.grad.detach(), float(loss.detach())


@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_mixed_weights_match_autograd(cuda_device, obs_dim, n_out):
    from paintrl_b200 import ppo
    n_rows, n = 1500, 1000
    pol, learner = _per_learner(cuda_device, obs_dim, n_out)
    target = ppo.flat_params(_policy(obs_dim, n_out, cuda_device, seed=11))
    buf = _transitions(n_rows, obs_dim, n_out, cuda_device, seed=obs_dim + n_out, reward_scale=1.5)
    g = torch.Generator(device=cuda_device).manual_seed(1)
    idx = torch.randperm(n_rows, generator=g, device=cuda_device)[:n].to(torch.int32)
    w = torch.rand(n, generator=g, device=cuda_device) * 0.95 + 0.05
    fwd = _Forward(pol, n)
    grad, stats, td = torch.zeros_like(learner.params), torch.zeros(8, device=cuda_device), torch.zeros(n, device=cuda_device)
    learner.grad_weighted_into(buf, idx, w, td, grad, stats, target=target)
    ref, loss = _weighted_reference_grad(learner.params, target, buf, idx, w, 0.99, obs_dim, n_out, fwd)
    report = {name: _errors(a, b) for name, a, b in zip(('w1', 'b1', 'w2', 'b2', 'w3', 'b3'), _split(grad, obs_dim, n_out),
                                                        _split(ref, obs_dim, n_out))}
    print('weighted DQN grad errors obs %d n_out %d: %s' % (obs_dim, n_out, report))
    for name, (rel, cos) in report.items():
        assert rel <= GRAD_RTOL and cos >= GRAD_COS, (name, rel, cos)
    s = stats.cpu().numpy()
    assert abs(s[0] - loss) <= 2e-2 * abs(loss) and abs(s[4] - float(w.mean())) <= 1e-5
    fwd.close()
    learner.close()


def test_prioritized_nstep_learners_are_reproducible(cuda_device):
    from paintrl_b200 import dqn
    from paintrl_b200.batched_env import BatchedPaintEnv
    from paintrl_b200.config import EnvConfig
    from paintrl_b200.rollout import MlpPolicy, RolloutWorker
    from paintrl_b200.train import C2_SETTINGS
    n, T = 256, 20
    env = BatchedPaintEnv(n, EnvConfig(dict(C2_SETTINGS), auto_reset=True, seed=4), device=cuda_device)
    pol = MlpPolicy(env.obs_dim, 4, device=cuda_device, seed=6)
    eps = torch.full((1,), 0.5, device=cuda_device)
    worker = RolloutWorker(env, pol, fragment_length=T, use_cuda_graph=True, epsilon=eps)
    cfg = dqn.DQNConfig(minibatch_size=512, replay_capacity=16384, learning_starts=n * T, train_intensity=2.0,
                        target_update_freq=5, seed=2, prioritized_replay=True, n_step=3)
    learners = [dqn.DQNLearner(pol, cfg), dqn.DQNLearner(MlpPolicy(env.obs_dim, 4, device=cuda_device, seed=6), cfg)]
    worker.start((np.arange(n) % env.n_starts).astype(np.int32))
    outs = []
    for it in range(4):
        frag, _ = worker.collect()
        outs.append([L.update(frag) for L in learners])
    assert outs[0][0]['grad_steps'] == 0 and outs[0][0]['replay_size'] == (T - 2) * n
    assert outs[1][0]['grad_steps'] == 20 and outs[1][0]['replay_size'] == (2 * T - 2) * n
    for L in learners[1:]:
        assert torch.equal(learners[0].params, L.params) and torch.equal(learners[0].target, L.target)
        assert torch.equal(learners[0].replay.sum_tree, L.replay.sum_tree)
    last = outs[3][0]
    assert outs[3][0] == outs[3][1] and all(np.isfinite(last[k]) for k in dqn.PER_STAT_NAMES + ('grad_norm',))
    assert 0.0 < last['weight_mean'] <= 1.0
    s = learners[0].replay.sum_tree
    assert float(learners[0].replay.max_priority) >= 1.0 and float(s[1]) > 0.0
    for L in learners:
        L.close()
    env.close()


def test_weighted_loss_falls_on_a_fixed_buffer(cuda_device):
    from paintrl_b200 import dqn
    cfg = dqn.DQNConfig(minibatch_size=1024, replay_capacity=16384, target_update_freq=10 ** 9, lr=1e-3, seed=1,
                        prioritized_replay=True)
    pol = _policy(6, 4, cuda_device, seed=3)
    pol.head_w.mul_(0.1)
    learner = dqn.DQNLearner(pol, cfg)
    src = _transitions(cfg.replay_capacity, 6, 4, cuda_device, seed=3, learnable=True)
    rb = learner.replay
    for k in ('obs', 'next_obs', 'actions', 'reward', 'done'):
        getattr(rb, k).copy_(getattr(src, k))
    rb.size = cfg.replay_capacity
    _fill(rb.sum_tree, rb.min_tree, rb.L, rb.capacity, 0, rb.capacity, rb.max_priority, rb.alpha)
    stats = learner.train_steps(300).cpu().numpy()
    first, last = stats[:20, 0].mean(), stats[-20:, 0].mean()
    print('weighted Huber loss: first 20 steps %.4f, last 20 steps %.4f; mean weight %.3f -> %.3f'
          % (first, last, stats[:20, 4].mean(), stats[-20:, 4].mean()))
    assert np.isfinite(stats).all() and (stats[:, 4] <= 1.0).all() and (stats[:, 4] > 0.0).all()
    assert last < 0.8 * first, (first, last)
    learner.close()


def test_train_script_prioritized_nstep(cuda_device, tmp_path, capsys):
    from paintrl_b200 import train
    path = str(tmp_path / 'door_apex.pt')
    train.main(['--algo', 'dqn', '--prioritized-replay', '--n-step', '3', '--envs', '512', '--samples', str(512 * 100 * 2),
                '--checkpoint', path])
    lines = [json.loads(l) for l in capsys.readouterr().out.splitlines() if l.startswith('{')]
    assert len(lines) == 2
    assert lines[0]['learner']['grad_steps'] == 0 and lines[0]['learner']['replay_size'] == 98 * 512
    last = lines[-1]['learner']
    assert last['grad_steps'] == 100
    assert all(np.isfinite(last[k]) for k in ('loss', 'abs_td', 'q_mean', 'target_mean', 'weight_mean', 'grad_norm'))
    assert 0.0 < last['weight_mean'] <= 1.0
    ck = torch.load(path, map_location='cpu', weights_only=False)
    assert ck['algo'] == 'dqn'
    c = ck['learner']['config']
    assert c['prioritized_replay'] is True and c['n_step'] == 3 and c['prioritized_replay_alpha'] == 0.6
    pol = train.load_policy(path, cuda_device)
    out, _ = pol.forward(torch.zeros(3, pol.obs_dim, device=cuda_device, dtype=torch.float64))
    assert torch.isfinite(out).all()
