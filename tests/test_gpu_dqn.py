"""GPU: double DQN (paintrl_b200.dqn; the epsilon-greedy act kernel of csrc/paintrl_policy.cuh and the DQN loss stage of
csrc/paintrl_learn.cuh).

- epsilon-greedy act: at epsilon 0 the actions are the shared greedy rule on the logits of the same launch, and those
  logits are paintrl_policy_act's bit for bit; at epsilon 0.3 and 1 the exploration decisions and random actions are a
  NumPy replica of the documented draws; a captured graph follows epsilon.fill_() between replays;
- TD targets bit for bit against a NumPy replica on the kernel's own head outputs (distinct online and target
  parameters, dones cutting the bootstrap, the tie rule), and close to a plain torch FP32 network;
- the gradient against torch autograd on the same Huber dueling loss (layer-2 operands rounded to BF16 straight-through);
- clipping against torch.nn.utils.clip_grad_norm_; target sync cadence; reproducibility; learning."""
import ctypes

import numpy as np
import pytest
import torch

from test_gpu_policy import _uniform

pytestmark = pytest.mark.gpu

GRAD_RTOL, GRAD_COS = 2e-2, 0.999


def _policy(obs_dim, n_out, device, seed=5, discrete=True):
    from paintrl_b200.rollout import MlpPolicy
    pol = MlpPolicy(obs_dim, n_out, device=device, seed=seed, discrete=discrete)
    for w in pol.weights():
        if w.dim() == 1:
            w.copy_(torch.linspace(-0.3, 0.3, w.numel(), device=device))
    pol.head_w.mul_(10.0)
    return pol


def _split(p, obs_dim, n_out):
    sizes = [(obs_dim, 256), (256,), (256, 128), (128,), (128, n_out + 1), (n_out + 1,)]
    out, off = [], 0
    for s in sizes:
        n = int(np.prod(s))
        out.append(p[off:off + n].view(s))
        off += n
    return out


def _q_greedy(head, n_out):
    """dqn_q_values of paintrl_policy.cuh in float32: Q = V + (A - sum(A) / n_out), the sum in column order; the greedy
    action is the first maximum."""
    head = np.asarray(head, dtype=np.float32)
    sa = np.zeros(head.shape[0], dtype=np.float32)
    for o in range(n_out):
        sa = (sa + head[:, o]).astype(np.float32)
    ma = (sa / np.float32(n_out)).astype(np.float32)
    q = (head[:, n_out:n_out + 1] + (head[:, :n_out] - ma[:, None])).astype(np.float32)
    return q, q.argmax(axis=1)                    # numpy's argmax returns the first maximum


def _explore_replica(seed, batch, ctr, eps, greedy, n_out):
    env = np.arange(batch)
    explore = _uniform(seed, env, ctr, 0) < np.float32(eps)
    rand = np.minimum((_uniform(seed, env, ctr, 1) * np.float32(n_out)).astype(np.int64), n_out - 1)
    return explore, np.where(explore, rand, greedy)


def _tie(pol, n_out):
    """Columns 1 and 2 of the head identical and dominant: A_1 == A_2 > every other A on every row."""
    pol.head_w[:, 2] = pol.head_w[:, 1]
    pol.head_b[1] = 5.0
    pol.head_b[2] = 5.0


@pytest.mark.parametrize('obs_dim,n_out,batch', [(6, 4, 1000), (16, 8, 300), (32, 15, 4096)])
def test_epsilon_greedy_act(cuda_device, obs_dim, n_out, batch):
    from paintrl_b200.rollout import NativePolicy
    pol = _policy(obs_dim, n_out, cuda_device)
    assert pol.enable_native(batch)
    tied = _policy(obs_dim, n_out, cuda_device)
    _tie(tied, n_out)
    tied_native = NativePolicy(obs_dim, n_out, True, tied.weights(), batch, cuda_device, seed=5)
    g = torch.Generator(device=cuda_device).manual_seed(obs_dim)
    obs = torch.rand(batch, obs_dim, generator=g, device=cuda_device, dtype=torch.float64)
    actions = torch.full((batch,), -1, dtype=torch.int64, device=cuda_device)
    value = torch.zeros(batch, device=cuda_device)
    logits = torch.zeros(batch, n_out + 1, device=cuda_device)
    ref_logits = torch.zeros_like(logits)
    ref_value = torch.zeros_like(value)
    eps = torch.zeros(1, dtype=torch.float32, device=cuda_device)
    pol.native.act_into(obs, None, None, ref_value, logits=ref_logits, sample=False)      # no draw, counters untouched
    for ctr, e in enumerate((0.0, 0.3, 1.0, 0.0)):
        eps.fill_(e)
        pol.native.act_epsilon_into(obs, actions, value, eps, logits=logits)
        assert torch.equal(logits, ref_logits) and torch.equal(value, ref_value)
        _, greedy = _q_greedy(logits.cpu().numpy(), n_out)
        explore, expect = _explore_replica(5, batch, ctr, e, greedy, n_out)
        a = actions.cpu().numpy()
        assert np.array_equal(a, expect), (e, int((a != expect).sum()))
        if e == 0.0:
            assert not explore.any() and np.array_equal(a, greedy)
        elif e == 1.0:
            assert explore.all()
            if batch >= 1000:
                assert np.bincount(a, minlength=n_out).min() > 0
        else:
            assert 0.2 < explore.mean() < 0.4
    # ties: the lowest index
    tied_native.act_epsilon_into(obs, actions, value, torch.zeros(1, device=cuda_device), logits=logits)
    lg = logits.cpu().numpy()
    assert np.array_equal(lg[:, 1], lg[:, 2])
    assert (actions.cpu().numpy() == 1).all()
    tied_native.close()
    pol.native.close()


def test_epsilon_greedy_refuses_continuous_engines(cuda_device):
    from paintrl_b200 import _capi
    pol = _policy(6, 2, cuda_device, discrete=False)
    assert pol.enable_native(128)
    lib = _capi.lib()
    obs = torch.zeros(128, 6, dtype=torch.float64, device=cuda_device)
    buf = torch.zeros(128 * 4, device=cuda_device)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    assert lib.paintrl_policy_act_epsilon(pol.native._h, P(obs), 128, P(buf), P(buf), None, P(buf), None) == -1
    assert b'discrete' in lib.paintrl_last_error()
    with pytest.raises(ValueError, match='discrete'):
        pol.native.act_epsilon_into(obs, buf, buf, buf[:1])
    pol.native.close()


def test_captured_graph_follows_epsilon(cuda_device):
    obs_dim, n_out, batch = 6, 4, 512
    pol = _policy(obs_dim, n_out, cuda_device)
    assert pol.enable_native(batch)
    obs = torch.rand(batch, obs_dim, device=cuda_device, dtype=torch.float64)
    actions = torch.zeros(batch, dtype=torch.int64, device=cuda_device)
    value = torch.zeros(batch, device=cuda_device)
    logits = torch.zeros(batch, n_out + 1, device=cuda_device)
    eps = torch.zeros(1, device=cuda_device)
    s = torch.cuda.Stream(cuda_device)
    with torch.cuda.stream(s):
        pol.native.act_epsilon_into(obs, actions, value, eps, logits=logits)          # warm-up launch: counter 0
    torch.cuda.synchronize(cuda_device)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pol.native.act_epsilon_into(obs, actions, value, eps, logits=logits)
    _, greedy = _q_greedy(logits.cpu().numpy(), n_out)
    for ctr, e in zip((1, 2, 3), (1.0, 0.0, 0.3)):
        eps.fill_(e)
        graph.replay()
        _, expect = _explore_replica(5, batch, ctr, e, greedy, n_out)
        assert np.array_equal(actions.cpu().numpy(), expect), e
    pol.native.close()


def _transitions(n_rows, obs_dim, n_out, device, seed, reward_scale=1.0, learnable=False):
    g = torch.Generator(device=device).manual_seed(seed)

    class Buf(object):
        pass
    b = Buf()
    b.obs = torch.rand(n_rows, obs_dim, generator=g, device=device, dtype=torch.float64)
    b.next_obs = torch.rand(n_rows, obs_dim, generator=g, device=device, dtype=torch.float64)
    b.actions = torch.randint(0, n_out, (n_rows,), generator=g, device=device)
    b.reward = reward_scale * torch.randn(n_rows, generator=g, device=device)
    b.done = (torch.rand(n_rows, generator=g, device=device) < 0.3).to(torch.uint8)
    if learnable:                                  # a reward the network can fit: a function of s and a
        b.reward = (3.0 * (b.obs[:, 0] - 0.5) + (b.actions - 1.5)).float()
    return b


class _Forward(object):
    """paintrl_ppo_forward on arbitrary flat parameters: the kernel's own head outputs."""

    def __init__(self, pol, n):
        from paintrl_b200 import ppo
        self.ppo = ppo.PPOLearner(pol, ppo.PPOConfig(minibatch_size=((n + 127) // 128) * 128))
        self.n_out = pol.n_out

    def __call__(self, params, obs, idx):
        from paintrl_b200 import _capi
        out = torch.empty(idx.numel(), self.n_out + 1, device=obs.device)
        P = lambda t: ctypes.c_void_p(t.data_ptr())
        _capi.check(self.ppo._lib.paintrl_ppo_forward(self.ppo._h, P(params), P(idx), idx.numel(), P(obs), P(out),
                                                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return out

    def close(self):
        self.ppo.close()


def _torch_head(params, obs, obs_dim, n_out):
    torch.backends.cuda.matmul.allow_tf32 = False
    w1, b1, w2, b2, w3, b3 = _split(params, obs_dim, n_out)
    return torch.tanh(torch.tanh(obs.float() @ w1 + b1) @ w2 + b2) @ w3 + b3


def test_td_targets(cuda_device):
    from paintrl_b200 import dqn, ppo
    obs_dim, n_out, rows = 6, 4, 48
    online_pol = _policy(obs_dim, n_out, cuda_device, seed=1)
    _tie(online_pol, n_out)                        # argmax_a Q_online(s', a) is a tie of 1 and 2 on every row
    target_pol = _policy(obs_dim, n_out, cuda_device, seed=2)
    learner = dqn.DQNLearner(online_pol, dqn.DQNConfig(minibatch_size=128, gamma=0.9, replay_capacity=128))
    target = ppo.flat_params(target_pol)
    fwd = _Forward(online_pol, rows)
    buf = _transitions(rows, obs_dim, n_out, cuda_device, seed=7)
    idx_all = torch.arange(rows, dtype=torch.int32, device=cuda_device)
    head_o = fwd(learner.params, buf.next_obs, idx_all).cpu().numpy()
    head_t = fwd(target, buf.next_obs, idx_all).cpu().numpy()
    head_s = fwd(learner.params, buf.obs, idx_all).cpu().numpy()
    assert np.array_equal(head_o[:, 1], head_o[:, 2])
    qo, an = _q_greedy(head_o, n_out)
    qt, _ = _q_greedy(head_t, n_out)
    qs, _ = _q_greedy(head_s, n_out)
    assert (an == 1).all()
    assert (qt[:, 1] != qt[:, 2]).all()            # the tie rule decides which target value is taken
    r = buf.reward.cpu().numpy()
    nd = np.where(buf.done.cpu().numpy() != 0, np.float32(0), np.float32(1))
    y_ref = (r + (np.float32(0.9) * nd) * qt[np.arange(rows), an]).astype(np.float32)
    a = buf.actions.cpu().numpy()
    stats = torch.zeros(rows, 8, device=cuda_device)
    for k in range(rows):                          # n = 1: the statistics are that row's own values
        learner.grad_into(buf, idx_all[k:k + 1], learner.grad, stats[k], target=target)
    st = stats.cpu().numpy()
    assert np.array_equal(st[:, 3], y_ref)
    assert np.array_equal(st[:, 2], qs[np.arange(rows), a])
    done = buf.done.cpu().numpy() != 0
    assert done.any() and (~done).any()
    assert np.array_equal(st[done, 3], r[done])    # done cuts the bootstrap
    td = st[:, 2] - st[:, 3]
    huber = np.where(np.abs(td) <= 1, 0.5 * td * td, np.abs(td) - 0.5)
    assert np.allclose(st[:, 0], huber, rtol=1e-6, atol=1e-7) and np.allclose(st[:, 1], np.abs(td), rtol=1e-6)
    # against a plain torch FP32 network: the kernel runs layer 2 in BF16, so within 2e-2 of the Q scale
    ht = _torch_head(target, buf.next_obs, obs_dim, n_out).cpu().numpy()
    qt_ref = ht[:, n_out:] + ht[:, :n_out] - ht[:, :n_out].mean(1, keepdims=True)
    y_torch = r + 0.9 * nd * qt_ref[:, 1]
    assert np.abs(st[:, 3] - y_torch).max() < 2e-2 * max(1.0, np.abs(qt_ref).max())
    fwd.close()
    learner.close()


def _reference_grad(params, target, buf, idx, gamma, obs_dim, n_out, fwd):
    """The DQN loss in torch autograd (layer-2 operands rounded to BF16 straight-through, FP32 elsewhere); y from the
    kernel's own head outputs on s', a constant."""
    torch.backends.cuda.matmul.allow_tf32 = False
    i = idx.long()
    qo, an = _q_greedy(fwd(params, buf.next_obs, idx).cpu().numpy(), n_out)
    qt, _ = _q_greedy(fwd(target, buf.next_obs, idx).cpu().numpy(), n_out)
    nd = 1.0 - buf.done[i].float()
    y = buf.reward[i] + gamma * nd * torch.from_numpy(qt[np.arange(len(an)), an]).to(params.device)
    p = params.detach().clone().requires_grad_(True)
    w1, b1, w2, b2, w3, b3 = _split(p, obs_dim, n_out)
    bf = lambda t: t + (t.to(torch.bfloat16).float() - t).detach()
    h1 = torch.tanh(buf.obs[i].float() @ w1 + b1)
    h2 = torch.tanh(bf(h1) @ bf(w2) + b2)
    out = h2 @ w3 + b3
    A, V = out[:, :n_out], out[:, n_out:]
    Q = V + A - A.mean(1, keepdim=True)
    qsa = Q.gather(1, buf.actions[i][:, None])[:, 0]
    loss = torch.nn.functional.huber_loss(qsa, y, delta=1.0)
    loss.backward()
    big = float(((qsa - y).abs() > 1.0).float().mean())
    return p.grad.detach(), big, float(loss.detach())


def _errors(a, b):
    rel = float((a - b).norm() / b.norm().clamp_min(1e-30))
    cos = float((a * b).sum() / (a.norm() * b.norm()).clamp_min(1e-30))
    return rel, cos


@pytest.mark.parametrize('obs_dim,n_out', [(6, 4), (16, 8), (32, 15)])
def test_gradient_matches_autograd(cuda_device, obs_dim, n_out):
    from paintrl_b200 import dqn, ppo
    n_rows, n = 1500, 1000                        # n = 1000: a ragged last tile
    pol = _policy(obs_dim, n_out, cuda_device)
    learner = dqn.DQNLearner(pol, dqn.DQNConfig(minibatch_size=1024, gamma=0.99, replay_capacity=128))
    target = ppo.flat_params(_policy(obs_dim, n_out, cuda_device, seed=11))
    buf = _transitions(n_rows, obs_dim, n_out, cuda_device, seed=obs_dim + n_out, reward_scale=1.5)
    g = torch.Generator(device=cuda_device).manual_seed(1)
    idx = torch.randperm(n_rows, generator=g, device=cuda_device)[:n].to(torch.int32)
    fwd = _Forward(pol, n)
    grad = torch.zeros_like(learner.params)
    stats = torch.zeros(8, device=cuda_device)
    learner.grad_into(buf, idx, grad, stats, target=target)
    ref, big, loss = _reference_grad(learner.params, target, buf, idx, 0.99, obs_dim, n_out, fwd)
    assert 0.05 < big < 0.95, big                 # |td| on both sides of delta = 1
    report = {}
    for name, a, b in zip(('w1', 'b1', 'w2', 'b2', 'w3', 'b3'), _split(grad, obs_dim, n_out), _split(ref, obs_dim, n_out)):
        report[name] = _errors(a, b)
    worst = max(r for r, _ in report.values()), min(c for _, c in report.values())
    print('DQN grad errors obs %d n_out %d: worst rel Frobenius %.3g, lowest cosine %.7f; %s' % (obs_dim, n_out, worst[0], worst[1], report))
    for name, (rel, cos) in report.items():
        assert rel <= GRAD_RTOL and cos >= GRAD_COS, (name, rel, cos)
    s = stats.cpu().numpy()
    assert abs(s[0] - loss) <= 2e-2 * abs(loss) and np.isfinite(s).all()
    fwd.close()
    learner.close()


def test_clip_grad_norm_matches_torch(cuda_device):
    from paintrl_b200 import _capi
    lib = _capi.lib()
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device=cuda_device).manual_seed(0)
    for n in (1, 1000, 43077, 300001):
        grad = torch.randn(n, generator=g, device=cuda_device) * 3.0
        norm = torch.zeros(1, device=cuda_device)
        ref = grad.clone().requires_grad_(False)
        p = torch.nn.Parameter(torch.zeros(n, device=cuda_device))
        p.grad = ref
        max_norm = 0.5 * float(torch.linalg.vector_norm(grad))
        ref_norm = float(torch.nn.utils.clip_grad_norm_([p], max_norm))
        _capi.check(lib.paintrl_clip_grad_norm(P(grad), n, max_norm, P(norm), stream))
        assert abs(float(norm) - ref_norm) <= 1e-5 * ref_norm, (n, float(norm), ref_norm)
        torch.testing.assert_close(grad, p.grad, rtol=1e-5, atol=1e-7)
        # under max_norm: untouched, bit for bit
        before = grad.clone()
        _capi.check(lib.paintrl_clip_grad_norm(P(grad), n, 2.0 * max_norm, P(norm), stream))
        assert torch.equal(grad, before)
        assert abs(float(norm) - 0.5 * ref_norm) <= 1e-5 * ref_norm
    # the norm is the same on every run
    grad = torch.randn(43077, generator=g, device=cuda_device)
    norms = torch.zeros(3, device=cuda_device)
    for k in range(3):
        _capi.check(lib.paintrl_clip_grad_norm(P(grad), grad.numel(), 1e9, P(norms[k:]), stream))
    assert norms[0] == norms[1] == norms[2]


def _filled_learner(cuda_device, cfg, seed=0, learnable=False):
    from paintrl_b200 import dqn
    obs_dim, n_out = 6, 4
    pol = _policy(obs_dim, n_out, cuda_device, seed=3)
    pol.head_w.mul_(0.1)
    learner = dqn.DQNLearner(pol, cfg)
    src = _transitions(cfg.replay_capacity, obs_dim, n_out, cuda_device, seed=seed, learnable=learnable)
    for k in ('obs', 'next_obs', 'actions', 'reward', 'done'):
        getattr(learner.replay, k).copy_(getattr(src, k))
    learner.replay.size = cfg.replay_capacity
    return learner


def test_target_sync_cadence_and_reproducibility(cuda_device):
    from paintrl_b200 import dqn
    cfg = dqn.DQNConfig(minibatch_size=256, replay_capacity=4096, target_update_freq=3, lr=1e-3, seed=4)
    learner = _filled_learner(cuda_device, cfg)
    assert torch.equal(learner.target, learner.params)
    synced = learner.params.clone()
    for step in range(1, 8):
        learner.train_steps(1)
        assert learner.step == step
        if step % 3 == 0:
            assert torch.equal(learner.target, learner.params)
            synced = learner.params.clone()
        else:
            assert torch.equal(learner.target, synced) and not torch.equal(learner.target, learner.params)
    # two learners with the same seed and data: identical parameters, and a resumed learner continues bit for bit
    twin = _filled_learner(cuda_device, cfg)
    twin.train_steps(7)
    assert torch.equal(twin.params, learner.params) and torch.equal(twin.target, learner.target)
    sd = learner.state_dict()
    learner.train_steps(5)
    resumed = _filled_learner(cuda_device, cfg)
    resumed.load_state_dict(sd)
    resumed.train_steps(5)
    assert torch.equal(resumed.params, learner.params) and torch.equal(resumed.target, learner.target)
    for x in (learner, twin, resumed):
        x.close()


def test_update_from_fragments_is_reproducible(cuda_device):
    """Two learners with the same seed on the same fragments (collected epsilon-greedily in a captured graph): identical
    parameters; the first fragment only fills the buffer (learning_starts)."""
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
    cfg = dqn.DQNConfig(minibatch_size=512, replay_capacity=8192, learning_starts=n * T + 1, train_intensity=2.0,
                        target_update_freq=5, seed=2)
    learners = [dqn.DQNLearner(pol, cfg), dqn.DQNLearner(MlpPolicy(env.obs_dim, 4, device=cuda_device, seed=6), cfg)]
    worker.start((np.arange(n) % env.n_starts).astype(np.int32))
    outs = []
    for it in range(3):
        frag, _ = worker.collect()
        a = frag.actions.cpu().numpy()
        assert a.min() >= 0 and a.max() <= 3
        outs.append([L.update(frag) for L in learners])
    assert worker._graph is not None, worker.graph_error
    assert outs[0][0]['grad_steps'] == 0 and outs[1][0]['grad_steps'] == 20       # ceil(2 * 5120 / 512)
    assert torch.equal(learners[0].params, learners[1].params) and torch.equal(learners[0].target, learners[1].target)
    assert outs[2][0] == outs[2][1] and all(np.isfinite(outs[2][0][k]) for k in dqn.STAT_NAMES)
    assert torch.equal(dqn.flat_params(pol), learners[0].params)
    for L in learners:
        L.close()
    env.close()


def test_huber_loss_falls_on_a_fixed_buffer(cuda_device):
    from paintrl_b200 import dqn
    cfg = dqn.DQNConfig(minibatch_size=1024, replay_capacity=16384, target_update_freq=10 ** 9, lr=1e-3, seed=1)
    learner = _filled_learner(cuda_device, cfg, seed=3, learnable=True)
    stats = learner.train_steps(300).cpu().numpy()
    first, last = stats[:20, 0].mean(), stats[-20:, 0].mean()
    print('Huber loss: first 20 steps %.4f, last 20 steps %.4f' % (first, last))
    assert np.isfinite(stats).all()
    assert last < 0.8 * first, (first, last)
    learner.close()


def test_train_script_dqn_on_the_door(cuda_device, tmp_path, capsys):
    import json
    from paintrl_b200 import train
    path = str(tmp_path / 'door_dqn.pt')
    train.main(['--algo', 'dqn', '--envs', '512', '--samples', str(512 * 100 * 4), '--checkpoint', path])
    lines = [json.loads(l) for l in capsys.readouterr().out.splitlines() if l.startswith('{')]
    assert len(lines) == 4
    assert lines[0]['epsilon'] == 1.0 and lines[-1]['epsilon'] < lines[0]['epsilon']
    assert lines[0]['learner']['grad_steps'] == 0                   # learning_starts 65536 > 51200
    last = lines[-1]['learner']
    assert last['grad_steps'] == 100 and all(np.isfinite(last[k]) for k in ('loss', 'abs_td', 'q_mean', 'target_mean', 'grad_norm'))
    ck = torch.load(path, map_location='cpu', weights_only=False)
    assert ck['algo'] == 'dqn' and 'target_params' in ck['learner']
    pol = train.load_policy(path, cuda_device)
    out, _ = pol.forward(torch.zeros(3, pol.obs_dim, device=cuda_device, dtype=torch.float64))
    assert torch.isfinite(out).all()
