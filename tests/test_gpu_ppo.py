"""GPU: the PPO learner (paintrl_b200.ppo, csrc/paintrl_learn.cuh).

- the learner kernel's forward equals the act kernel's logits / value bit for bit, and the first minibatch of an
  update sees ratios of exactly 1;
- its gradient against torch autograd on the same loss (layer-2 operands rounded to BF16 straight-through, FP32
  elsewhere), with policy and value clipping both active on part of the rows;
- Adam against torch.optim.Adam, the in-place weight refresh against a freshly created engine, a captured rollout
  graph picking up new weights, reproducibility, and learning on the door panel."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GRAD_RTOL, GRAD_COS = 2e-2, 0.999


def _policy(obs_dim, n_out, discrete, device, seed=5):
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


def _reference_grad(params, rows, idx, cfg, kl_coeff, obs_dim, n_out, discrete):
    """The learner's loss in torch autograd: layer-2 operands rounded to BF16 (straight-through), FP32 elsewhere."""
    torch.backends.cuda.matmul.allow_tf32 = False
    p = params.detach().clone().requires_grad_(True)
    w1, b1, w2, b2, w3, b3 = _split(p, obs_dim, n_out)
    i = idx.long()
    x = rows['obs'][i].float()
    bf = lambda t: t + (t.to(torch.bfloat16).float() - t).detach()
    h1 = torch.tanh(x @ w1 + b1)
    h2 = torch.tanh(bf(h1) @ bf(w2) + b2)
    out = h2 @ w3 + b3
    logits, v = out[:, :n_out], out[:, n_out]
    old = rows['logits'][i][:, :n_out]
    if discrete:
        lp_all = torch.log_softmax(logits, 1)
        logp = lp_all.gather(1, rows['actions'][i][:, None])[:, 0]
        lpo = torch.log_softmax(old, 1)
        kl = (lpo.exp() * (lpo - lp_all)).sum(1)
        ent = -(lp_all.exp() * lp_all).sum(1)
    else:
        mu = torch.tanh(logits)
        logp = (-0.5 * (rows['actions'][i].float() - mu) ** 2 - 0.5 * math.log(2 * math.pi)).sum(1)
        kl = 0.5 * ((torch.tanh(old) - mu) ** 2).sum(1)
        ent = torch.full_like(v, n_out * (0.5 + 0.5 * math.log(2 * math.pi)))
    A, R, vold = rows['adv'][i], rows['vtarg'][i], rows['value'][i]
    r = torch.exp(logp - rows['logp'][i])
    surr = torch.min(A * r, A * torch.clamp(r, 1 - cfg.clip_param, 1 + cfg.clip_param))
    vf1 = (v - R) ** 2
    vf2 = (vold + torch.clamp(v - vold, -cfg.vf_clip_param, cfg.vf_clip_param) - R) ** 2
    loss = (-surr + kl_coeff * kl + cfg.vf_loss_coeff * torch.max(vf1, vf2) - cfg.entropy_coeff * ent).mean()
    loss.backward()
    frac_clip = float(((r - 1).abs() > cfg.clip_param).float().mean())
    frac_vclip = float(((v - vold).abs() > cfg.vf_clip_param).float().mean())
    return p.grad.detach(), frac_clip, frac_vclip, float(loss.detach())


def _rows(pol, n_rows, obs_dim, n_out, discrete, device, seed):
    """A synthetic flattened fragment sampled by the act kernel: obs, actions, logp, value, logits (the 'old' policy)."""
    g = torch.Generator(device=device).manual_seed(seed)
    assert pol.enable_native(n_rows)
    obs = torch.rand(n_rows, obs_dim, generator=g, device=device, dtype=torch.float64)
    actions = (torch.zeros(n_rows, dtype=torch.int64, device=device) if discrete else
               torch.zeros(n_rows, n_out, dtype=torch.float64, device=device))
    logp = torch.zeros(n_rows, dtype=torch.float32, device=device)
    value = torch.zeros(n_rows, dtype=torch.float32, device=device)
    logits = torch.zeros(n_rows, n_out + 1, dtype=torch.float32, device=device)
    pol.native.act_into(obs, actions, logp, value, logits=logits)
    adv = torch.randn(n_rows, generator=g, device=device)
    vtarg = value + 0.5 * torch.randn(n_rows, generator=g, device=device)
    return {'obs': obs, 'actions': actions, 'logp': logp, 'value': value, 'logits': logits, 'adv': adv, 'vtarg': vtarg}


def _errors(a, b):
    rel = float((a - b).norm() / b.norm().clamp_min(1e-30))
    cos = float((a * b).sum() / (a.norm() * b.norm()).clamp_min(1e-30))
    return rel, cos


@pytest.mark.parametrize('discrete', [True, False])
@pytest.mark.parametrize('obs_dim,n_out', [(6, 4), (16, 2), (32, 15)])
def test_gradient_matches_autograd(cuda_device, obs_dim, n_out, discrete):
    from paintrl_b200 import ppo
    n_rows, n = 1500, 1000                        # n = 1000: a ragged last tile
    pol = _policy(obs_dim, n_out, discrete, cuda_device)
    rows = _rows(pol, n_rows, obs_dim, n_out, discrete, cuda_device, seed=obs_dim + n_out)
    g = torch.Generator(device=cuda_device).manual_seed(1)
    params = ppo.flat_params(pol)
    for t in _split(params, obs_dim, n_out):                  # each tensor by 20 % of its spread
        t.add_(0.2 * t.std() * torch.randn(t.shape, generator=g, device=cuda_device))
    idx = torch.randperm(n_rows, generator=g, device=cuda_device)[:n].to(torch.int32)
    # value clip at the median value change, so that about half of the rows are clipped
    w1, b1, w2, b2, w3, b3 = _split(params, obs_dim, n_out)
    v_new = (torch.tanh(torch.tanh(rows['obs'][idx.long()].float() @ w1 + b1) @ w2 + b2) @ w3 + b3)[:, n_out]
    vf_clip = float((v_new - rows['value'][idx.long()]).abs().median())
    cfg = ppo.PPOConfig(minibatch_size=1024, clip_param=0.1, vf_clip_param=vf_clip, entropy_coeff=0.01)
    learner = ppo.PPOLearner(pol, cfg)
    learner.params.copy_(params)
    grad = torch.zeros_like(learner.params)
    stats = torch.zeros(8, device=cuda_device)
    learner.grad_into(rows, idx, 0.2, grad, stats)
    ref, frac_clip, frac_vclip, loss = _reference_grad(learner.params, rows, idx, cfg, 0.2, obs_dim, n_out, discrete)
    assert 0.05 < frac_clip < 0.95, frac_clip           # the perturbation puts both clips to work on part of the rows
    assert 0.05 < frac_vclip < 0.95, frac_vclip
    names = ('w1', 'b1', 'w2', 'b2', 'w3', 'b3')
    report = {}
    for name, a, b in zip(names, _split(grad, obs_dim, n_out), _split(ref, obs_dim, n_out)):
        report[name] = _errors(a, b)
    print('grad errors (rel Frobenius, cosine) obs %d n_out %d discrete %s: %s' % (obs_dim, n_out, discrete, report))
    for name, (rel, cos) in report.items():
        assert rel <= GRAD_RTOL and cos >= GRAD_COS, (name, rel, cos)
    s = stats.cpu().numpy()
    assert abs(s[4] - frac_clip) < 0.01
    assert np.isfinite(s).all()
    learner.close()
    pol.native.close()


def test_forward_parity_and_unit_ratio_on_a_fragment(cuda_device):
    from paintrl_b200 import ppo
    from paintrl_b200.batched_env import BatchedPaintEnv
    from paintrl_b200.config import EnvConfig
    from paintrl_b200.rollout import MlpPolicy, RolloutWorker
    from paintrl_b200.train import C2_SETTINGS
    n, T = 512, 16
    env = BatchedPaintEnv(n, EnvConfig(dict(C2_SETTINGS), auto_reset=True, seed=2), device=cuda_device)
    pol = MlpPolicy(env.obs_dim, 4, device=cuda_device, seed=3)
    worker = RolloutWorker(env, pol, fragment_length=T, keep_logits=True)
    worker.start((np.arange(n) % env.n_starts).astype(np.int32))
    frag, _ = worker.collect()
    learner = ppo.PPOLearner(pol, ppo.PPOConfig(minibatch_size=4096))
    rows = learner.flatten(frag)
    N = rows['n']
    idx = torch.randperm(N, device=cuda_device).to(torch.int32)
    out = learner.forward(rows['obs'], idx)
    assert torch.equal(out, rows['logits'][idx.long()])
    assert torch.equal(out[:, 4], rows['value'][idx.long()])
    stats = torch.zeros(8, device=cuda_device)
    learner.grad_into(rows, idx[:4096], learner.kl_coeff, learner.grad, stats)
    s = stats.cpu().numpy()
    assert s[5] == 1.0 and s[4] == 0.0 and s[2] == 0.0, s          # mean ratio, clip fraction, KL
    learner.close()
    env.close()


def test_adam_matches_torch(cuda_device):
    from paintrl_b200 import _capi
    import ctypes
    lib = _capi.lib()
    g = torch.Generator(device=cuda_device).manual_seed(0)
    n = 100003
    p = torch.randn(n, generator=g, device=cuda_device)
    ref = p.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    for step in range(1, 6):
        grad = torch.randn(n, generator=g, device=cuda_device) * (10.0 ** (step - 3))
        _capi.check(lib.paintrl_adam_step(P(p), P(grad), P(m), P(v), n, 1e-3, 0.9, 0.999, 1e-8, step,
                                          ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        ref.grad = grad.clone()
        opt.step()
        torch.testing.assert_close(p, ref.detach(), rtol=1e-6, atol=1e-6)


def test_set_params_equals_a_fresh_engine(cuda_device):
    from paintrl_b200 import ppo
    from paintrl_b200.rollout import NativePolicy
    obs_dim, n_out, B = 16, 4, 1000
    a = _policy(obs_dim, n_out, True, cuda_device, seed=1)
    b = _policy(obs_dim, n_out, True, cuda_device, seed=2)
    assert a.enable_native(B)
    obs = torch.rand(B, obs_dim, device=cuda_device, dtype=torch.float64)
    value = torch.zeros(B, device=cuda_device)
    la = torch.zeros(B, n_out + 1, device=cuda_device)
    lb = torch.zeros_like(la)
    a.native.act_into(obs, None, None, value, logits=la, sample=False)
    a.native.set_params(ppo.flat_params(b))
    a.native.act_into(obs, None, None, value, logits=la, sample=False)
    fresh = NativePolicy(obs_dim, n_out, True, b.weights(), B, cuda_device)
    fresh.act_into(obs, None, None, value, logits=lb, sample=False)
    assert torch.equal(la, lb)
    fresh.close()
    a.native.close()


def _snapshot(frag):
    class F(object):
        pass
    s = F()
    for k, v in vars(frag).items():
        setattr(s, k, v.clone() if torch.is_tensor(v) else v)
    return s


def test_captured_graph_samples_with_updated_weights(cuda_device):
    """A worker whose graph was captured before an update replays with the new weights: its next fragment equals the
    one an eager twin (same environments, policy and learner) collects."""
    from paintrl_b200 import ppo
    from paintrl_b200.batched_env import BatchedPaintEnv
    from paintrl_b200.config import EnvConfig
    from paintrl_b200.rollout import MlpPolicy, RolloutWorker
    from paintrl_b200.train import C2_SETTINGS
    n, T = 256, 20
    runs = []
    for graph in (True, False):
        env = BatchedPaintEnv(n, EnvConfig(dict(C2_SETTINGS), auto_reset=True, seed=4), device=cuda_device)
        pol = MlpPolicy(env.obs_dim, 4, device=cuda_device, seed=6)
        worker = RolloutWorker(env, pol, fragment_length=T, use_cuda_graph=graph, keep_logits=True)
        learner = ppo.PPOLearner(pol, ppo.PPOConfig(minibatch_size=1024, num_sgd_iter=2, lr=1e-3, seed=1))
        worker.start((np.arange(n) % env.n_starts).astype(np.int32))
        worker.collect()
        frag, _ = worker.collect()                # graph: captured here
        if graph:
            assert worker._graph is not None, worker.graph_error
        before = _snapshot(frag)
        learner.update(frag)
        frag, _ = worker.collect()                # graph: replayed with the refreshed weights
        after = _snapshot(frag)
        rows = learner.flatten(frag)
        idx = torch.arange(rows['n'], device=cuda_device, dtype=torch.int32)
        assert torch.equal(learner.forward(rows['obs'], idx), rows['logits'])
        assert not torch.equal(before.logits, after.logits)
        runs.append((after, learner.params.clone()))
        learner.close()
        env.close()
    (fa, pa), (fb, pb) = runs
    assert torch.equal(pa, pb)
    for k in ('obs', 'actions', 'logits', 'logp', 'value', 'reward', 'done'):
        assert torch.equal(getattr(fa, k), getattr(fb, k)), k


def test_training_is_reproducible_and_resumable(cuda_device):
    from paintrl_b200 import ppo
    from paintrl_b200.rollout import MlpPolicy
    from paintrl_b200.train import Trainer
    cfg = dict(minibatch_size=1024, num_sgd_iter=2, lr=3e-4, seed=3)
    finals = []
    for run in range(2):
        tr = Trainer(0, 512, 20, seed=3, device=cuda_device, config=ppo.PPOConfig(**cfg))
        for _ in range(3):
            tr.iteration()
        finals.append(tr.learner.params.clone())
        if run == 1:
            sd = tr.learner.state_dict()
            frag, _ = tr.worker.collect()
            snap = _snapshot(frag)
            tr.learner.update(frag)
            cont = tr.learner.params.clone()
            pol = MlpPolicy(tr.policy.obs_dim, 4, device=cuda_device, seed=99)
            fresh = ppo.PPOLearner(pol, ppo.PPOConfig(**cfg))
            fresh.load_state_dict(sd)
            fresh.update(snap)
            assert torch.equal(fresh.params, cont)
            assert torch.equal(ppo.flat_params(pol), cont)
            fresh.close()
        tr.close()
    assert torch.equal(finals[0], finals[1])


# Learning on the door (C2 settings), 2048 environments x 100 steps per iteration, 8 iterations (about 2 s of GPU time).
def test_learning_on_the_door(cuda_device):
    from paintrl_b200 import ppo
    from paintrl_b200.train import Trainer
    tr = Trainer(0, 2048, 100, seed=0, device=cuda_device, config=ppo.PPOConfig(minibatch_size=4096, num_sgd_iter=8, lr=1e-3, seed=0))
    hist = [tr.iteration() for _ in range(8)]
    tr.close()
    print('learning curve:', [(h['env_steps'], h['mean_return'], h['coverage'], h['length_ratio']) for h in hist])
    # Measured on a B200 with these settings: mean episode return 0.86 -> 30.2 and coverage 0.039 -> 0.596 from the first
    # to the eighth iteration.  The thresholds ask for about a third of those gains: a policy that does not learn
    # stays near the first iteration's values, one that learns at all clears them with a wide margin.
    first, last = hist[0], hist[-1]
    assert last['mean_return'] > first['mean_return'] + 10.0
    assert last['coverage'] > first['coverage'] + 0.2
