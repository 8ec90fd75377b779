"""GPU: PPO's diagonal-Gaussian head (RLlib's DiagGaussian, a learned log-std): the act kernel's DIAG instantiations
(policy_act_kernel<MO, MX, false, true>, csrc/paintrl_policy.cuh) and the learner's kLossPpoDiag stage
(ppo_grad_kernel<MO, MX, 3>, csrc/paintrl_learn.cuh), at every <MO, MX> cap.

- act kernel: samples equal a NumPy replay of the counter-based draws, standardised samples pass a KS test against
  N(0, 1) at several sigma, logp is within its FP32 bound, logits / value equal the learner's forward bit for bit;
- learner: the first minibatch after a collection has ratios of exactly 1 (clip fraction 0, KL 0); per-sample stage
  checks against FP64 (learner_stages.py, diag_gaussian_stages.py) with each loss coefficient alone and together and
  the branch coverage of test_gpu_learner_stages.py; a minibatch gradient equals the sum of its one-sample gradients;
  the gradient agrees with torch autograd on RLlib's formulas;
- end to end: two short Trainer runs with continuous-2 actions on the door are identical, and the train script writes a
  checkpoint that load_policy drives."""
import ctypes
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import diag_gaussian_stages as dg
import learner_stages as ls
from test_gpu_learner_stages import COEFFS, MARGIN, _caps, _check, _one_sample_grads, _ppo_rows, _sum_check
from test_gpu_policy import _uniform

pytestmark = pytest.mark.gpu

# (obs_dim, A), n_out = 2A: all four <MO, MX> caps
SHAPES = [(1, 1), (6, 2), (16, 2), (9, 2), (6, 7), (32, 7)]
ROWS = 64
MAX_MB = 2048
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _policy(obs_dim, A, device, seed=0):
    from paintrl_b200.rollout import MlpPolicy
    return MlpPolicy(obs_dim, A, device=device, seed=seed, discrete=False, dist='diag_gaussian')


def _learner(obs_dim, A, cf, params, device):
    from paintrl_b200 import ppo
    L = ppo.PPOLearner(_policy(obs_dim, A, device),
                       ppo.PPOConfig(minibatch_size=MAX_MB, clip_param=cf.clip, vf_clip_param=cf.vf_clip, vf_loss_coeff=cf.vf_coeff,
                                     entropy_coeff=cf.ent_coeff))
    L.params.copy_(params)
    return L


def _native(params, obs_dim, n_out, capacity, device, seed=1):
    from paintrl_b200.rollout import NativePolicy
    P = ls.split_flat(params.cpu().numpy(), obs_dim, n_out)
    weights = [torch.as_tensor(np.ascontiguousarray(P[k])) for k in ('w1', 'b1', 'w2', 'b2', 'w3', 'b3')]
    return NativePolicy(obs_dim, n_out, False, weights, capacity, device, seed=seed)


def _act(pol, obs, A):
    B = obs.shape[0]
    d = obs.device
    actions = torch.zeros(B, A, dtype=torch.float64, device=d)
    logp, value = torch.zeros(B, device=d), torch.zeros(B, device=d)
    logits = torch.zeros(B, 2 * A + 1, device=d)
    pol.act_diag_gaussian_into(obs, actions, logp, value, logits=logits)
    return actions, logp, value, logits


def _params(obs_dim, n_out, log_std_bias=0.0):
    """learner_stages.make_params with the log-std columns' bias moved by log_std_bias."""
    p = ls.make_params(obs_dim, n_out, seed=obs_dim + n_out)
    ls.split_flat(p, obs_dim, n_out)['b3'][n_out // 2:n_out] += np.float32(log_std_bias)
    return p


# ---- the act kernel ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('obs_dim,A', SHAPES)
def test_act_kernel_samples(cuda_device, obs_dim, A):
    from scipy import stats as sps
    n_out, B = 2 * A, 4096
    env = np.arange(B)
    obs = torch.rand(B, obs_dim, generator=torch.Generator(device=cuda_device).manual_seed(7), device=cuda_device, dtype=torch.float64)
    ratios, pvals = {}, []
    for bias in (-2.0, 0.0, 1.0):                      # several sigma: e^-2 .. e^1 around the head's own spread
        params = torch.as_tensor(_params(obs_dim, n_out, bias), device=cuda_device)
        pol = _native(params, obs_dim, n_out, B, cuda_device, seed=9)
        L = _learner(obs_dim, A, COEFFS, params, cuda_device)
        ref = L.forward(obs, torch.arange(B, dtype=torch.int32, device=cuda_device))
        for draw in range(2):
            actions, logp, value, logits = _act(pol, obs, A)
            assert torch.equal(logits, ref) and torch.equal(value, ref[:, n_out]), (bias, draw)
            a, lg = actions.cpu().numpy(), logits.cpu().numpy()
            assert np.array_equal(a, ls.f32(a).astype(np.float64))                  # FP32 values
            # the replay: z from the counter-based draws k = 2o, 2o + 1 of this launch's counter, a = fl(fl(sigma z) + mu)
            z = np.stack([np.sqrt(-2 * np.log(_uniform(9, env, draw, 2 * o))) * np.cos(2 * np.pi * _uniform(9, env, draw, 2 * o + 1))
                          for o in range(A)], axis=1)
            sig = np.exp(lg[:, A:n_out].astype(np.float64))
            want = lg[:, :A].astype(np.float64) + sig * z
            assert np.abs(a - want).max() <= 2e-3 * sig.max() + 1e-5, np.abs(a - want).max()
            zk = dg.standardised(lg, a, n_out)
            assert np.abs(zk - z).max() < 2e-3
            ratios['logp'] = max(ratios.get('logp', 0), ls.ratio(logp.cpu().numpy(), dg.logp_reference(lg, a, n_out)))
            pvals += [sps.kstest(zk[:, o], 'norm').pvalue for o in range(A)]
        # the bootstrap call leaves the counters alone; the act call after it draws with the next counter
        pol.act_into(obs, None, None, value, sample=False)
        actions, _, _, _ = _act(pol, obs, A)
        z2 = np.sqrt(-2 * np.log(_uniform(9, env, 2, 0))) * np.cos(2 * np.pi * _uniform(9, env, 2, 1))
        assert np.abs(dg.standardised(lg, actions.cpu().numpy(), n_out)[:, 0] - z2).max() < 2e-3
        pol.close()
        L.close()
    print('[diag act] obs %d A %d, policy_act_kernel<%d, %d, false, true>: logp ratio %.3g, lowest KS p-value %.3g'
          % ((obs_dim, A) + _caps(obs_dim, n_out) + (ratios['logp'], min(pvals))))
    assert ratios['logp'] <= 1.0
    # 6 A KS tests (2 draws x 3 sigma) per shape: each at 1e-4
    assert min(pvals) > 1e-4, pvals


@pytest.mark.parametrize('obs_dim,A', SHAPES)
def test_first_minibatch_ratio_is_exactly_one(cuda_device, obs_dim, A):
    n_out, B = 2 * A, 1024                  # a power of two: the mean of 1024 ratios of 1 is 1 exactly
    params = torch.as_tensor(_params(obs_dim, n_out), device=cuda_device)
    obs = torch.rand(B, obs_dim, generator=torch.Generator(device=cuda_device).manual_seed(3), device=cuda_device, dtype=torch.float64)
    pol = _native(params, obs_dim, n_out, B, cuda_device)
    actions, logp, value, logits = _act(pol, obs, A)
    pol.close()
    L = _learner(obs_dim, A, COEFFS, params, cuda_device)
    g = torch.Generator(device=cuda_device).manual_seed(4)
    rows = {'obs': obs, 'actions': actions, 'logp': logp, 'value': value, 'logits': logits,
            'adv': torch.randn(B, generator=g, device=cuda_device), 'vtarg': value + torch.randn(B, generator=g, device=cuda_device)}
    grad, stats = torch.zeros_like(L.params), torch.zeros(8, device=cuda_device)
    for idx in (torch.randperm(B, generator=g, device=cuda_device).to(torch.int32), torch.arange(1, dtype=torch.int32, device=cuda_device)):
        L.grad_into(rows, idx, COEFFS.kl_coeff, grad, stats)
        s = stats.cpu().numpy()
        assert s[5] == 1.0 and s[4] == 0.0 and s[2] == 0.0, s
        ent = dg.entropy64(logits[idx.long()].cpu().numpy(), n_out).mean()
        assert abs(s[3] - ent) <= 1e-4 * max(1.0, abs(ent)), (s[3], ent)
    L.close()


# ---- per-sample stages --------------------------------------------------------------------------------------------
@pytest.mark.parametrize('obs_dim,A', SHAPES)
def test_diag_sample_stages(cuda_device, obs_dim, A):
    n_out = 2 * A
    params = torch.as_tensor(_params(obs_dim, n_out), device=cuda_device)
    obs = torch.rand(ROWS, obs_dim, generator=torch.Generator(device=cuda_device).manual_seed(1), device=cuda_device, dtype=torch.float64)
    x32 = obs.float().cpu().numpy()
    n_params = ls.num_params(obs_dim, n_out)
    L = _learner(obs_dim, A, COEFFS, params, cuda_device)
    out = L.forward(obs, torch.arange(ROWS, dtype=torch.int32, device=cuda_device)).cpu().numpy()
    L.close()
    inp = dg.diag_rows(out, n_out, COEFFS, seed=obs_dim)
    zero_adv = dict(inp, adv=np.zeros_like(inp['adv']))
    runs = [('surrogate', COEFFS.only('surrogate'), inp), ('kl', COEFFS.only('kl'), zero_adv),
            ('entropy', COEFFS.only('entropy'), zero_adv), ('value', COEFFS.only('value'), zero_adv), ('full', COEFFS, inp)]
    worst, refs = {}, {}
    for name, cf, rin in runs:
        L = _learner(obs_dim, A, cf, params, cuda_device)
        rows = _ppo_rows(obs, rin, cuda_device)
        G, S = _one_sample_grads(lambda i, gr, st: L.grad_into(rows, i, cf.kl_coeff, gr, st), ROWS, n_params, cuda_device)
        G, S = G.cpu().numpy(), S.cpu().numpy()
        L.close()
        stages, st = ls.check_sample_stages(params.cpu().numpy(), obs_dim, n_out, x32, G, out)
        dout = ls.split_flat(G, obs_dim, n_out)['b3']
        loss, ref, branch = dg.check_diag_loss(out, dout, S[:, :6], rin, cf, n_out)
        for k, v in dict(stages, **loss).items():
            worst[k] = max(worst.get(k, 0), v)
        refs[name] = (ref, dout)
        if name == 'full':
            assert st['live'].all()
            br = ls.ppo_branches(branch, COEFFS)
            assert br['margin'] >= MARGIN, br['margin']
            for cat, sign in ls.PPO_RATIO_CATS:
                assert ((br['ratio'] == cat) & (br['adv_pos'] == (sign > 0))).sum() >= 5, (cat, sign)
            for cat in ls.PPO_VALUE_CATS:
                assert (br['value'] == cat).sum() >= 10, cat
            assert (S[:, 4] == (br['ratio'] != 'inside')).all()
    full_ref, full_dout = refs['full']
    iso = sum(refs[k][0].v for k in ('surrogate', 'kl', 'entropy', 'value'))
    worst['sum_of_terms'] = ls.ratio(full_dout, ls.Bounded(iso, full_ref.e))
    mo, mx = _caps(obs_dim, n_out)
    print('[diag stages] obs %d A %d, ppo_grad_kernel<%d, %d, kLossPpoDiag>: %s'
          % (obs_dim, A, mo, mx, ', '.join('%s %s' % (k, v if k == 'exact' else '%.3g' % v) for k, v in sorted(worst.items()))))
    _check(worst)


def _diag_grad_fn(L, rows, kl):
    from paintrl_b200 import _capi

    def fn(idx, grad, stats, n=None):
        _capi.check(L._lib.paintrl_ppo_grad_diag_gaussian(
            L._h, _ptr(L.params), _ptr(idx), idx.numel() if n is None else n, _ptr(rows['obs']), _ptr(rows['actions']),
            _ptr(rows['logp']), _ptr(rows['value']), _ptr(rows['logits']), _ptr(rows['adv']), _ptr(rows['vtarg']), float(kl),
            _ptr(grad), _ptr(stats), L._stream()))
    return fn


@pytest.mark.parametrize('obs_dim,A', SHAPES)
def test_minibatch_is_the_sum_of_samples(cuda_device, obs_dim, A):
    from test_gpu_learner_stages import FAR, POOL
    n_out = 2 * A
    rng = np.random.default_rng(obs_dim * 100 + A)
    params = torch.as_tensor(_params(obs_dim, n_out), device=cuda_device)
    obs = torch.rand(POOL, obs_dim, generator=torch.Generator(device=cuda_device).manual_seed(4), device=cuda_device, dtype=torch.float64)
    x_pool = obs.float().cpu().numpy()
    L = _learner(obs_dim, A, COEFFS, params, cuda_device)
    out = L.forward(obs, torch.arange(POOL, dtype=torch.int32, device=cuda_device)).cpu().numpy()
    inp = dg.diag_rows(out, n_out, COEFFS, seed=obs_dim)
    inp['adv'][POOL - FAR:] = 1e3
    fn = _diag_grad_fn(L, _ppo_rows(obs, inp, cuda_device), COEFFS.kl_coeff)
    G, S = _one_sample_grads(fn, POOL - FAR, ls.num_params(obs_dim, n_out), cuda_device)
    _, st = ls.check_sample_stages(params.cpu().numpy(), obs_dim, n_out, x_pool[:POOL - FAR], G.cpu().numpy(), out[:POOL - FAR])
    r = _sum_check(obs_dim, n_out, params, x_pool[:POOL - FAR], G, S, st, fn, 6, rng, cuda_device)
    L.close()
    print('[diag lanes] obs %d A %d: %s' % (obs_dim, A, ', '.join('%s %.3g' % kv for kv in sorted(r.items()))))
    _check({k: v for k, v in r.items() if not k.endswith('exact')})


# ---- autograd ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('obs_dim,A', [(6, 2), (16, 2), (32, 7)])
def test_gradient_matches_autograd(cuda_device, obs_dim, A):
    """RLlib's DiagGaussian loss in torch autograd, layer-2 operands rounded to BF16 straight-through, FP32 elsewhere."""
    from paintrl_b200 import ppo
    from test_gpu_ppo import GRAD_COS, GRAD_RTOL, _errors, _split
    n_out, n_rows, n = 2 * A, 1500, 1000
    pol = _policy(obs_dim, A, cuda_device, seed=5)
    for w in pol.weights():
        if w.dim() == 1:
            w.copy_(torch.linspace(-0.3, 0.3, w.numel(), device=cuda_device))
    pol.head_w.mul_(5.0)
    assert pol.enable_native(n_rows)
    g = torch.Generator(device=cuda_device).manual_seed(obs_dim + A)
    obs = torch.rand(n_rows, obs_dim, generator=g, device=cuda_device, dtype=torch.float64)
    actions, logp, value, logits = _act(pol.native, obs, A)
    rows = {'obs': obs, 'actions': actions, 'logp': logp, 'value': value, 'logits': logits,
            'adv': torch.randn(n_rows, generator=g, device=cuda_device), 'vtarg': value + 0.5 * torch.randn(n_rows, generator=g, device=cuda_device)}
    params = ppo.flat_params(pol)
    for t in _split(params, obs_dim, n_out):
        t.add_(0.2 * t.std() * torch.randn(t.shape, generator=g, device=cuda_device))
    idx = torch.randperm(n_rows, generator=g, device=cuda_device)[:n].to(torch.int32)
    i = idx.long()
    a = actions[i].float()
    logp_of = lambda mu, log_std: (-0.5 * ((a - mu) / torch.exp(log_std)) ** 2 - log_std).sum(1) - 0.5 * A * math.log(2 * math.pi)
    # the ratio clip at the median |r - 1| of the perturbed parameters, so that about half of the rows are clipped
    with torch.no_grad():
        w1, b1, w2, b2, w3, b3 = _split(params, obs_dim, n_out)
        o = torch.tanh(torch.tanh(obs[i].float() @ w1 + b1) @ w2 + b2) @ w3 + b3
        clip = float((torch.exp(logp_of(o[:, :A], o[:, A:n_out]) - logp[i]) - 1).abs().median())
    cfg = ppo.PPOConfig(minibatch_size=1024, clip_param=clip, vf_clip_param=0.5, entropy_coeff=0.01)
    learner = ppo.PPOLearner(pol, cfg)
    learner.params.copy_(params)
    grad, stats = torch.zeros_like(learner.params), torch.zeros(8, device=cuda_device)
    learner.grad_into(rows, idx, 0.2, grad, stats)
    torch.backends.cuda.matmul.allow_tf32 = False
    p = learner.params.detach().clone().requires_grad_(True)
    w1, b1, w2, b2, w3, b3 = _split(p, obs_dim, n_out)
    bf = lambda t: t + (t.to(torch.bfloat16).float() - t).detach()
    h2 = torch.tanh(bf(torch.tanh(obs[i].float() @ w1 + b1)) @ bf(w2) + b2)
    out = h2 @ w3 + b3
    mu, log_std, v = out[:, :A], out[:, A:n_out], out[:, n_out]
    old = logits[i]
    muo, lso = old[:, :A], old[:, A:n_out]
    lp = logp_of(mu, log_std)
    kl = (log_std - lso + (torch.exp(2 * lso) + (muo - mu) ** 2) / (2 * torch.exp(2 * log_std)) - 0.5).sum(1)
    ent = (log_std + 0.5 + 0.5 * math.log(2 * math.pi)).sum(1)
    r = torch.exp(lp - logp[i])
    Adv, R, vold = rows['adv'][i], rows['vtarg'][i], value[i]
    surr = torch.min(Adv * r, Adv * torch.clamp(r, 1 - cfg.clip_param, 1 + cfg.clip_param))
    vf = torch.max((v - R) ** 2, (vold + torch.clamp(v - vold, -cfg.vf_clip_param, cfg.vf_clip_param) - R) ** 2)
    (-surr + 0.2 * kl + cfg.vf_loss_coeff * vf - cfg.entropy_coeff * ent).mean().backward()
    frac_clip = float(((r - 1).abs() > cfg.clip_param).float().mean())
    kl, ent = kl.detach(), ent.detach()
    assert 0.05 < frac_clip < 0.95, frac_clip
    report = {name: _errors(x, y) for name, x, y in zip(('w1', 'b1', 'w2', 'b2', 'w3', 'b3'), _split(grad, obs_dim, n_out), _split(p.grad, obs_dim, n_out))}
    print('[diag autograd] obs %d A %d (rel Frobenius, cosine): %s' % (obs_dim, A, report))
    for name, (rel, cos) in report.items():
        assert rel <= GRAD_RTOL and cos >= GRAD_COS, (name, rel, cos)
    s = stats.cpu().numpy()
    assert abs(s[4] - frac_clip) < 0.01
    assert abs(s[2] - float(kl.mean())) <= 1e-3 * max(1.0, abs(float(kl.mean())))
    assert abs(s[3] - float(ent.mean())) <= 1e-3 * max(1.0, abs(float(ent.mean())))
    learner.close()
    pol.native.close()


# ---- argument checks ----------------------------------------------------------------------------------------------
def test_entry_points_refuse_the_wrong_handle(cuda_device):
    from paintrl_b200 import _capi, ppo
    from paintrl_b200.rollout import MlpPolicy
    lib = _capi.lib()
    F = ctypes.c_void_p(16)
    obs = torch.zeros(4, 6, dtype=torch.float64, device=cuda_device)
    for discrete, n_out, msg in ((True, 4, b'continuous'), (False, 3, b'even n_out')):
        pol = MlpPolicy(6, n_out, device=cuda_device, discrete=discrete)
        assert pol.enable_native(4)
        assert lib.paintrl_policy_act_diag_gaussian(pol.native._h, _ptr(obs), 4, F, F, F, None, None) == -1
        assert msg in lib.paintrl_last_error(), lib.paintrl_last_error()
        with pytest.raises(ValueError):
            pol.native.act_diag_gaussian_into(obs, None, None, None)
        L = ppo.PPOLearner(pol, ppo.PPOConfig(minibatch_size=128))
        assert lib.paintrl_ppo_grad_diag_gaussian(L._h, F, F, 4, F, F, F, F, F, F, F, 0.2, F, F, None) == -1
        assert msg in lib.paintrl_last_error(), lib.paintrl_last_error()
        L.close()
        pol.native.close()
    pol = _policy(6, 2, cuda_device)
    assert pol.enable_native(4)
    h = pol.native._h
    for args in ((h, None, 4, F, F, F, None, None), (h, _ptr(obs), 4, None, F, F, None, None), (h, _ptr(obs), 4, F, None, F, None, None),
                 (h, _ptr(obs), 4, F, F, None, None, None)):
        assert lib.paintrl_policy_act_diag_gaussian(*args) == -1 and b'null' in lib.paintrl_last_error()
    assert lib.paintrl_policy_act_diag_gaussian(h, _ptr(obs), 5, F, F, F, None, None) == -1
    assert b'capacity' in lib.paintrl_last_error()
    L = ppo.PPOLearner(pol, ppo.PPOConfig(minibatch_size=128))
    assert lib.paintrl_ppo_grad_diag_gaussian(L._h, F, F, 4, F, None, F, F, F, F, F, 0.2, F, F, None) == -1
    assert b'null' in lib.paintrl_last_error()
    assert lib.paintrl_ppo_grad_diag_gaussian(L._h, F, F, 0, F, F, F, F, F, F, F, 0.2, F, F, None) == -1
    assert lib.paintrl_ppo_grad_diag_gaussian(L._h, F, F, 4, F, F, F, F, F, F, F, -1.0, F, F, None) == -1
    L.close()
    pol.native.close()


# ---- end to end --------------------------------------------------------------------------------------------------
def test_rollout_worker_refuses_mismatched_action_dims(cuda_device):
    from paintrl_b200.rollout import RolloutWorker
    from paintrl_b200.train import make_env
    env = make_env(0, 128, 0, cuda_device, dict(action_mode='continuous', action_shape=2))
    with pytest.raises(ValueError, match='does not fit'):
        RolloutWorker(env, _policy(env.obs_dim, 1, cuda_device), fragment_length=4)
    env.close()
    env = make_env(0, 128, 0, cuda_device)
    with pytest.raises(ValueError, match='does not fit'):
        RolloutWorker(env, _policy(env.obs_dim, 1, cuda_device), fragment_length=4)
    env.close()


def _trainer_run(device):
    from paintrl_b200 import ppo
    from paintrl_b200.train import Trainer
    tr = Trainer(0, 512, 20, seed=3, device=device, config=ppo.PPOConfig(seed=3, lr=1e-3, minibatch_size=1024, num_sgd_iter=4),
                 spaces=dict(action_mode='continuous', action_shape=2))
    assert tr.policy.dist == 'diag_gaussian' and tr.policy.native is not None
    lines = []
    for _ in range(3):
        r = tr.iteration()
        lines.append({k: v for k, v in r.items() if not k.endswith('_s')})
    params = tr.learner.params.clone()
    frag = tr.worker.frag
    assert tuple(frag.actions.shape) == (20, 512, 2)
    tr.close()
    return lines, params


def test_trainer_is_reproducible(cuda_device):
    a, pa = _trainer_run(cuda_device)
    b, pb = _trainer_run(cuda_device)
    assert a == b
    assert torch.equal(pa, pb)
    assert a[0]['learner']['mean_ratio'] > 0 and all(math.isfinite(x['learner']['entropy']) for x in a)


def test_train_script_and_load_policy(cuda_device, tmp_path):
    from paintrl_b200 import train
    from paintrl_b200.batched_env import BatchedPaintEnv
    from paintrl_b200.config import EnvConfig
    ck = str(tmp_path / 'cont.pt')
    res = subprocess.run([sys.executable, '-m', 'paintrl_b200.train', '--action-mode', 'continuous', '--action-shape', '2', '--iters', '2',
                          '--envs', '256', '--fragment', '20', '--minibatch', '1024', '--sgd-iters', '2', '--checkpoint', ck],
                         cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [json.loads(x) for x in res.stdout.splitlines() if x.startswith('{')]
    assert len(lines) == 2 and lines[-1]['env_steps'] == 2 * 256 * 20
    pol = train.load_policy(ck, cuda_device)
    assert (pol.dist, pol.action_dim, pol.n_out) == ('diag_gaussian', 2, 4)
    sp = train.checkpoint_spaces(torch.load(ck, weights_only=False))
    assert (sp['action_mode'], sp['action_shape']) == ('continuous', 2)
    # drive: the mean action, in the checkpoint's spaces
    cfg = EnvConfig(dict(train.C2_SETTINGS), action_mode=sp['action_mode'], action_shape=sp['action_shape'], obs_mode=sp['obs_mode'],
                    obs_grad=sp['obs_grad'], auto_reset=False)
    env = BatchedPaintEnv(4, cfg, device=cuda_device)
    obs = env.reset(np.arange(4, dtype=np.int32) % env.n_starts)
    for _ in range(5):
        out, _ = pol.forward(obs)
        obs, actual, done, info = env.step(out[:, :pol.action_dim].double().contiguous())
        assert torch.isfinite(obs).all() and torch.isfinite(actual).all()
    env.close()
