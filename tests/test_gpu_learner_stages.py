"""GPU: the learner kernel (ppo_grad_kernel, csrc/paintrl_learn.cuh) stage by stage, and the act kernel's forward pass
(policy_act_kernel, csrc/paintrl_policy.cuh) against it, at every <MO, MX> instantiation and on both sides of each cap.

- per sample: one-sample gradients expose every intermediate (learner_stages.py); each stage is checked against an
  FP64 reference built from the kernel's own values of the stage before, PPO with discrete and continuous heads and
  each loss coefficient alone, DQN with the online-argmax tie;
- lanes and tiles: the forward of a permuted index list with duplicates equals the one-sample forwards bit for bit; the
  gradient of a minibatch equals the sum of its one-sample gradients over n to an FP32 reordering bound (exact scaling
  for n a power of two, a BF16 half-ulp term for ragged n); index entries past n are not read;
- the act kernel's logits and value equal the learner's forward bit for bit, sampling and epsilon-greedy.

Each check prints its worst error-to-bound ratio (<= 1 passes) per shape."""
import ctypes

import numpy as np
import pytest
import torch

import learner_stages as ls

pytestmark = pytest.mark.gpu

# (obs_dim, n_out): every <MO, MX> cap and both sides of each boundary (obs_dim 8 | 9, n_out + 1 = 8 | 9), and n_out 1
SHAPES = [(1, 1), (6, 4), (8, 7), (8, 8), (9, 7), (32, 15)]
ROWS = 64                      # per-sample stage rows
POOL, FAR = 300, 50            # lane-test rows; the last FAR have huge advantages / rewards and are reached only past n
MAX_MB = 2048
COEFFS = ls.PpoCoeffs(clip=0.2, vf_clip=0.5, vf_coeff=0.5, ent_coeff=0.01, kl_coeff=0.2)
GAMMA = 0.9
MARGIN = 0.1                   # every row at least 10 % (relative) away from each branch boundary
FWD_NS = (1, 63, 64, 127, 128, 129, 255, 256, 1000, MAX_MB)
POW2_NS, RAGGED_NS = (64, 128, 256, 1024), (129, 1000)


def _caps(obs_dim, n_out):
    """with_caps of paintrl_capi.cu."""
    return (8 if obs_dim <= 8 else 32), (8 if n_out + 1 <= 8 else 16)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _report(what, losses, obs_dim, n_out, ratios):
    """One log line: the instantiations exercised and each check's worst error-to-bound ratio (exact checks: the count
    of broken identities)."""
    mo, mx = _caps(obs_dim, n_out)
    kernels = ' '.join('ppo_grad_kernel<%d, %d, %s>' % (mo, mx, loss) for loss in losses)
    body = ', '.join('%s %s' % (k, v if isinstance(v, (int, np.integer)) else '%.3g' % v) for k, v in sorted(ratios.items()))
    print('[%s] obs %d n_out %d, %s: %s' % (what, obs_dim, n_out, kernels, body))


def _check(ratios):
    bad = {k: v for k, v in ratios.items() if not (v == 0 if k == 'exact' else v <= 1.0)}
    assert not bad, bad


def _policy(obs_dim, n_out, discrete, device):
    from paintrl_b200.rollout import MlpPolicy
    return MlpPolicy(obs_dim, n_out, device=device, seed=0, discrete=discrete)


def _ppo(obs_dim, n_out, discrete, cf, params, device):
    from paintrl_b200 import ppo
    L = ppo.PPOLearner(_policy(obs_dim, n_out, discrete, device),
                       ppo.PPOConfig(minibatch_size=MAX_MB, clip_param=cf.clip, vf_clip_param=cf.vf_clip, vf_loss_coeff=cf.vf_coeff,
                                     entropy_coeff=cf.ent_coeff))
    L.params.copy_(params)
    return L


def _dqn(obs_dim, n_out, params, device):
    from paintrl_b200 import dqn
    L = dqn.DQNLearner(_policy(obs_dim, n_out, True, device), dqn.DQNConfig(minibatch_size=MAX_MB, gamma=GAMMA, replay_capacity=128))
    L.params.copy_(params)
    return L


def _forward(L, params, obs, idx):
    """paintrl_ppo_forward: the kernel's head outputs for rows idx of obs."""
    out = torch.empty(idx.numel(), L.n_out + 1, device=obs.device)
    from paintrl_b200 import _capi
    _capi.check(L._lib.paintrl_ppo_forward(L._h, _ptr(params), _ptr(idx), idx.numel(), _ptr(obs), _ptr(out), L._stream()))
    return out


def _ppo_rows(obs, inp, device):
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=device)
    return {'obs': obs, 'actions': t(inp['actions'], torch.int64 if inp['actions'].ndim == 1 else torch.float64),
            'logp': t(inp['logp_old'], torch.float32), 'value': t(inp['value_old'], torch.float32),
            'logits': t(inp['logits_old'], torch.float32), 'adv': t(inp['adv'], torch.float32), 'vtarg': t(inp['vtarg'], torch.float32)}


class _Buf(object):
    def __init__(self, obs, next_obs, inp, device):
        self.obs, self.next_obs = obs, next_obs
        self.actions = torch.as_tensor(inp['actions'], dtype=torch.int64, device=device)
        self.reward = torch.as_tensor(inp['reward'], dtype=torch.float32, device=device)
        self.done = torch.as_tensor(inp['done'], dtype=torch.uint8, device=device)


def _one_sample_grads(grad_fn, n_rows, n_params, device):
    """grad_fn(idx, grad, stats) for each row alone (n = 1) into [n_rows, n_params] and [n_rows, 8], read back once."""
    idx = torch.arange(n_rows, dtype=torch.int32, device=device)
    G = torch.zeros(n_rows, n_params, device=device)
    S = torch.zeros(n_rows, 8, device=device)
    for j in range(n_rows):
        grad_fn(idx[j:j + 1], G[j], S[j])
    return G, S


def _setup(obs_dim, n_out, n_rows, device, seed):
    params = torch.as_tensor(ls.make_params(obs_dim, n_out, seed=obs_dim + n_out), device=device)
    g = torch.Generator(device=device).manual_seed(seed)
    obs = torch.rand(n_rows, obs_dim, generator=g, device=device, dtype=torch.float64)
    return params, obs


# ---- per-sample stages ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('discrete', [True, False])
@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_ppo_sample_stages(cuda_device, obs_dim, n_out, discrete):
    params, obs = _setup(obs_dim, n_out, ROWS, cuda_device, seed=1)
    x32 = obs.float().cpu().numpy()
    n_params = ls.num_params(obs_dim, n_out)
    L = _ppo(obs_dim, n_out, discrete, COEFFS, params, cuda_device)
    out = _forward(L, params, obs, torch.arange(ROWS, dtype=torch.int32, device=cuda_device)).cpu().numpy()
    L.close()
    inp = ls.ppo_rows(out, n_out, discrete, COEFFS, seed=obs_dim)
    zero_adv = dict(inp, adv=np.zeros_like(inp['adv']))
    # each coefficient alone (the surrogate with the others 0, the rest with A = 0), then all of them
    runs = [('surrogate', COEFFS.only('surrogate'), inp), ('kl', COEFFS.only('kl'), zero_adv),
            ('entropy', COEFFS.only('entropy'), zero_adv), ('value', COEFFS.only('value'), zero_adv), ('full', COEFFS, inp)]
    worst, refs = {}, {}
    for name, cf, rin in runs:
        L = _ppo(obs_dim, n_out, discrete, cf, params, cuda_device)
        rows = _ppo_rows(obs, rin, cuda_device)
        G, S = _one_sample_grads(lambda i, gr, st: L.grad_into(rows, i, cf.kl_coeff, gr, st), ROWS, n_params, cuda_device)
        G, S = G.cpu().numpy(), S.cpu().numpy()
        L.close()
        stages, st = ls.check_sample_stages(params.cpu().numpy(), obs_dim, n_out, x32, G, out)
        dout = ls.split_flat(G, obs_dim, n_out)['b3']
        loss, ref, branch = ls.check_ppo_loss(out, dout, S[:, :6], rin, cf, discrete, n_out)
        for k, v in dict(stages, **loss).items():
            worst[k] = max(worst.get(k, 0), v)
        refs[name] = (ref, dout)
        if name == 'full':
            assert st['live'].sum() >= ROWS // 2, st['live'].sum()
            br = ls.ppo_branches(branch, COEFFS)
            assert br['margin'] >= MARGIN, br['margin']
            for cat, sign in ls.PPO_RATIO_CATS:
                assert ((br['ratio'] == cat) & (br['adv_pos'] == (sign > 0))).sum() >= 5, (cat, sign)
            for cat in ls.PPO_VALUE_CATS:
                assert (br['value'] == cat).sum() >= 10, cat
            assert (S[:, 4] == (br['ratio'] != 'inside')).all()          # the clip fraction of each row
            if discrete:
                assert set(inp['actions'].tolist()) == set(range(n_out))
    # the full run against the FP64 sum of the isolated references
    full_ref, full_dout = refs['full']
    iso = sum(refs[k][0].v for k in ('surrogate', 'kl', 'entropy', 'value'))
    worst['sum_of_terms'] = ls.ratio(full_dout, ls.Bounded(iso, full_ref.e))
    _report('ppo %s' % ('discrete' if discrete else 'continuous'), ['kLossPpo'], obs_dim, n_out, worst)
    _check(worst)


@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_dqn_sample_stages(cuda_device, obs_dim, n_out):
    params, obs = _setup(obs_dim, n_out, ROWS, cuda_device, seed=2)
    if n_out >= 3:
        params = torch.as_tensor(ls.make_tie(params.cpu().numpy(), obs_dim, n_out), device=cuda_device)
    target = torch.as_tensor(ls.make_params(obs_dim, n_out, seed=100 + obs_dim), device=cuda_device)
    g = torch.Generator(device=cuda_device).manual_seed(3)
    next_obs = torch.rand(ROWS, obs_dim, generator=g, device=cuda_device, dtype=torch.float64)
    x32 = obs.float().cpu().numpy()
    F = _ppo(obs_dim, n_out, True, COEFFS, params, cuda_device)           # paintrl_ppo_forward needs a PPO handle
    idx = torch.arange(ROWS, dtype=torch.int32, device=cuda_device)
    out, head_on, head_tn = [_forward(F, p, o, idx).cpu().numpy() for p, o in ((params, obs), (params, next_obs), (target, next_obs))]
    F.close()
    L = _dqn(obs_dim, n_out, params, cuda_device)
    inp = ls.dqn_rows(out, head_on, head_tn, n_out, GAMMA, seed=obs_dim)
    buf = _Buf(obs, next_obs, inp, cuda_device)
    G, S = _one_sample_grads(lambda i, gr, st: L.grad_into(buf, i, gr, st, target=target), ROWS, ls.num_params(obs_dim, n_out), cuda_device)
    G, S = G.cpu().numpy(), S.cpu().numpy()
    L.close()
    stages, st = ls.check_sample_stages(params.cpu().numpy(), obs_dim, n_out, x32, G, out)
    loss, td, rep = ls.check_dqn_loss(out, head_on, head_tn, ls.split_flat(G, obs_dim, n_out)['b3'], S[:, :4], inp, GAMMA, n_out)
    assert st['live'].all()
    # row coverage: |td| on both sides of 1, done both ways, every action, and the tie on s'
    assert (np.abs(td) < 1).sum() >= 20 and (np.abs(td) > 1).sum() >= 20
    assert np.abs(np.abs(td) - 1).min() >= MARGIN
    assert inp['done'].any() and (inp['done'] == 0).any()
    assert set(inp['actions'].tolist()) == set(range(n_out))
    if n_out >= 3:
        assert np.array_equal(head_on[:, 1], head_on[:, 2]) and (rep['an'] == 1).all()
        qt, _ = ls.q_values32(head_tn, n_out)
        assert (qt[:, 1] != qt[:, 2]).all()                                # the tie rule decides the target
    ratios = dict(stages, **loss)
    _report('dqn', ['kLossDqn'], obs_dim, n_out, ratios)
    _check(ratios)


# ---- lanes and tiles --------------------------------------------------------------------------------------------
def _index_list(n, rng, device, high=POOL - FAR):
    """n rows drawn with replacement from [0, high), so permuted and with duplicates."""
    return torch.as_tensor(rng.integers(0, high, n), dtype=torch.int32, device=device)


def _sum_check(obs_dim, n_out, params, x_pool, G, S, st, grad_fn, nstats, rng, device):
    """The minibatch gradient and statistics against the FP64 sum of the one-sample ones, for every n in POW2_NS and
    RAGGED_NS; and entries past n not read.  Returns name -> worst ratio."""
    P = ls.split_flat(params.cpu().numpy(), obs_dim, n_out)
    n_params = G.shape[1]
    rows = G.shape[0]
    G64 = G.double()
    A64 = G64.abs()
    # per-row magnitudes of the ragged bounds (ls.ragged_factors): M_b2 = (1 - h2^2) sum_o |dout w3|, carried to b1
    # through |bf16(W2)| and to w1 / w2 through |x| / |h1_bf16|
    live = st['live']
    mb2 = np.zeros((rows, ls.H2))
    h1b = np.zeros((rows, ls.H1))
    mb2[live] = (1 - st['h2'].astype(np.float64) ** 2) * (np.abs(st['dout'].astype(np.float64)) @ np.abs(P['w3'].astype(np.float64)).T)
    h1b[live] = np.abs(st['h1b'].astype(np.float64))
    w2b = np.abs(ls.bf16(P['w2']).astype(np.float64))
    dev = lambda a: torch.as_tensor(a, dtype=torch.float64, device=device)
    MB2, MB1, H1B, X = dev(mb2), dev(mb2 @ w2b.T), dev(h1b), dev(np.abs(x_pool.astype(np.float64)))
    rag = ls.ragged_factors(n_out)
    worst = {}
    grad = torch.zeros(n_params, device=device)
    stats = torch.zeros(8, device=device)
    for n in POW2_NS + RAGGED_NS:
        idx = _index_list(n, rng, device)
        grad_fn(idx, grad, stats)
        c = torch.bincount(idx.long(), minlength=rows).double()
        ref = (c @ G64) / n
        mag = (c @ A64) / n
        ctas = (n + 127) // 128
        f = ls.sum_factors(ctas)
        bound = torch.zeros(n_params, dtype=torch.float64, device=device)
        off = 0
        for name, shape in (('w1', (obs_dim, ls.H1)), ('b1', (ls.H1,)), ('w2', (ls.H1, ls.H2)), ('b2', (ls.H2,)),
                            ('w3', (ls.H2, n_out + 1)), ('b3', (n_out + 1,))):
            k = int(np.prod(shape))
            sl = slice(off, off + k)
            bound[sl] = f[name] * mag[sl]
            if n not in POW2_NS:
                if name in ('w3', 'b3'):
                    bound[sl] += rag['dout'] * mag[sl]
                elif name == 'b2':
                    bound[sl] += rag['dz2'] * (c @ MB2) / n
                elif name == 'w2':
                    bound[sl] += (rag['dz2b'] * (H1B.T @ (c[:, None] * MB2)) / n).reshape(-1)
                elif name == 'b1':
                    bound[sl] += rag['dz1'] * (c @ MB1) / n
                else:
                    bound[sl] += (rag['x_dz1'] * (X.T @ (c[:, None] * MB1)) / n).reshape(-1)
            off += k
        err = (grad.double() - ref).abs()
        r = float(torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err == 0, 0.0, float('inf'))).max())
        key = 'grad_pow2' if n in POW2_NS else 'grad_ragged'
        worst[key] = max(worst.get(key, 0), r)
        s_ref = (c @ S.double()[:, :nstats]) / n
        s_bound = ls.gamma(128 + ctas + 2) * (c @ S.double()[:, :nstats].abs()) / n
        s_err = (stats[:nstats].double() - s_ref).abs()
        worst['stats'] = max(worst.get('stats', 0), float(torch.where(s_bound > 0, s_err / s_bound.clamp_min(1e-300),
                                                                      torch.where(s_err == 0, 0.0, float('inf'))).max()))
        if n in RAGGED_NS:
            # entries past n are not read: a buffer whose tail points at valid rows with huge advantages / rewards gives
            # the bits of one whose tail points at ordinary rows
            got = [(grad.clone(), stats.clone())]
            for lo, hi in ((0, POOL - FAR), (POOL - FAR, POOL)):
                buf = torch.cat([idx, torch.as_tensor(rng.integers(lo, hi, MAX_MB - n), dtype=torch.int32, device=device)])
                grad_fn(buf, grad, stats, n)
                got.append((grad.clone(), stats.clone()))
            for g_, s_ in got[1:]:
                assert torch.equal(g_, got[0][0]) and torch.equal(s_, got[0][1]), n
            worst['past_n_exact'] = 0
    return worst


def _ppo_grad_fn(L, rows, kl):
    from paintrl_b200 import _capi

    def fn(idx, grad, stats, n=None):
        _capi.check(L._lib.paintrl_ppo_grad(
            L._h, _ptr(L.params), _ptr(idx), idx.numel() if n is None else n, _ptr(rows['obs']), _ptr(rows['actions']),
            _ptr(rows['logp']), _ptr(rows['value']), _ptr(rows['logits']), _ptr(rows['adv']), _ptr(rows['vtarg']), float(kl),
            _ptr(grad), _ptr(stats), L._stream()))
    return fn


def _dqn_grad_fn(L, buf, target):
    from paintrl_b200 import _capi

    def fn(idx, grad, stats, n=None):
        _capi.check(L._lib.paintrl_dqn_grad(
            L._h, _ptr(L.params), _ptr(target), _ptr(idx), idx.numel() if n is None else n, _ptr(buf.obs), _ptr(buf.actions),
            _ptr(buf.reward), _ptr(buf.next_obs), _ptr(buf.done), _ptr(grad), _ptr(stats), L._stream()))
    return fn


@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_lanes_and_tiles(cuda_device, obs_dim, n_out):
    rng = np.random.default_rng(obs_dim * 100 + n_out)
    params, obs = _setup(obs_dim, n_out, POOL, cuda_device, seed=4)
    n_params = ls.num_params(obs_dim, n_out)
    x_pool = obs.float().cpu().numpy()
    pool = torch.arange(POOL, dtype=torch.int32, device=cuda_device)
    F = _ppo(obs_dim, n_out, True, COEFFS, params, cuda_device)           # paintrl_ppo_forward needs a PPO handle
    # forward: every lane of every CTA, ragged last tiles included, equals the one-sample forward
    single = torch.cat([_forward(F, params, obs, pool[j:j + 1]) for j in range(POOL)])
    for n in FWD_NS:
        idx = _index_list(n, rng, cuda_device, high=POOL)
        assert torch.equal(_forward(F, params, obs, idx), single[idx.long()]), n
    out = single.cpu().numpy()
    ratios = {'forward_exact': 0}
    for mode in ('ppo_discrete', 'ppo_continuous', 'dqn'):
        if mode == 'dqn':
            L = _dqn(obs_dim, n_out, params, cuda_device)
            target = torch.as_tensor(ls.make_params(obs_dim, n_out, seed=100 + obs_dim), device=cuda_device)
            next_obs = torch.rand(POOL, obs_dim, generator=torch.Generator(device=cuda_device).manual_seed(5), device=cuda_device,
                                  dtype=torch.float64)
            heads = [_forward(F, p, next_obs, pool).cpu().numpy() for p in (params, target)]
            inp = ls.dqn_rows(out, heads[0], heads[1], n_out, GAMMA, seed=obs_dim)
            inp['reward'][POOL - FAR:] = 1e3
            fn = _dqn_grad_fn(L, _Buf(obs, next_obs, inp, cuda_device), target)
            nstats = 4
        else:
            discrete = mode == 'ppo_discrete'
            L = _ppo(obs_dim, n_out, discrete, COEFFS, params, cuda_device)
            inp = ls.ppo_rows(out, n_out, discrete, COEFFS, seed=obs_dim)
            inp['adv'][POOL - FAR:] = 1e3
            fn = _ppo_grad_fn(L, _ppo_rows(obs, inp, cuda_device), COEFFS.kl_coeff)
            nstats = 6
        G, S = _one_sample_grads(fn, POOL - FAR, n_params, cuda_device)
        _, st = ls.check_sample_stages(params.cpu().numpy(), obs_dim, n_out, x_pool[:POOL - FAR], G.cpu().numpy(), out[:POOL - FAR])
        r = _sum_check(obs_dim, n_out, params, x_pool[:POOL - FAR], G, S, st, fn, nstats, rng, cuda_device)
        L.close()
        for k, v in r.items():
            ratios['%s_%s' % (mode, k)] = v
    F.close()
    _report('lanes', ['kLossPpo', 'kLossDqn'], obs_dim, n_out, ratios)
    _check({k: v for k, v in ratios.items() if not k.endswith('exact')})


# ---- the act kernel against the learner's forward ----------------------------------------------------------------
@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_act_kernel_equals_learner_forward(cuda_device, obs_dim, n_out):
    from paintrl_b200.rollout import NativePolicy
    params, obs = _setup(obs_dim, n_out, 129, cuda_device, seed=6)
    P = ls.split_flat(params.cpu().numpy(), obs_dim, n_out)
    weights = [torch.as_tensor(np.ascontiguousarray(P[k])) for k in ('w1', 'b1', 'w2', 'b2', 'w3', 'b3')]
    L = _ppo(obs_dim, n_out, True, COEFFS, params, cuda_device)
    names = []
    for discrete in (True, False):
        pol = NativePolicy(obs_dim, n_out, discrete, weights, 129, cuda_device, seed=1)
        for B in (1, 127, 129):
            ref = _forward(L, params, obs, torch.arange(B, dtype=torch.int32, device=cuda_device))
            o = obs[:B].contiguous()
            value = torch.zeros(B, device=cuda_device)
            logits = torch.zeros(B, n_out + 1, device=cuda_device)
            logp = torch.zeros(B, device=cuda_device)
            actions = (torch.zeros(B, dtype=torch.int64, device=cuda_device) if discrete else
                       torch.zeros(B, n_out, dtype=torch.float64, device=cuda_device))
            pol.act_into(o, actions, logp, value, logits=logits)
            assert torch.equal(logits, ref) and torch.equal(value, ref[:, n_out]), (discrete, B)
            if discrete:
                logits.zero_()
                pol.act_epsilon_into(o, actions, value, torch.full((1,), 0.5, device=cuda_device), logits=logits)
                assert torch.equal(value, ref[:, n_out]) and torch.equal(logits, ref), B
        pol.close()
        mo, mx = _caps(obs_dim, n_out)
        names += ['policy_act_kernel<%d, %d, %s>' % (mo, mx, eps) for eps in (('false', 'true') if discrete else ('false',))]
    L.close()
    print('[act parity] obs %d n_out %d: %s bit for bit with the learner forward at batches 1, 127, 129' % (obs_dim, n_out, sorted(set(names))))
