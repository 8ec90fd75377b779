"""The diagonal-Gaussian PPO head without a GPU: the loss-stage checker of diag_gaussian_stages.py accepts a NumPy
restatement of the kernel and rejects each planted bug by the check that names it; the new C entry points, the
trainer's space options and the checkpoints check what they are given."""
import ctypes
import math

import numpy as np
import pytest
import torch

import diag_gaussian_stages as dg
import learner_stages as ls
from test_learner_stages_cpu import _forward, _sample_grads

# (obs_dim, A): every <MO, MX> cap (n_out = 2A, n_out + 1 <= 8 or not; obs_dim <= 8 or not)
SHAPES = [(1, 1), (6, 2), (16, 2), (9, 2), (6, 7), (32, 7)]
ROWS = 64
COEFFS = ls.PpoCoeffs(clip=0.2, vf_clip=0.5, vf_coeff=0.5, ent_coeff=0.01, kl_coeff=0.2)

f64 = lambda a: np.asarray(a, dtype=np.float64)


def _diag_loss(out, inp, cf, n_out, bug=None):
    """The kLossPpoDiag stage in FP64, rounded once to FP32; `bug` plants one mistake."""
    A = n_out // 2
    rows = len(out)
    o, old = f64(out), f64(inp['logits_old'])
    ls_col = A + 1 if bug == 'logstd_column_off' else A
    mu, lsig = o[:, :A], o[:, ls_col:ls_col + A]
    muo, lso = old[:, :A], old[:, A:2 * A]
    if bug == 'actions_stride_n_out':               # row j read at j * n_out, as if the actions had n_out columns
        flat = f64(ls.f32(inp['actions'])).ravel()
        a = np.take(flat, np.arange(rows)[:, None] * n_out + np.arange(A)[None, :], mode='wrap')
    else:
        a = f64(ls.f32(inp['actions']))
    sig, sigo = np.exp(lsig), np.exp(lso)
    u = (a - mu) / sig
    logp = (-0.5 * u * u - lsig).sum(1) - A * ls.LOG_SQRT_2PI
    d = mu - muo
    if bug == 'kl_reversed':                         # KL(new || old)
        q = (sig * sig + d * d) / (sigo * sigo)
        kl = (lso - lsig + 0.5 * q - 0.5).sum(1)
        dkl_mu, dkl_ls = d / (sigo * sigo), 1.0 * (sig * sig) / (sigo * sigo) - 1.0
    else:
        s2o = sigo if bug == 'kl_sigma_not_squared' else sigo * sigo
        q = (s2o + d * d) / (sig * sig)
        kl = (lsig - lso + 0.5 * q - 0.5).sum(1)
        dkl_mu, dkl_ls = d / (sig * sig), 1.0 - q
    ent = (lsig + ls.GAUSS_ENTROPY).sum(1)
    Adv, R, vold = f64(inp['adv']), f64(inp['vtarg']), f64(inp['value_old'])
    r = np.exp(logp - f64(inp['logp_old']))
    rc = np.clip(r, 1 - cf.clip, 1 + cf.clip)
    s1, s2 = Adv * r, Adv * rc
    g_logp = np.where(s1 <= s2, -Adv * r, 0.0)[:, None]
    v = o[:, n_out]
    vf1 = (v - R) ** 2
    dv = v - vold
    vcl = vold + np.clip(dv, -cf.vf_clip, cf.vf_clip)
    vf2 = (vcl - R) ** 2
    g_v = np.where(vf1 >= vf2, 2 * (v - R), np.where(np.abs(dv) <= cf.vf_clip, 2 * (vcl - R), 0.0))
    dmu = g_logp * (u if bug == 'u_not_over_sigma' else u / sig) + cf.kl_coeff * dkl_mu
    dls = g_logp * (u * u if bug == 'dlogp_dlogstd_no_minus_one' else u * u - 1.0) + cf.kl_coeff * dkl_ls - cf.ent_coeff
    dout = np.concatenate([dmu, dls, (cf.vf_coeff * g_v)[:, None]], axis=1)
    stats = np.stack([-np.minimum(s1, s2), np.maximum(vf1, vf2), kl, ent, (np.abs(r - 1) > cf.clip).astype(np.float64), r], axis=1)
    return ls.f32(dout), ls.f32(stats), ls.f32(logp)


def _run(obs_dim, A, bug=None, seed=0, cf=COEFFS):
    n_out = 2 * A
    rng = np.random.default_rng(seed)
    x32 = ls.f32(rng.uniform(0, 1, (ROWS, obs_dim)))
    params = ls.make_params(obs_dim, n_out, seed=obs_dim + n_out)
    fw = _forward(params, obs_dim, n_out, x32)
    out = fw['out']
    inp = dg.diag_rows(out, n_out, cf, seed)
    dout, stats, logp = _diag_loss(out, inp, cf, n_out, bug)
    r, _, branch = dg.check_diag_loss(out, dout, stats, inp, cf, n_out)
    r['logp'] = ls.ratio(logp, dg.logp_reference(out, inp['actions'], n_out))
    grads = _sample_grads(params, obs_dim, n_out, x32, fw, dout)
    stages, _ = ls.check_sample_stages(params, obs_dim, n_out, x32, grads, out)
    return dict(stages, **r), branch


@pytest.mark.parametrize('obs_dim,A', SHAPES)
def test_checker_accepts_the_restatement(obs_dim, A):
    r, branch = _run(obs_dim, A)
    assert r.pop('exact') == 0
    assert all(v <= 1.0 for v in r.values()), r
    br = ls.ppo_branches(branch, COEFFS)
    assert br['margin'] > 0.1, br['margin']
    for cat, sign in ls.PPO_RATIO_CATS:
        assert ((br['ratio'] == cat) & (br['adv_pos'] == (sign > 0))).sum() >= 5, (cat, sign)
    for cat in ls.PPO_VALUE_CATS:
        assert (br['value'] == cat).sum() >= 10, cat


# bug -> the check that must reject it
BUGS = {
    'kl_reversed': 'ppo_stats',
    'kl_sigma_not_squared': 'ppo_stats',
    'dlogp_dlogstd_no_minus_one': 'diag_logstd',
    'u_not_over_sigma': 'diag_mean',
    'logstd_column_off': 'diag_logstd',
    'actions_stride_n_out': 'diag_mean',
}


@pytest.mark.parametrize('obs_dim,A', [(6, 2), (9, 7)])
@pytest.mark.parametrize('bug', sorted(BUGS))
def test_each_check_rejects_its_bug(bug, obs_dim, A):
    r, _ = _run(obs_dim, A, bug=bug)
    assert r[BUGS[bug]] > 1.0, (bug, r)


def test_reference_formulas():
    """diag_reference's FP64 values are RLlib's DiagGaussian formulas: logp, KL(old || new), entropy, and dout equal to
    a central-difference derivative of the loss."""
    rng = np.random.default_rng(3)
    n_out, rows = 4, 32
    out = ls.f32(rng.normal(0, 0.7, (rows, n_out + 1)))
    inp = dg.diag_rows(out, n_out, COEFFS, 1)
    dout, stats, _ = dg.diag_reference(out, inp, COEFFS, n_out)
    old = ls.f32(inp['logits_old'])
    assert np.allclose(stats[2].v, dg.kl64(old, out, n_out), rtol=1e-12)
    assert np.allclose(stats[3].v, dg.entropy64(out, n_out), rtol=1e-12)
    A = n_out // 2
    # scipy-free normal log-density
    a = f64(inp['actions'])
    lp = (-0.5 * ((a - f64(out[:, :A])) / np.exp(f64(out[:, A:n_out]))) ** 2 - f64(out[:, A:n_out]) - 0.5 * math.log(2 * math.pi)).sum(1)
    assert np.allclose(dg.diag_logp64(out, a, n_out), lp, rtol=1e-12)

    def loss(o):
        lp_ = dg.diag_logp64(o, a, n_out)
        r = np.exp(lp_ - f64(inp['logp_old']))
        Adv = f64(inp['adv'])
        surr = -np.minimum(Adv * r, Adv * np.clip(r, 1 - COEFFS.clip, 1 + COEFFS.clip))
        return surr + COEFFS.kl_coeff * dg.kl64(old, o, n_out) - COEFFS.ent_coeff * dg.entropy64(o, n_out)
    h = 1e-6
    for c in range(n_out):
        up, dn = f64(out).copy(), f64(out).copy()
        up[:, c] += h
        dn[:, c] -= h
        fd = (loss(up) - loss(dn)) / (2 * h)
        assert np.allclose(dout.v[:, c], fd, rtol=1e-5, atol=1e-7), c


def test_torch_act_is_the_diagonal_gaussian():
    from paintrl_b200.rollout import MlpPolicy
    pol = MlpPolicy(6, 2, device='cpu', seed=2, discrete=False, dist='diag_gaussian')
    assert (pol.n_out, pol.action_dim, pol.dist, tuple(pol.head_w.shape)) == (4, 2, 'diag_gaussian', (128, 5))
    pol.head_b[2:4] = torch.tensor([-1.0, 0.5])                      # log-stds
    obs = torch.rand(20000, 6, dtype=torch.float64)
    a, logp, value = pol.act(obs)
    out, v = pol.forward(obs)
    assert a.dtype == torch.float64 and tuple(a.shape) == (20000, 2) and torch.equal(v, value)
    z = dg.standardised(out.numpy(), a.numpy(), 4)
    assert np.abs(z.mean(0)).max() < 0.03 and np.abs(z.std(0) - 1).max() < 0.03
    ref = dg.diag_logp64(out.numpy(), a.float().numpy(), 4)
    assert np.allclose(logp.numpy(), ref, atol=1e-4)
    for bad in (dict(discrete=True, dist='diag_gaussian'), dict(discrete=False, dist='categorical'), dict(discrete=False, dist='beta')):
        with pytest.raises(ValueError):
            MlpPolicy(6, 2, device='cpu', **bad)
    assert MlpPolicy(6, 2, device='cpu', discrete=False).dist == 'tanh_gaussian'
    assert MlpPolicy(6, 4, device='cpu').dist == 'categorical'


def _lib():
    from paintrl_b200 import _capi
    try:
        return _capi.lib()
    except RuntimeError as exc:
        pytest.skip(str(exc))


def test_entry_points_check_their_arguments():
    lib = _lib()
    F = ctypes.c_void_p(16)
    assert lib.paintrl_policy_act_diag_gaussian(None, F, 1, F, F, F, None, None) == -1
    assert b'null handle' in lib.paintrl_last_error()
    assert lib.paintrl_ppo_grad_diag_gaussian(None, F, F, 128, F, F, F, F, F, F, F, 0.2, F, F, None) == -1
    assert b'null handle' in lib.paintrl_last_error()
    header = open(__import__('os').path.join(__import__('os').path.dirname(__file__), '..', 'include', 'paintrl.h')).read()
    for name in ('paintrl_policy_act_diag_gaussian', 'paintrl_ppo_grad_diag_gaussian'):
        assert name + '(' in header


def test_trainer_refuses_spaces_the_kernels_do_not_take():
    from paintrl_b200 import train
    ok = dict(algo='ppo', action_mode='discrete', action_shape=1, granularity=4, obs_mode='section', obs_grad=4)
    assert train.check_spaces(**ok) == (6, 4)
    assert train.check_spaces(**dict(ok, action_mode='continuous', action_shape=2, obs_mode='grid')) == (16, 4)
    assert train.check_spaces(**dict(ok, action_mode='continuous', action_shape=1)) == (6, 2)
    assert train.check_spaces(**dict(ok, granularity=15, obs_grad=30)) == (32, 15)
    for bad, msg in ((dict(obs_mode='grid', obs_grad=6), '36 entries'), (dict(obs_grad=31), '33 entries'),
                     (dict(granularity=16), '1..15'), (dict(granularity=0), '1..15'),
                     (dict(algo='dqn', action_mode='continuous', action_shape=2), 'discrete actions only'),
                     (dict(action_mode='continuous', action_shape=3), 'action shape'), (dict(obs_mode='image'), 'obs mode'),
                     (dict(algo='sac'), 'algo')):
        with pytest.raises(ValueError, match=msg):
            train.check_spaces(**dict(ok, **bad))
    # the command line refuses before any work starts (no CUDA needed to get there)
    for argv in (['--algo', 'dqn', '--action-mode', 'continuous'], ['--granularity', '16'], ['--obs-mode', 'grid', '--obs-grad', '6'],
                 ['--action-shape', '2'], ['--action-mode', 'continuous', '--granularity', '5']):
        with pytest.raises(SystemExit) as e:
            train.main(argv)
        assert e.value.code == 2, argv


def _checkpoint(tmp_path, obs_dim, A, dist, with_dist=True, spaces=None):
    """A checkpoint laid out as Trainer.save writes it, with random parameters."""
    from paintrl_b200 import ppo
    n_out = 2 * A if dist == 'diag_gaussian' else A
    n = ppo.num_params(obs_dim, n_out)
    g = torch.Generator().manual_seed(1)
    learner = {'config': ppo.PPOConfig().to_dict(), 'obs_dim': obs_dim, 'n_out': n_out, 'discrete': dist == 'categorical',
               'params': torch.randn(n, generator=g), 'adam_m': torch.zeros(n), 'adam_v': torch.zeros(n), 'step': 3,
               'generator': g.get_state(), 'kl_coeff': 0.2}
    ck = {'learner': learner, 'obs_dim': obs_dim, 'n_out': n_out, 'discrete': dist == 'categorical', 'env_settings': {}}
    if with_dist:
        learner['dist'] = dist
        ck['dist'] = dist
        ck['spaces'] = spaces
    path = tmp_path / ('%s_%d.pt' % (dist, with_dist))
    torch.save(ck, path)
    return path, ck


def test_checkpoint_round_trips(tmp_path):
    from paintrl_b200 import ppo, train
    from paintrl_b200.learner import flat_params
    spaces = dict(train.C2_SPACES, action_mode='continuous', action_shape=2, obs_mode='grid')
    path, ck = _checkpoint(tmp_path, 16, 2, 'diag_gaussian', spaces=spaces)
    pol = train.load_policy(path, 'cpu')
    assert (pol.dist, pol.n_out, pol.action_dim, pol.obs_dim) == ('diag_gaussian', 4, 2, 16)
    assert torch.equal(flat_params(pol), ck['learner']['params'])
    assert train.checkpoint_spaces(torch.load(path, weights_only=False)) == spaces
    # a state of another distribution is refused
    with pytest.raises(ValueError, match='distribution'):
        ppo.check_state_dict(ck['learner'], 16, 4, False, 'tanh_gaussian')
    # checkpoints written before `dist` and `spaces` were recorded load as before: C2's spaces, the distribution every
    # policy had then
    for dist, A in (('categorical', 4), ('tanh_gaussian', 2)):
        path, ck = _checkpoint(tmp_path, 6, A, dist, with_dist=False)
        pol = train.load_policy(path, 'cpu')
        assert (pol.dist, pol.n_out) == (dist, A)
        assert torch.equal(flat_params(pol), ck['learner']['params'])
        assert train.checkpoint_spaces(ck) == train.C2_SPACES
        ppo.check_state_dict(ck['learner'], 6, A, dist == 'categorical', dist)
        ppo.check_state_dict(ck['learner'], 6, A, dist == 'categorical')
