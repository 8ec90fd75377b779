"""The stage checkers of learner_stages.py can fail: a NumPy restatement of one-sample learner gradients (FP32 values,
h1 and dz2 rounded to BF16 where the kernel rounds them, tanh / exp / log computed exactly and rounded once) passes
every checker at every shape the GPU tests use, and a restatement carrying one planted bug is rejected by the checker
that names it.  This is the evidence that test_gpu_learner_stages.py would fail on a subtly wrong kernel."""
import numpy as np
import pytest

import learner_stages as ls

SHAPES = [(1, 1), (6, 4), (8, 7), (8, 8), (9, 7), (32, 15)]
ROWS = 64
COEFFS = ls.PpoCoeffs(clip=0.2, vf_clip=0.5, vf_coeff=0.5, ent_coeff=0.01, kl_coeff=0.2)
GAMMA = 0.9

f64 = lambda a: np.asarray(a, dtype=np.float64)


def _forward(params, obs_dim, n_out, x32, bug=None):
    P = ls.split_flat(params, obs_dim, n_out)
    h1 = ls.f32(np.tanh(f64(x32) @ f64(P['w1']) + f64(P['b1'])))
    h1b = ls.bf16(h1)
    z2 = ls.f32(f64(h1b) @ f64(ls.bf16(P['w2'])))
    h2 = ls.f32(np.tanh(z2 if bug == 'no_b2' else ls.f32(z2 + P['b2'])))
    out = ls.f32(f64(h2) @ f64(P['w3']) + f64(P['b3']))
    if bug == 'head_column_dropped':             # a cap one short: the value column is never summed
        out[:, n_out] = 0.0
    return {'h1': h1, 'h1b': h1b, 'h2': h2, 'out': out}


def _ppo_loss(out, inp, cf, discrete, n_out, bug=None):
    o, old = f64(out), f64(inp['logits_old'])
    rows = len(o)
    if discrete:
        act = inp['actions']
        lsm = lambda z: z - z.max(1, keepdims=True) - np.log(np.exp(z - z.max(1, keepdims=True)).sum(1, keepdims=True))
        lp, lpo = lsm(o[:, :n_out]), lsm(old[:, :n_out])
        p, po = np.exp(lp), np.exp(lpo)
        logp = lp[np.arange(rows), act]
        ent = -(p * lp).sum(1)
        if bug == 'kl_reversed':                 # KL(new || old)
            kl = (p * (lp - lpo)).sum(1)
            dkl = p * ((lp - lpo) - kl[:, None])
        else:
            kl = (po * (lpo - lp)).sum(1)
            dkl = p - po
    else:
        a = f64(ls.f32(inp['actions']))
        mu, muo = np.tanh(o[:, :n_out]), np.tanh(old[:, :n_out])
        logp = (-0.5 * (a - mu) ** 2 - ls.LOG_SQRT_2PI).sum(1)
        kl = 0.5 * ((muo - mu) ** 2).sum(1)
        ent = np.full(rows, n_out * ls.GAUSS_ENTROPY)
    A, R, vold = f64(inp['adv']), f64(inp['vtarg']), f64(inp['value_old'])
    r = np.exp(logp - f64(inp['logp_old']))
    rc = np.clip(r, 1 - cf.clip, 1 + cf.clip)
    s1, s2 = A * r, A * rc
    g_logp = -A * r if bug == 'surrogate_on_clipped' else np.where(s1 <= s2, -A * r, 0.0)
    v = o[:, n_out]
    vf1 = (v - R) ** 2
    dv = v - vold
    vcl = vold + np.clip(dv, -cf.vf_clip, cf.vf_clip)
    vf2 = (vcl - R) ** 2
    take1 = vf1 < vf2 if bug == 'value_branch' else vf1 >= vf2
    g_v = np.where(take1, 2 * (v - R), np.where(np.abs(dv) <= cf.vf_clip, 2 * (vcl - R), 0.0))
    if discrete:
        onehot = np.arange(n_out)[None, :] == act[:, None]
        esign = -1.0 if bug == 'entropy_sign' else 1.0
        d = g_logp[:, None] * (onehot - p) + cf.kl_coeff * dkl + esign * cf.ent_coeff * p * (lp + ent[:, None])
    else:
        d = (g_logp[:, None] * (a - mu) + cf.kl_coeff * (mu - muo)) * (1 - mu * mu)
    dout = np.concatenate([d, (cf.vf_coeff * g_v)[:, None]], axis=1)
    stats = np.stack([-np.minimum(s1, s2), np.maximum(vf1, vf2), kl * (2.0 if bug == 'kl_stat_double' else 1.0), ent,
                      (np.abs(r - 1) > cf.clip).astype(np.float64), r], axis=1)
    return ls.f32(dout), ls.f32(stats)


def _dqn_loss(out, head_on, head_tn, inp, gamma, n_out, bug=None):
    """The DQN stage has no transcendental function: restated in the kernel's FP32 operation order."""
    f32 = ls.f32

    def q(head):
        sa = np.zeros(len(head), np.float32)
        for o in range(n_out):
            sa = f32(sa + head[:, o])
        return f32(head[:, n_out:] + f32(head[:, :n_out] - f32(sa / np.float32(n_out))[:, None]))
    rows = np.arange(len(out))
    act = inp['actions']
    qs, qo, qt = q(out), q(head_on), q(head_tn)
    an = qo.argmax(1)
    nd = np.where(inp['done'] != 0, np.float32(0), np.float32(1))
    y = f32(inp['reward'] + f32(f32(np.float32(gamma) * nd) * qt[rows, an]))
    qsa = qs[rows, act]
    td = f32(qsa - y)
    g = f32(np.clip(td, -1, 1))
    onehot = (np.arange(n_out)[None, :] == act[:, None]).astype(np.float32)
    centre = np.float32(0) if bug == 'dqn_no_centring' else np.float32(1) / np.float32(n_out)
    dout = np.concatenate([f32(g[:, None] * f32(onehot - centre)), g[:, None]], axis=1)
    atd = np.abs(td)
    huber = np.where(atd <= 1, f32(f32(np.float32(0.5) * td) * td), f32(atd - np.float32(0.5)))
    return dout, np.stack([huber, atd, qsa, y], axis=1)


def _sample_grads(params, obs_dim, n_out, x32, fw, dout, bug=None):
    """The flat one-sample gradient of each row, laid out as the kernel's n = 1 launch writes it."""
    P = ls.split_flat(params, obs_dim, n_out)
    h2 = fw['h2']
    dW3 = ls.f32(h2[:, :, None] * dout[:, None, :])
    dh = f64(dout) @ f64(P['w3']).T
    dz2 = ls.f32(dh if bug == 'dz2_no_tanh_grad' else dh * (1 - f64(h2) ** 2))
    dz2b = ls.bf16(dz2)
    dW2 = ls.f32(fw['h1b'][:, :, None] * dz2b[:, None, :])
    dz1 = ls.f32((f64(dz2b) @ f64(ls.bf16(P['w2'])).T) * (1 - f64(fw['h1']) ** 2))
    dW1 = ls.f32(x32[:, :, None] * dz1[:, None, :])
    rows = len(x32)
    return np.concatenate([dW1.reshape(rows, -1), dz1, dW2.reshape(rows, -1), dz2, dW3.reshape(rows, -1), dout], axis=1)


def _run(obs_dim, n_out, mode, bug=None, seed=0):
    """Every checker's worst ratio for the restatement of ROWS one-sample launches."""
    rng = np.random.default_rng(seed)
    x32 = ls.f32(rng.uniform(0, 1, (ROWS, obs_dim)))
    params = ls.make_params(obs_dim, n_out, seed=obs_dim + n_out)
    if mode == 'dqn' and n_out >= 3:
        params = ls.make_tie(params, obs_dim, n_out)
    fw = _forward(params, obs_dim, n_out, x32, bug)
    out = fw['out']
    if mode == 'dqn':
        xn = ls.f32(rng.uniform(0, 1, (ROWS, obs_dim)))
        target = ls.make_params(obs_dim, n_out, seed=100 + obs_dim)
        head_on = _forward(params, obs_dim, n_out, xn, bug)['out']
        head_tn = _forward(target, obs_dim, n_out, xn, bug)['out']
        inp = ls.dqn_rows(out, head_on, head_tn, n_out, GAMMA, seed)
        dout, stats = _dqn_loss(out, head_on, head_tn, inp, GAMMA, n_out, bug)
        loss, _, _ = ls.check_dqn_loss(out, head_on, head_tn, dout, stats, inp, GAMMA, n_out)
    else:
        discrete = mode == 'ppo_discrete'
        inp = ls.ppo_rows(out, n_out, discrete, COEFFS, seed)
        dout, stats = _ppo_loss(out, inp, COEFFS, discrete, n_out, bug)
        loss, _, branch = ls.check_ppo_loss(out, dout, stats, inp, COEFFS, discrete, n_out)
        if bug is None:
            br = ls.ppo_branches(branch, COEFFS)
            assert br['margin'] > 0.1, br['margin']
            for cat, sign in ls.PPO_RATIO_CATS:
                assert ((br['ratio'] == cat) & (br['adv_pos'] == (sign > 0))).sum() >= 5, (cat, sign)
            for cat in ls.PPO_VALUE_CATS:
                assert (br['value'] == cat).sum() >= 10, cat
    grads = _sample_grads(params, obs_dim, n_out, x32, fw, dout, bug)
    stages, _ = ls.check_sample_stages(params, obs_dim, n_out, x32, grads, out)
    return dict(stages, **loss)


@pytest.mark.parametrize('mode', ['ppo_discrete', 'ppo_continuous', 'dqn'])
@pytest.mark.parametrize('obs_dim,n_out', SHAPES)
def test_checkers_accept_the_restatement(obs_dim, n_out, mode):
    r = _run(obs_dim, n_out, mode)
    assert r.pop('exact') == 0
    assert all(v <= 1.0 for v in r.values()), r


# bug -> (the loss it needs, the checker that must reject it)
BUGS = {
    'entropy_sign': ('ppo_discrete', 'ppo_loss'),
    'kl_reversed': ('ppo_discrete', 'ppo_loss'),
    'value_branch': ('ppo_discrete', 'ppo_loss'),
    'surrogate_on_clipped': ('ppo_discrete', 'ppo_loss'),
    'no_b2': ('ppo_discrete', 'layer2'),
    'head_column_dropped': ('ppo_continuous', 'head'),
    'dz2_no_tanh_grad': ('ppo_discrete', 'head_backward'),
    'dqn_no_centring': ('dqn', 'dqn_loss'),
    'kl_stat_double': ('ppo_discrete', 'ppo_stats'),
}


@pytest.mark.parametrize('obs_dim,n_out', [(6, 4), (9, 7)])
@pytest.mark.parametrize('bug', sorted(BUGS))
def test_each_checker_rejects_its_bug(bug, obs_dim, n_out):
    mode, checker = BUGS[bug]
    r = _run(obs_dim, n_out, mode, bug=bug)
    assert r[checker] > 1.0, (bug, checker, r)


def test_bf16_rounds_to_nearest_even():
    x = np.array([1.0, 1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, 1.0 + 2 ** -8 + 2 ** -20, -3.0 - 2 ** -7], dtype=np.float32)
    assert ls.bf16(x).tolist() == [1.0, 1.0, 1.0 + 2 ** -6, 1.0 + 2 ** -7, -3.0]
