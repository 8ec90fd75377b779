"""FP64 reference of the learner kernel's diagonal-Gaussian PPO loss stage (kLossPpoDiag, paintrl_b200/csrc/
paintrl_learn.cuh) and of the act kernel's diagonal-Gaussian log-probability (pol_diag_logp, paintrl_policy.cuh), built
on learner_stages.py's running error analysis (class Bounded and its per-operation constants).  Pure functions on
NumPy arrays: no GPU calls.  test_gpu_diag_gaussian.py feeds them the kernels' outputs; test_diag_gaussian_cpu.py feeds
them a NumPy restatement, with and without planted bugs.

The head has n_out = 2A outputs before the value: the mean mu_o in column o and log sigma_o in column A + o.  The
kernel's operations, each one FP32 rounding (the library is built with -fmad=false, so no product is fused into an
add), per dimension o in order:

    sigma = expf(log sigma), sigma_old = expf(log sigma_old)                       (learner_stages.EXPF_ULP)
    u     = (a - mu) / sigma;  logp = (logp - (0.5 u) u) - log sigma;  at the end logp - A * 0.9189385f
    d     = mu - mu_old;  q = (sigma_old sigma_old + d d) / (sigma sigma)
    KL   += ((log sigma - log sigma_old) + 0.5 q) - 0.5;  H += log sigma + 1.4189385f
    dout[mu]        = s (g_logp (u / sigma) + kl_coeff (d is2)),  is2 = 1 / (sigma sigma)
    dout[log sigma] = s ((g_logp (u u - 1) + kl_coeff (1 - q2)) - ent_coeff),  q2 = (sigma_old sigma_old + d d) is2

The surrogate, the value loss and the six statistics are kLossPpo's, restated here as learner_stages.ppo_reference
computes them.
"""
import numpy as np

import learner_stages as ls
from learner_stages import Bounded, U32, add, expf, mul, neg, sub, where, maximum, minimum

LOG_SQRT_2PI = ls.LOG_SQRT_2PI        # 0.9189385332046727f in the kernel
GAUSS_ENTROPY = ls.GAUSS_ENTROPY      # 1.4189385332046727f: log(2 pi e) / 2


def div(a, b):
    """a / b, one FP32 rounding (IEEE division): |a'/b' - a/b| <= (e_a + |a / b| e_b) / (|b| - e_b)."""
    a, b = ls._c(a), ls._c(b)
    assert (b.e < np.abs(b.v)).all()
    v = a.v / b.v
    return ls._round(v, (a.e + np.abs(v) * b.e) / (np.abs(b.v) - b.e))


def columns(out, n_out):
    """(A, mu, log sigma) of head outputs [rows, >= n_out] in FP64."""
    A = n_out // 2
    o = np.asarray(out, dtype=np.float64)
    return A, o[:, :A], o[:, A:2 * A]


def diag_logp64(out, actions, n_out):
    """log N(a; mu, diag sigma^2) in FP64 of the FP32 actions."""
    A, mu, lsig = columns(out, n_out)
    a = ls.f32(actions).astype(np.float64)
    u = (a - mu) / np.exp(lsig)
    return (-0.5 * u * u - lsig).sum(axis=1) - A * LOG_SQRT_2PI


def logp_reference(out, actions, n_out):
    """pol_diag_logp as Bounded: the act kernel's logp output and the learner's logp."""
    A, mu, lsig = columns(out, n_out)
    a = ls.f32(actions).astype(np.float64)
    logp = Bounded(np.zeros(len(mu)))
    for o in range(A):
        u = div(sub(a[:, o], mu[:, o]), expf(Bounded(lsig[:, o])))
        logp = sub(sub(logp, mul(mul(0.5, u), u)), lsig[:, o])
    return sub(logp, mul(float(A), ls._const(LOG_SQRT_2PI)))


def _dim(out, old, a, n_out, o):
    """The per-dimension Bounded quantities both passes of the stage compute."""
    A, mu, lsig = columns(out, n_out)
    _, muo, lso = columns(old, n_out)
    sig, sigo = expf(Bounded(lsig[:, o])), expf(Bounded(lso[:, o]))
    u = div(sub(a[:, o], mu[:, o]), sig)
    d = sub(mu[:, o], muo[:, o])
    num = add(mul(sigo, sigo), mul(d, d))
    return {'mu': mu[:, o], 'ls': lsig[:, o], 'lso': lso[:, o], 'sig': sig, 'u': u, 'd': d, 'num': num, 'sig2': mul(sig, sig)}


def diag_reference(out, inp, cf, n_out, inv_n=1.0):
    """The kLossPpoDiag stage for each row on the kernel's head outputs `out` [rows, n_out + 1]: Bounded dout [rows,
    n_out + 1], the six statistics and the FP64 branch quantities (learner_stages.ppo_branches takes them).  `inp` as
    learner_stages.ppo_reference's, with actions float64 [rows, n_out / 2]."""
    rows = out.shape[0]
    A = n_out // 2
    old = ls.f32(inp['logits_old'])
    a = ls.f32(inp['actions']).astype(np.float64).reshape(rows, A)
    s = Bounded(np.full(rows, inv_n), U32 * inv_n if inv_n != 1.0 else 0.0)
    v = Bounded(np.asarray(out, dtype=np.float64)[:, n_out])
    logp = logp_reference(out, a, n_out)
    kl, ent = Bounded(np.zeros(rows)), Bounded(np.zeros(rows))
    dims = [_dim(out, old, a, n_out, o) for o in range(A)]
    for q in dims:
        kl = add(kl, sub(add(sub(q['ls'], q['lso']), mul(0.5, div(q['num'], q['sig2']))), 0.5))
        ent = add(ent, add(q['ls'], ls._const(GAUSS_ENTROPY)))
    # the surrogate and the value loss: learner_stages.ppo_reference's tail
    Adv, R, vold = [Bounded(ls.f32(inp[k]).astype(np.float64)) for k in ('adv', 'vtarg', 'value_old')]
    r = expf(sub(logp, ls.f32(inp['logp_old']).astype(np.float64)))
    lo, hi = Bounded(1.0 - cf.clip, U32), Bounded(1.0 + cf.clip, U32)
    rc = where(r.v < lo.v, lo, where(r.v > hi.v, hi, r))
    s1, s2 = mul(Adv, r), mul(Adv, rc)
    g_logp = where(s1.v <= s2.v, neg(mul(Adv, r)), 0.0)
    dvR = sub(v, R)
    vf1 = mul(dvR, dvR)
    dv = sub(v, vold)
    vfc = Bounded(cf.vf_clip)
    dvc = where(dv.v < -vfc.v, neg(vfc), where(dv.v > vfc.v, vfc, dv))
    vcl = add(vold, dvc)
    dcR = sub(vcl, R)
    vf2 = mul(dcR, dcR)
    inside = np.abs(dv.v) <= cf.vf_clip
    g_in = Bounded(2.0 * dvR.v, np.maximum(mul(2.0, dvR).e, mul(2.0, dcR).e + 2.0 * np.abs(dcR.v - dvR.v)))
    g_v = where(inside, g_in, where(vf1.v >= vf2.v, mul(2.0, dvR), 0.0))
    dmu, dls = [], []
    for q in dims:
        is2 = div(1.0, q['sig2'])
        dmu.append(mul(s, add(mul(g_logp, div(q['u'], q['sig'])), mul(cf.kl_coeff, mul(q['d'], is2)))))
        q2 = mul(q['num'], is2)
        dls.append(mul(s, sub(add(mul(g_logp, sub(mul(q['u'], q['u']), 1.0)), mul(cf.kl_coeff, sub(1.0, q2))), cf.ent_coeff)))
    dout = ls._stack(dmu + dls + [mul(mul(s, cf.vf_coeff), g_v)])
    stats = [neg(minimum(s1, s2)), maximum(vf1, vf2), kl, ent, Bounded((np.abs(r.v - 1.0) > cf.clip).astype(np.float64)), r]
    branch = {'r': r.v, 'adv': Adv.v, 'dv': dv.v, 'vf1': vf1.v, 'vf2': vf2.v}
    return dout, stats, branch


def check_diag_loss(out, dout, stats, inp, cf, n_out):
    """dout (the sample's db3) and the six statistics against diag_reference: {'diag_mean' (the mean columns),
    'diag_logstd' (the log-std columns), 'diag_value' (the value column), 'ppo_stats'}, plus the Bounded dout reference
    and the branch quantities."""
    ref, st_ref, branch = diag_reference(out, inp, cf, n_out)
    A = n_out // 2
    dout, stats = np.asarray(dout), np.asarray(stats)
    r = {'diag_mean': ls.ratio(dout[:, :A], ref[:, :A]), 'diag_logstd': ls.ratio(dout[:, A:n_out], ref[:, A:n_out]),
         'diag_value': ls.ratio(dout[:, n_out], ref[:, n_out]),
         'ppo_stats': max(ls.ratio(stats[:, i], st_ref[i]) for i in range(6))}
    return r, ref, branch


def diag_rows(out, n_out, cf, seed):
    """Inputs for rows whose head outputs are `out`: actions mu + sigma z in FP32 (float64 [rows, A]), and the ratio,
    sign of A and value categories of learner_stages.ppo_rows (row j: (ratio, sign) category j mod 6, value category
    (j // 6) mod 3), logp_old set so that the ratio lands where the category says."""
    rng = np.random.default_rng(seed + 1000)
    rows = out.shape[0]
    A, mu, lsig = columns(out, n_out)
    actions = ls.f32(mu + np.exp(lsig) * rng.standard_normal((rows, A))).astype(np.float64)
    base = ls.ppo_rows(out, n_out, True, cf, seed)      # value_old, vtarg, adv and logits_old; its actions are replaced
    cat = [ls.PPO_RATIO_CATS[k % 6] for k in range(rows)]
    target = np.array([{'inside': 1 + 0.4 * cf.clip * sg, 'above': 1 + 2 * cf.clip, 'below': 1 - 2 * cf.clip}[c] for c, sg in cat])
    return dict(base, actions=actions, logp_old=ls.f32(diag_logp64(out, actions, n_out) - np.log(target)))


def standardised(out, actions, n_out):
    """(a - mu) / sigma in FP64: N(0, 1) draws when the actions come from the head."""
    A, mu, lsig = columns(out, n_out)
    return (np.asarray(actions, dtype=np.float64).reshape(len(mu), A) - mu) / np.exp(lsig)


def entropy64(out, n_out):
    A, _, lsig = columns(out, n_out)
    return (lsig + GAUSS_ENTROPY).sum(axis=1)


def kl64(old, new, n_out):
    """KL(old || new) of two diagonal Gaussians in FP64 (RLlib's prev_dist.kl(curr_dist))."""
    A, muo, lso = columns(old, n_out)
    _, mu, lsn = columns(new, n_out)
    return (lsn - lso + (np.exp(2 * lso) + (muo - mu) ** 2) / (2 * np.exp(2 * lsn)) - 0.5).sum(axis=1)

