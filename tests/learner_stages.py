"""Stage-by-stage FP64 references for the learner kernel (ppo_grad_kernel, paintrl_b200/csrc/paintrl_learn.cuh) and
the act kernel's forward pass it shares (paintrl_policy.cuh).  Pure functions on NumPy arrays: no GPU calls.  The GPU
tests (test_gpu_learner_stages.py) feed them the kernel's outputs; test_learner_stages_cpu.py feeds them a NumPy
restatement, with and without planted bugs, to show that each checker can fail.

Why a minibatch of one sample exposes every intermediate
--------------------------------------------------------
For n = 1 the launch has one CTA and inv_n = 1.  Row 0 is the sample; rows 1..127 are invalid: their dout is set to 0
before the loss stage, so their dz2 = dh * (1 - h2^2) is 0 (dh is an FMA chain over zeros), their BF16 dz2 tile rows
are 0, their dz1 is written as 0 and their x row is loaded as 0.  Every cross-sample sum therefore adds one non-zero
term to zeros, and ppo_reduce_kernel adds one partial to 0.  Reading the flat gradient of that launch:

    db3[o]     = 0 + dout[o]                                  dout itself, bitwise
    dW3[c, o]  = fmaf(h2[c], dout[o], 0)  = fl(h2[c] dout[o])  one rounding: h2 is recovered as the FP32 value whose
                                                               products reproduce the whole row of dW3 (exact identity)
    db2[c]     = 0 + dz2[c]                                   dz2 in FP32, before the BF16 pack, bitwise
    dW2[k, n]  = bf16(dz2[n]) bf16(h1[k])  (tcgen05.mma)      a product of two BF16 values is exact in FP32 and every
                                                               other product of the K = 128 sample reduction is 0: the
                                                               matrix is exactly rank 1 and gives the forward's BF16 h1
    db1[k]     = 0 + dz1[k],  dz1 = dh1 (1 - h1^2)            bitwise (h1 here is the FP32 value the backward
                                                               recomputes with the forward's arithmetic)
    dW1[i, k]  = fmaf(x[i], dz1[k], 0)    = fl(x[i] dz1[k])   bitwise
    stats      = the row's own statistics                      bitwise (0 + s, times inv_n = 1)

paintrl_ppo_forward returns the head outputs `out` of the same forward code.  So every stage below is compared with an
FP64 computation whose inputs are the kernel's own values from the stage before, and only that stage's arithmetic
enters its tolerance.

Tolerances
----------
Each bound is a running error analysis of the kernel's own sequence of FP32 operations (class Bounded): every value
carries the FP64 result of the exact operation and a bound on how far the kernel's FP32 result can be from it, built
from the per-operation constants below.  A checker returns the worst |kernel - reference| / bound over its elements
(<= 1 passes), so a test can print its margin.  Branch decisions (ratio clip, value clip, Huber) are taken in FP64;
the row recipes keep every row a stated margin away from each boundary, far outside these bounds, and the tests assert
that margin.
"""
import math

import numpy as np

H1, H2 = 256, 128

# ---- per-operation error constants -------------------------------------------------------------------------------
# FP32 round to nearest even: |fl(x) - x| <= 2^-24 |x| (unit roundoff), one ulp of y is at most 2^-23 |y|.
U32 = 2.0 ** -24
ULP32 = 2.0 ** -23
# BF16 (8 significand bits) round to nearest even: |bf16(x) - x| <= 2^-8 |x|.
U_BF16 = 2.0 ** -8
# PTX ISA, tanh: tanh.approx.f32 has a maximum relative error of 2^-11 over the full range of inputs.  pol_tanh is
# tanh.approx.f32.
TANH_APPROX_REL = 2.0 ** -11
# CUDA C++ Programming Guide, mathematical functions, maximum ulp error of the full-range single-precision function:
# expf(x): 2 ulp.  (The library is built without --use_fast_math, so expf is not __expf.)
EXPF_ULP = 2
# CUDA C++ Programming Guide, intrinsic functions: __expf(x): "The maximum ulp error is 2 + floor(abs(1.173 * x))";
# __logf(x): "For x in [0.5, 2], the maximum absolute error is 2^-21.41, otherwise, the maximum ulp error is 3."
LOGF_INTR_ABS, LOGF_INTR_ULP = 2.0 ** -21.41, 3
# Tensor-core FP32 accumulation (tcgen05.mma kind::f16, FP32 accumulator).  The PTX ISA does not state the
# accumulation order or the rounding of the intermediate sums.  Measurements on earlier tensor cores (Fasi, Higham,
# Mikaitis, Pranesh, "Numerical behavior of NVIDIA tensor cores", PeerJ CS 2021) found products exact and additions
# truncated rather than rounded: up to one FP32 ulp, 2^-23 relative to the running magnitude, per addition.  Assumed
# here: a K-term accumulation is within K * 2^-23 * sum |products| of the exact sum.  The GPU test prints the worst
# observed ratio of the stages this assumption enters (layer 2 forward, dh1 / dz1).
TC_ULP = 2.0 ** -23
# The FP64 reference's own rounding: a few dozen FP64 operations, each 2^-53 relative; 2^-40 relative covers it.
REF64 = 2.0 ** -40


def gamma(m, u=U32):
    """Recursive summation of m + 1 terms: |error| <= gamma(m) sum |terms| (Higham, Accuracy and Stability, 3.1)."""
    return m * u / (1.0 - m * u)


def bf16(a):
    """Round float32 values to BF16 (round to nearest even, as __float2bfloat16_rn), returned as float32."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    u = a.view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return r.astype(np.uint32).view(np.float32).reshape(a.shape)


def f32(a):
    return np.asarray(a, dtype=np.float32)


# ---- the flat parameter layout (paintrl_policy.cuh pol_num_params) ----------------------------------------------
def num_params(obs_dim, n_out):
    return obs_dim * H1 + H1 + H1 * H2 + H2 + H2 * (n_out + 1) + (n_out + 1)


def split_flat(p, obs_dim, n_out):
    """w1 [obs, 256] | b1 | w2 [256, 128] | b2 | w3 [128, n_out + 1] | b3 of a flat vector (or of the last axis of a
    [rows, n_params] array), as views."""
    p = np.asarray(p)
    lead = p.shape[:-1]
    sizes = (('w1', (obs_dim, H1)), ('b1', (H1,)), ('w2', (H1, H2)), ('b2', (H2,)), ('w3', (H2, n_out + 1)), ('b3', (n_out + 1,)))
    out, off = {}, 0
    for name, s in sizes:
        n = int(np.prod(s))
        out[name] = p[..., off:off + n].reshape(lead + s)
        off += n
    assert off == p.shape[-1], (off, p.shape)
    return out


def make_params(obs_dim, n_out, seed):
    """A flat float32 parameter vector at the rollout policy's initial scale, with non-zero biases and a head whose
    outputs are of order 1."""
    rng = np.random.default_rng(seed)
    nout1 = n_out + 1
    parts = [rng.uniform(-1, 1, (obs_dim, H1)) / math.sqrt(obs_dim), np.linspace(-0.3, 0.3, H1),
             rng.uniform(-1, 1, (H1, H2)) / math.sqrt(H1), np.linspace(-0.3, 0.3, H2),
             rng.uniform(-1, 1, (H2, nout1)) / math.sqrt(H2) * 2.0, np.linspace(-0.3, 0.3, nout1)]
    return f32(np.concatenate([np.ravel(x) for x in parts]))


def make_tie(params, obs_dim, n_out):
    """Head columns 1 and 2 identical and dominant: on every row A_1 == A_2 > every other A, so the greedy action is a
    tie that the lowest-index rule decides (n_out >= 3)."""
    p = f32(params).copy()
    s = split_flat(p, obs_dim, n_out)
    s['w3'][:, 2] = s['w3'][:, 1]
    s['b3'][1] = s['b3'][2] = 5.0
    return p


# ---- running error analysis ---------------------------------------------------------------------------------------
class Bounded(object):
    """v: the exact operation's result in FP64; e: a bound on |kernel FP32 result - v|.  Each helper below is one FP32
    operation of the kernel, rounded once (or an exact one)."""
    __slots__ = ('v', 'e')

    def __init__(self, v, e=0.0):
        self.v = np.asarray(v, dtype=np.float64)
        self.e = np.broadcast_to(np.asarray(e, dtype=np.float64), self.v.shape).copy()

    def __getitem__(self, k):
        return Bounded(self.v[k], self.e[k])


def _c(x):
    return x if isinstance(x, Bounded) else Bounded(x)


def _round(v, e):
    return Bounded(v, e + U32 * (np.abs(v) + e))


def add(a, b):
    a, b = _c(a), _c(b)
    return _round(a.v + b.v, a.e + b.e)


def sub(a, b):
    a, b = _c(a), _c(b)
    return _round(a.v - b.v, a.e + b.e)


def mul(a, b):
    a, b = _c(a), _c(b)
    return _round(a.v * b.v, np.abs(a.v) * b.e + np.abs(b.v) * a.e + a.e * b.e)


def fma(a, b, c):
    """fmaf(a, b, c): one rounding of a b + c."""
    a, b, c = _c(a), _c(b), _c(c)
    return _round(a.v * b.v + c.v, np.abs(a.v) * b.e + np.abs(b.v) * a.e + a.e * b.e + c.e)


def neg(a):
    return Bounded(-a.v, a.e)


def absb(a):
    return Bounded(np.abs(a.v), a.e)


def minimum(a, b):
    a, b = _c(a), _c(b)
    return Bounded(np.minimum(a.v, b.v), np.maximum(a.e, b.e))


def maximum(a, b):
    a, b = _c(a), _c(b)
    return Bounded(np.maximum(a.v, b.v), np.maximum(a.e, b.e))


def where(cond, a, b):
    a, b = _c(a), _c(b)
    return Bounded(np.where(cond, a.v, b.v), np.where(cond, a.e, b.e))


def expf(a, intrinsic=False):
    """expf (EXPF_ULP) or __expf (2 + floor(1.173 |x|) ulp at the kernel's argument, |x| <= |v| + e)."""
    v = np.exp(a.v)
    ulps = 2.0 + np.floor(1.173 * (np.abs(a.v) + a.e)) if intrinsic else EXPF_ULP
    grow = np.exp(a.e)
    return Bounded(v, v * (grow - 1.0) + ulps * ULP32 * v * grow)


def logf_intrinsic(a):
    """__logf of a positive argument: the argument's error through log, then the larger of the two documented cases
    (the FP32 argument may land on either side of 2)."""
    assert (a.e < a.v).all()
    v = np.log(a.v)
    prop = -np.log1p(-a.e / a.v)
    return Bounded(v, prop + np.maximum(LOGF_INTR_ABS, LOGF_INTR_ULP * ULP32 * (np.abs(v) + prop)))


def tanh_approx(a):
    """tanh.approx.f32: the argument's error through tanh (slope at most 1 - tanh^2 of the smallest |x| in range),
    then TANH_APPROX_REL of the result."""
    v = np.tanh(a.v)
    slope = 1.0 - np.tanh(np.maximum(np.abs(a.v) - a.e, 0.0)) ** 2
    prop = slope * a.e
    return Bounded(v, prop + TANH_APPROX_REL * (np.abs(v) + prop))


def ratio(kernel, ref):
    """Worst |kernel - ref.v| / bound; an element whose bound is 0 must be equal (else inf)."""
    k = np.asarray(kernel, dtype=np.float64)
    bound = ref.e + REF64 * np.abs(ref.v)
    err = np.abs(k - ref.v)
    if not np.isfinite(k).all():
        return float('inf')
    r = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err == 0, 0.0, np.inf))
    return float(r.max()) if r.size else 0.0


# ---- splitting an n = 1 gradient --------------------------------------------------------------------------------
def split_sample_grads(grads, obs_dim, n_out):
    """grads float32 [rows, n_params], each row the gradient of a one-sample launch.  Returns the intermediates of the
    table in the module docstring, h1_bf16 recovered from dW2 and h2 from dW3, 'live' (rows with a non-zero dout: a
    row whose loss gradient is 0, such as a clipped value on a one-action head, carries no intermediate and must have
    an all-zero gradient) and 'exact_fail': per row, the number of entries that break an exact identity (dW2 rank 1
    with BF16 factors, dW3 = fl(h2 dout), a dead row's gradient all zero)."""
    g = split_flat(f32(grads), obs_dim, n_out)
    rows = g['b3'].shape[0]
    dout, dz2, dz1 = g['b3'], g['b2'], g['b1']
    dz2b = bf16(dz2)
    fail = np.zeros(rows, dtype=np.int64)
    live = (dout != 0).any(axis=1)
    fail += np.where(live, 0, (f32(grads) != 0).sum(axis=1))
    # h1_bf16 from the column of dW2 with the largest |bf16(dz2)|: the quotient of an exact product is exact
    nstar = np.abs(dz2b).argmax(axis=1)
    piv = dz2b[np.arange(rows), nstar].astype(np.float64)
    fail += live & (piv == 0)
    h1b = f32(g['w2'][np.arange(rows), :, nstar].astype(np.float64) / np.where(piv == 0, 1.0, piv)[:, None])
    fail += np.where(live, (bf16(h1b) != h1b).sum(axis=1), 0)
    fail += np.where(live, (f32(h1b[:, :, None].astype(np.float64) * dz2b[:, None, :].astype(np.float64)) != g['w2']).sum(axis=(1, 2)), 0)
    # h2: of the FP32 neighbours of dW3 / dout at the largest |dout|, the one whose products reproduce the whole row
    ostar = np.abs(dout).argmax(axis=1)
    dpiv = dout[np.arange(rows), ostar].astype(np.float64)
    fail += live & (dpiv == 0)
    q = f32(g['w3'][np.arange(rows), :, ostar].astype(np.float64) / np.where(dpiv == 0, 1.0, dpiv)[:, None])
    h2 = q.copy()
    found = np.zeros(q.shape, dtype=bool)
    for cand in (q, np.nextafter(q, f32(np.inf)), np.nextafter(q, f32(-np.inf))):
        ok = (f32(cand[:, :, None] * dout[:, None, :]) == g['w3']).all(axis=2) & ~found
        h2[ok] = cand[ok]
        found |= ok
    fail += np.where(live, (~found).sum(axis=1), 0)
    return {'live': live, 'dout': dout, 'dW3': g['w3'], 'dz2': dz2, 'dW2': g['w2'], 'dz1': dz1, 'dW1': g['w1'], 'h1b': h1b, 'h2': h2,
            'exact_fail': fail}


# ---- exact identities --------------------------------------------------------------------------------------------
def check_exact(st, x32):
    """The bitwise identities: the recovery identities of split_sample_grads, and dW1[i, k] = fl(x[i] dz1[k]).
    Returns the number of entries that break one (0 passes)."""
    dw1 = f32(x32.astype(np.float32)[:, :, None] * st['dz1'][:, None, :])
    return int(st['exact_fail'].sum() + (dw1 != st['dW1']).sum())


# ---- forward stages ----------------------------------------------------------------------------------------------
def _layer1_pre(x32, w1, b1):
    """h = b1; h = fmaf(x[i], w1[i, k], h) for i in order: pol_layer1 and the backward's recomputation."""
    pre = Bounded(np.broadcast_to(b1.astype(np.float64), (x32.shape[0], H1)))
    for i in range(x32.shape[1]):
        pre = fma(x32[:, i:i + 1].astype(np.float64), w1[i][None, :].astype(np.float64), pre)
    return pre


def check_layer1(P, x32, h1b):
    """h1_bf16 against tanh(x W1 + b1) in FP64: the FMA chain, tanh.approx, then the BF16 rounding U_BF16 |t|."""
    t = tanh_approx(_layer1_pre(x32, P['w1'], P['b1']))
    return ratio(h1b, Bounded(t.v, t.e + U_BF16 * (np.abs(t.v) + t.e)))


def check_layer2(P, h1b, h2):
    """h2 against tanh(sum_k h1_bf16[k] bf16(W2[k, n]) + b2[n]) in FP64: 256 exact products accumulated on the tensor
    core (TC_ULP per addition), the FP32 add of b2, tanh.approx; plus one ulp for a recovered h2 that two FP32 values
    would reproduce."""
    w2b = bf16(P['w2']).astype(np.float64)
    h = h1b.astype(np.float64)
    z = Bounded(h @ w2b, H1 * TC_ULP * (np.abs(h) @ np.abs(w2b)))
    t = tanh_approx(add(z, P['b2'].astype(np.float64)))
    return ratio(h2, Bounded(t.v, t.e + ULP32 * np.abs(t.v)))


def head_partials(P, h2, n_out):
    """pol_head_partial / pol_head_combine: four partial sums over 32 columns each (part 0 starts at b3), each an FMA
    chain in column order, then added in part order."""
    nout1 = n_out + 1
    w3 = P['w3'].astype(np.float64)
    h = Bounded(h2.astype(np.float64), ULP32 * np.abs(h2.astype(np.float64)))
    parts = []
    for q in range(4):
        acc = Bounded(np.broadcast_to(P['b3'].astype(np.float64) if q == 0 else np.zeros(nout1), (h2.shape[0], nout1)))
        for c in range(32 * q, 32 * q + 32):
            acc = fma(h[:, c:c + 1], w3[c][None, :], acc)
        parts.append(acc)
    return add(add(add(parts[0], parts[1]), parts[2]), parts[3])


def check_head(P, h2, out, n_out):
    """out = b3 + sum_c h2[c] w3[c, o] in the kernel's summation order, to its FP32 bound."""
    return ratio(out, head_partials(P, h2, n_out))


# ---- backward stages ---------------------------------------------------------------------------------------------
def check_head_backward(P, h2, dout, dz2):
    """dz2 = (sum_o dout[o] w3[c, o]) (1 - h2^2): the FMA chain over o, then h2 * h2, 1 - that, the product."""
    w3 = P['w3'].astype(np.float64)
    dh = Bounded(np.zeros(h2.shape))
    for o in range(dout.shape[1]):
        dh = fma(dout[:, o:o + 1].astype(np.float64), w3[:, o][None, :], dh)
    h = Bounded(h2.astype(np.float64), ULP32 * np.abs(h2.astype(np.float64)))
    return ratio(dz2, mul(dh, sub(1.0, mul(h, h))))


def check_layer1_backward(P, x32, dz2, dz1):
    """dz1 = dh1 (1 - h1^2) with dh1 = sum_n bf16(dz2[n]) bf16(W2[k, n]) (128 exact products on the tensor core,
    TC_ULP per addition) and h1 the FP32 tanh.approx of the forward's FMA chain."""
    w2b = bf16(P['w2']).astype(np.float64)
    d = bf16(dz2).astype(np.float64)
    dh1 = Bounded(d @ w2b.T, H2 * TC_ULP * (np.abs(d) @ np.abs(w2b).T))
    h = tanh_approx(_layer1_pre(x32, P['w1'], P['b1']))
    return ratio(dz1, mul(dh1, sub(1.0, mul(h, h))))


def check_sample_stages(params, obs_dim, n_out, x32, grads, out):
    """Every loss-independent check of one-sample gradients `grads` [rows, n_params] of observations x32 [rows, obs_dim]
    with head outputs `out` [rows, n_out + 1].  Returns (name -> worst ratio, with 'exact' the count of broken
    identities), and the split intermediates of the live rows (split_sample_grads: rows with a non-zero dout)."""
    P = split_flat(f32(params), obs_dim, n_out)
    st = split_sample_grads(grads, obs_dim, n_out)
    x32 = f32(x32)
    exact = check_exact(st, x32)
    live = st['live']
    st = {k: (v[live] if k != 'live' else v) for k, v in st.items()}
    x32, out = x32[live], out[live]
    r = {'exact': exact,
         'layer1': check_layer1(P, x32, st['h1b']),
         'layer2': check_layer2(P, st['h1b'], st['h2']),
         'head': check_head(P, st['h2'], out, n_out),
         'head_backward': check_head_backward(P, st['h2'], st['dout'], st['dz2']),
         'layer1_backward': check_layer1_backward(P, x32, st['dz2'], st['dz1'])}
    return r, st


# ---- the PPO loss stage ------------------------------------------------------------------------------------------
LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)
GAUSS_ENTROPY = 0.5 + LOG_SQRT_2PI


class PpoCoeffs(object):
    """The loss's FP32 hyper-parameters as the kernel receives them."""

    def __init__(self, clip, vf_clip, vf_coeff, ent_coeff, kl_coeff):
        self.clip, self.vf_clip, self.vf_coeff, self.ent_coeff, self.kl_coeff = [float(np.float32(v)) for v in (clip, vf_clip, vf_coeff, ent_coeff, kl_coeff)]

    def only(self, term):
        """The same clips with one loss coefficient kept and the others 0 ('surrogate' keeps none of them)."""
        keep = {'surrogate': (0, 0, 0), 'kl': (0, 0, self.kl_coeff), 'entropy': (0, self.ent_coeff, 0), 'value': (self.vf_coeff, 0, 0)}[term]
        return PpoCoeffs(self.clip, self.vf_clip, *keep)


def _const(c):
    """A float literal of the kernel: the exact constant, off by its FP32 rounding."""
    return Bounded(c, U32 * abs(c))


def ppo_reference(out, inp, cf, discrete, n_out, inv_n=1.0):
    """The PPO loss stage of ppo_grad_kernel for each row, on the kernel's head outputs `out` [rows, n_out + 1]:
    Bounded dout [rows, n_out + 1], the six statistics and the FP64 branch quantities.  `inp` holds the row inputs
    as the kernel reads them: actions (int64 [rows] | float64 [rows, n_out]), logp_old, value_old, logits_old
    [rows, n_out + 1], adv, vtarg (float32)."""
    rows = out.shape[0]
    o64 = out.astype(np.float64)
    old64 = f32(inp['logits_old']).astype(np.float64)
    s = Bounded(np.full(rows, inv_n), U32 * inv_n if inv_n != 1.0 else 0.0)
    v = Bounded(o64[:, n_out])
    logp, kl, ent = Bounded(np.zeros(rows)), Bounded(np.zeros(rows)), Bounded(np.zeros(rows))
    if discrete:
        act = np.asarray(inp['actions'], dtype=np.int64)
        mx, mo = Bounded(o64[:, :n_out].max(axis=1)), Bounded(old64[:, :n_out].max(axis=1))
        se, so = Bounded(np.zeros(rows)), Bounded(np.zeros(rows))
        for o in range(n_out):
            se = add(se, expf(sub(o64[:, o], mx), intrinsic=True))
            so = add(so, expf(sub(old64[:, o], mo), intrinsic=True))
        lse, lseo = add(mx, logf_intrinsic(se)), add(mo, logf_intrinsic(so))
        lp, p, po = [], [], []
        for o in range(n_out):
            lp.append(sub(o64[:, o], lse))
            lpo = sub(old64[:, o], lseo)
            p.append(expf(lp[o]))
            po.append(expf(lpo))
            kl = add(kl, mul(po[o], sub(lpo, lp[o])))
            ent = sub(ent, mul(p[o], lp[o]))
        logp = where(act == 0, lp[0], Bounded(np.zeros(rows)))
        for o in range(1, n_out):
            logp = where(act == o, lp[o], logp)
    else:
        ac = f32(inp['actions']).astype(np.float64)
        mu, muo = [], []
        for o in range(n_out):
            mu.append(tanh_approx(Bounded(o64[:, o])))
            muo.append(tanh_approx(Bounded(old64[:, o])))
            d = sub(ac[:, o], mu[o])
            logp = add(logp, sub(mul(mul(-0.5, d), d), _const(LOG_SQRT_2PI)))
            dm = sub(muo[o], mu[o])
            kl = add(kl, mul(mul(0.5, dm), dm))
        ent = mul(float(n_out), _const(GAUSS_ENTROPY))
    A, R, vold = [Bounded(f32(inp[k]).astype(np.float64)) for k in ('adv', 'vtarg', 'value_old')]
    r = expf(sub(logp, f32(inp['logp_old']).astype(np.float64)))
    lo, hi = Bounded(1.0 - cf.clip, U32), Bounded(1.0 + cf.clip, U32)
    rc = where(r.v < lo.v, lo, where(r.v > hi.v, hi, r))
    s1, s2 = mul(A, r), mul(A, rc)
    g_logp = where(s1.v <= s2.v, neg(mul(A, r)), 0.0)
    dvR = sub(v, R)
    vf1 = mul(dvR, dvR)
    dv = sub(v, vold)
    vfc = Bounded(cf.vf_clip)
    dvc = where(dv.v < -vfc.v, neg(vfc), where(dv.v > vfc.v, vfc, dv))
    vcl = add(vold, dvc)
    dcR = sub(vcl, R)
    vf2 = mul(dcR, dcR)
    inside = np.abs(dv.v) <= cf.vf_clip
    # inside the value clip vcl = v exactly in FP64, and the kernel may take either branch on the FP32 rounding of
    # vf1 against vf2: 2 (v - R) and 2 (vcl - R) then differ by vcl's rounding, which the vcl path's bound covers
    g_in = Bounded(2.0 * dvR.v, np.maximum(mul(2.0, dvR).e, mul(2.0, dcR).e + 2.0 * np.abs(dcR.v - dvR.v)))
    g_v = where(inside, g_in, where(vf1.v >= vf2.v, mul(2.0, dvR), 0.0))
    dout = []
    for o in range(n_out):
        if discrete:
            onehot = (act == o).astype(np.float64)
            t1 = mul(g_logp, sub(onehot, p[o]))
            t2 = mul(cf.kl_coeff, sub(p[o], po[o]))
            t3 = mul(mul(cf.ent_coeff, p[o]), add(lp[o], ent))
            dout.append(mul(s, add(add(t1, t2), t3)))
        else:
            t1 = mul(g_logp, sub(ac[:, o], mu[o]))
            t2 = mul(cf.kl_coeff, sub(mu[o], muo[o]))
            om = sub(1.0, mul(mu[o], mu[o]))
            dout.append(mul(mul(s, add(t1, t2)), om))
    dout.append(mul(mul(s, cf.vf_coeff), g_v))
    stats = [neg(minimum(s1, s2)), maximum(vf1, vf2), kl, ent,
             Bounded((np.abs(r.v - 1.0) > cf.clip).astype(np.float64)), r]
    branch = {'r': r.v, 'adv': A.v, 'dv': dv.v, 'vf1': vf1.v, 'vf2': vf2.v}
    return _stack(dout), stats, branch


def _stack(bs):
    return Bounded(np.stack([b.v for b in bs], axis=1), np.stack([b.e for b in bs], axis=1))


def check_ppo_loss(out, dout, stats, inp, cf, discrete, n_out):
    """dout (the sample's db3) and the six statistics against ppo_reference: {'ppo_loss', 'ppo_stats'}, plus the
    Bounded dout reference and the branch quantities."""
    ref, st_ref, branch = ppo_reference(out, inp, cf, discrete, n_out)
    stats = np.asarray(stats)
    r_stats = max(ratio(stats[:, i], st_ref[i]) for i in range(6))
    return {'ppo_loss': ratio(dout, ref), 'ppo_stats': r_stats}, ref, branch


def ppo_branches(branch, cf):
    """Branch labels and margins of each row, from ppo_reference's FP64 quantities.  Labels: 'ratio' in {'inside',
    'above', 'below'}, 'adv_pos', 'value' in {'inside', 'vf1_ge_vf2', 'vf1_lt_vf2'}.  Margins (relative distance to
    the nearest boundary): r = 1 +- clip, |dv| = vf_clip, and vf1 = vf2 on rows outside the value clip (inside it the
    two branches give the same gradient, see ppo_reference)."""
    r, dv, vf1, vf2 = branch['r'], branch['dv'], branch['vf1'], branch['vf2']
    ratio_lab = np.where(r > 1 + cf.clip, 'above', np.where(r < 1 - cf.clip, 'below', 'inside'))
    inside = np.abs(dv) <= cf.vf_clip
    value_lab = np.where(inside, 'inside', np.where(vf1 >= vf2, 'vf1_ge_vf2', 'vf1_lt_vf2'))
    m_r = np.minimum(np.abs(r - (1 - cf.clip)), np.abs(r - (1 + cf.clip))) / cf.clip
    m_v = np.abs(np.abs(dv) - cf.vf_clip) / cf.vf_clip
    m_vf = np.where(inside, np.inf, np.abs(vf1 - vf2) / np.maximum(np.maximum(vf1, vf2), 1e-30))
    return {'ratio': ratio_lab, 'adv_pos': branch['adv'] > 0, 'value': value_lab,
            'margin': float(min(m_r.min(), m_v.min(), m_vf.min()))}


# ---- the DQN loss stage ------------------------------------------------------------------------------------------
def q_values32(head, n_out):
    """dqn_q_values in FP32: Q = V + (A - sum(A) / n_out), the sum in column order; the greedy action is the first
    maximum."""
    head = f32(head)
    sa = np.zeros(head.shape[0], dtype=np.float32)
    for o in range(n_out):
        sa = f32(sa + head[:, o])
    ma = f32(sa / np.float32(n_out))
    q = f32(head[:, n_out:n_out + 1] + f32(head[:, :n_out] - ma[:, None]))
    return q, q.argmax(axis=1)


def _q_bounded(head, n_out):
    h = head.astype(np.float64)
    sa = Bounded(np.zeros(h.shape[0]))
    for o in range(n_out):
        sa = add(sa, h[:, o])
    ma = Bounded(sa.v / n_out, sa.e / n_out + U32 * (np.abs(sa.v) / n_out + sa.e / n_out))   # one FP32 division
    return [add(h[:, n_out], sub(h[:, o], ma)) for o in range(n_out)]


def dqn_reference(out, next_online, next_target, inp, gamma, n_out, inv_n=1.0):
    """The DQN loss stage for each row on the kernel's head outputs (s) and its forward outputs on s' under the online
    and the target parameters: Bounded dout, the four statistics, the FP64 td, and the FP32 replica (qsa, y, dout)
    that the kernel's arithmetic gives bit for bit."""
    rows = out.shape[0]
    act = np.asarray(inp['actions'], dtype=np.int64)
    reward = f32(inp['reward'])
    nd = np.where(np.asarray(inp['done']) != 0, 0.0, 1.0)
    q = _q_bounded(out, n_out)
    qt = _q_bounded(next_target, n_out)
    _, an = q_values32(next_online, n_out)
    qsa, qn = _pick(q, act), _pick(qt, an)
    y = add(reward.astype(np.float64), mul(mul(float(np.float32(gamma)), nd), qn))
    td = sub(qsa, y)
    g = where(td.v < -1, -1.0, where(td.v > 1, 1.0, td))
    s = Bounded(np.full(rows, inv_n), U32 * inv_n if inv_n != 1.0 else 0.0)
    g = mul(g, s)
    inv_nout = Bounded(1.0 / n_out, U32 / n_out)
    dout = [mul(g, sub((act == o).astype(np.float64), inv_nout)) for o in range(n_out)] + [g]
    atd = absb(td)
    huber = where(atd.v <= 1, mul(mul(0.5, td), td), sub(atd, 0.5))
    # FP32 replica
    q32, _ = q_values32(out, n_out)
    qt32, _ = q_values32(next_target, n_out)
    qsa32 = q32[np.arange(rows), act]
    y32 = f32(reward + f32(f32(np.float32(gamma) * f32(nd)) * qt32[np.arange(rows), an]))
    td32 = f32(qsa32 - y32)
    g32 = f32(np.clip(td32, -1, 1) * np.float32(inv_n))
    inv32 = np.float32(1) / np.float32(n_out)
    dout32 = np.concatenate([f32(g32[:, None] * f32((act[:, None] == np.arange(n_out)[None, :]).astype(np.float32) - inv32)),
                             g32[:, None]], axis=1)
    replica = {'qsa': qsa32, 'y': y32, 'dout': dout32, 'an': an}
    return _stack(dout), [huber, atd, qsa, y], td.v, replica


def _pick(qs, idx):
    out = qs[0]
    for o in range(1, len(qs)):
        out = where(idx == o, qs[o], out)
    return out


def check_dqn_loss(out, next_online, next_target, dout, stats, inp, gamma, n_out):
    """dout and the four statistics against dqn_reference in FP64, and Q(s, a), y and dout bit for bit against the
    FP32 replica: {'dqn_loss', 'dqn_stats'} (inf where a bitwise identity breaks), plus the FP64 td and the replica."""
    ref, st_ref, td, rep = dqn_reference(out, next_online, next_target, inp, gamma, n_out)
    stats = np.asarray(stats)
    r_loss = ratio(dout, ref)
    if not np.array_equal(f32(dout), rep['dout']):
        r_loss = float('inf')
    r_stats = max(ratio(stats[:, i], st_ref[i]) for i in range(4))
    if not (np.array_equal(f32(stats[:, 2]), rep['qsa']) and np.array_equal(f32(stats[:, 3]), rep['y'])):
        r_stats = float('inf')
    return {'dqn_loss': r_loss, 'dqn_stats': r_stats}, td, rep


# ---- row recipes -------------------------------------------------------------------------------------------------
def ppo_logp64(out, actions, discrete, n_out):
    """The log-probability of each row's action under the head outputs, in FP64."""
    o = out[:, :n_out].astype(np.float64)
    if discrete:
        m = o.max(axis=1, keepdims=True)
        lsm = o - m - np.log(np.exp(o - m).sum(axis=1, keepdims=True))
        return lsm[np.arange(len(o)), actions]
    a = f32(actions).astype(np.float64)
    return (-0.5 * (a - np.tanh(o)) ** 2 - LOG_SQRT_2PI).sum(axis=1)


# ratio targets: inside at 1 -+ 0.4 clip, outside at 1 -+ 2 clip; |dv| at 0.3 vf_clip inside, 2 vf_clip outside
PPO_RATIO_CATS = (('inside', 1), ('inside', -1), ('above', 1), ('above', -1), ('below', 1), ('below', -1))
PPO_VALUE_CATS = ('inside', 'vf1_ge_vf2', 'vf1_lt_vf2')


def ppo_rows(out, n_out, discrete, cf, seed):
    """Inputs for rows whose head outputs are `out`: row j takes action j mod n_out (discrete) or tanh(mean) + unit
    noise, the (ratio, sign of A) category j mod 6 and the value category (j // 6) mod 3.  logp_old, value_old and
    vtarg are set from `out` so that the ratio and the value clip land where the category says."""
    rng = np.random.default_rng(seed)
    rows = out.shape[0]
    j = np.arange(rows)
    o64 = out.astype(np.float64)
    if discrete:
        actions = (j % n_out).astype(np.int64)
    else:
        actions = np.tanh(o64[:, :n_out]) + rng.standard_normal((rows, n_out))
    logp = ppo_logp64(out, actions, discrete, n_out)
    cat = [PPO_RATIO_CATS[k % 6] for k in j]
    target = np.array([{'inside': 1 + 0.4 * cf.clip * sg, 'above': 1 + 2 * cf.clip, 'below': 1 - 2 * cf.clip}[c]
                       for c, sg in cat])
    sign = np.array([sg for _, sg in cat], dtype=np.float64)
    adv = sign * rng.uniform(0.5, 1.5, rows)
    v = o64[:, n_out]
    vcat = [PPO_VALUE_CATS[(k // 6) % 3] for k in j]
    side = np.where(rng.uniform(size=rows) < 0.5, -1.0, 1.0)           # sign of v - v_old
    dv = np.array([0.3 if c == 'inside' else 2.0 for c in vcat]) * cf.vf_clip * side
    vold = v - dv
    vcl = vold + np.clip(dv, -cf.vf_clip, cf.vf_clip)
    vtarg = np.where(np.array(vcat) == 'inside', v + rng.uniform(-1, 1, rows),
                     np.where(np.array(vcat) == 'vf1_ge_vf2', vcl - side * 0.3 * cf.vf_clip, v + side * 0.3 * cf.vf_clip))
    logits_old = f32(out + 0.3 * rng.standard_normal(out.shape))
    return {'actions': actions, 'logp_old': f32(logp - np.log(target)), 'value_old': f32(vold), 'logits_old': logits_old,
            'adv': f32(adv), 'vtarg': f32(vtarg)}


def dqn_rows(out, next_online, next_target, n_out, gamma, seed):
    """Inputs for rows with head outputs `out` on s and `next_*` on s': action j mod n_out, done on every third row, and
    the reward set so that td = Q(s, a) - y is +-(0.2 .. 0.8) on even rows and +-(1.5 .. 3) on odd rows."""
    rng = np.random.default_rng(seed)
    rows = out.shape[0]
    j = np.arange(rows)
    actions = (j % n_out).astype(np.int64)
    done = (j % 3 == 0).astype(np.uint8)
    q, _ = q_values32(out, n_out)
    qt, _ = q_values32(next_target, n_out)
    _, an = q_values32(next_online, n_out)
    mag = np.where(j % 2 == 0, rng.uniform(0.2, 0.8, rows), rng.uniform(1.5, 3.0, rows))
    td = mag * np.where(rng.uniform(size=rows) < 0.5, -1.0, 1.0)
    y = q[j, actions].astype(np.float64) - td
    reward = y - gamma * (1.0 - done) * qt[j, an].astype(np.float64)
    return {'actions': actions, 'reward': f32(reward), 'done': done}


# ---- minibatch gradient = sum of one-sample gradients ------------------------------------------------------------
def sum_factors(n_ctas):
    """Per-tensor relative factors of the bound |grad_n - sum_j g_j / n| <= f * sum_j |g_j| / n for n a power of two
    (every per-sample value scales exactly by 2^-m): the in-CTA sum over up to 128 samples (FP32 FMA / add chains, or
    the tensor core for dW2), one rounding of the exact product in place of the one-sample gradient's fl(product), and
    ppo_reduce_kernel's chain over n_ctas partials."""
    f = gamma(H2 + 1 + n_ctas)
    return {'w1': f, 'b1': f, 'w2': H2 * TC_ULP + gamma(n_ctas + 1), 'b2': f, 'w3': f, 'b3': f}


def ragged_factors(n_out):
    """For n not a power of two, inv_n = fl(1 / n) and every per-sample value is rounded anew.  Extra relative terms of
    the bound, per row, against the one-sample value over n:
      'dout'  dout = fl(fl(inv_n) E) or fl(fl(inv_n E1) E2): at most 4 roundings (w3, b3, relative to |g_j|);
      'dz2'   dz2 = fl(fl(dh) (1 - h2^2)), dh an FMA chain of n_out + 1 terms: 'dout' + both chains' gamma(n_out + 1) + two
              roundings, relative to M_b2 = (1 - h2^2) sum_o |dout[o] w3[c, o]| (b2);
      'dz2b'  the BF16 copies of dz2: two BF16 roundings on top, with |dz2| <= M_b2 (1 + gamma(n_out + 2)) < M_b2
              (1 + 2^-9) (w2, relative to |h1_bf16| M_b2);
      'dz1'   dh1 = bf16(dz2) W2^T carries 'dz2b' through |bf16(W2)|, plus both sides' tensor-core accumulation
              (H2 TC_ULP each, on sum_n |bf16(dz2)| |W2| with |bf16(dz2)| < M_b2 (1 + 2^-7)) and two roundings each side
              of dz1 = fl(dh1 (1 - h1^2)), 1 - h1^2 <= 1 (b1, relative to M_b2 |bf16(W2)|^T);
      'x_dz1' 'dz1' and the rounding of fl(x dz1) (w1, relative to |x| M_b2 |bf16(W2)|^T)."""
    dout = 4 * U32
    dz2 = dout + 2 * gamma(n_out + 1) + 2 * U32
    dz2b = 2 * U_BF16 * (1 + 2.0 ** -9) + dz2
    dz1 = dz2b + (2 * H2 * TC_ULP + 4 * U32) * (1 + 2.0 ** -7)
    return {'dout': dout, 'dz2': dz2, 'dz2b': dz2b, 'dz1': dz1, 'x_dz1': dz1 + U32}
