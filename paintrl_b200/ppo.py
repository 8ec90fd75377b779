"""PPO on the GPU: the learner of the reference's training script (paint_ppo.py trains RLlib's PPO, ray 0.x
`ppo_policy`), with its hot path in this repository's own kernels (csrc/paintrl_learn.cuh).

Per minibatch the learner issues three launches' worth of C ABI calls, all asynchronous on the current stream:
`paintrl_ppo_grad` (forward, loss and backward of the minibatch in one kernel, plus a fixed-order sum of the per-CTA
partial gradients), `paintrl_adam_step`, and `paintrl_policy_set_params`, which packs the new parameters into the rollout
policy kernel's weights in place -- so a `RolloutWorker` graph captured before the update samples with the new weights
on its next replay, without recapture.  `update()` reads the statistics back once, at its end; that is its only host
synchronisation.

    worker = RolloutWorker(env, policy, fragment_length=100, use_cuda_graph=True, keep_logits=True)
    learner = PPOLearner(policy, PPOConfig(minibatch_size=4096))
    frag, rollout_stats = worker.collect()
    learn_stats = learner.update(frag)
"""
import ctypes

import torch

from . import _capi
from .rollout import gae

# RLlib PPO's loss and optimiser defaults; num_sgd_iter is paint_ppo.py's (BASELINE.md section 1: train batch 1500,
# SGD minibatch 64 x 16 iterations).  The reference's minibatch of 64 becomes a multiple of 128 here (one kernel CTA
# per 128 samples); thousands of environments give fragments of hundreds of thousands of samples.
_DEFAULTS = dict(lr=5e-5, clip_param=0.3, vf_clip_param=10.0, vf_loss_coeff=1.0, entropy_coeff=0.0, kl_coeff=0.2,
                 kl_target=0.01, gamma=0.99, lam=1.0, num_sgd_iter=16, minibatch_size=4096, adam_beta1=0.9,
                 adam_beta2=0.999, adam_eps=1e-8, seed=0)
STAT_NAMES = ('policy_loss', 'vf_loss', 'kl', 'entropy', 'clip_fraction', 'mean_ratio')


class PPOConfig(object):
    """Hyper-parameters of `PPOLearner`.  Defaults: RLlib PPO (clip 0.3, vf_clip 10, vf_loss_coeff 1, entropy 0,
    kl_coeff 0.2 adapted toward kl_target 0.01, gamma 0.99, lambda 1.0, Adam lr 5e-5) and paint_ppo.py's 16 SGD
    iterations; minibatch_size must be a positive multiple of 128."""

    def __init__(self, **kw):
        unknown = set(kw) - set(_DEFAULTS)
        if unknown:
            raise TypeError('unknown PPOConfig fields: %s' % sorted(unknown))
        for k, v in _DEFAULTS.items():
            setattr(self, k, type(v)(kw.get(k, v)))
        if self.minibatch_size <= 0 or self.minibatch_size % 128:
            raise ValueError('minibatch_size must be a positive multiple of 128 (one learner CTA per 128 samples)')
        if self.num_sgd_iter <= 0:
            raise ValueError('num_sgd_iter must be positive')

    def to_dict(self):
        return {k: getattr(self, k) for k in _DEFAULTS}

    @classmethod
    def from_dict(cls, d):
        return cls(**d)

    def __repr__(self):
        return 'PPOConfig(%s)' % ', '.join('%s=%r' % kv for kv in self.to_dict().items())


def num_params(obs_dim, n_out):
    """Length of the flat parameter vector w1 | b1 | w2 | b2 | w3 | b3 (hidden layers 256, 128)."""
    return obs_dim * 256 + 256 + 256 * 128 + 128 + 128 * (n_out + 1) + (n_out + 1)


def check_policy(policy):
    """Raise ValueError for a policy the learner kernel does not take."""
    if len(policy.layers) != 2 or tuple(policy.layers[0][0].shape) != (policy.obs_dim, 256) or tuple(policy.layers[1][0].shape) != (256, 128):
        raise ValueError('the learner kernel takes hidden layers (256, 128) only')
    if not 1 <= policy.obs_dim <= 32:
        raise ValueError('the learner kernel takes observations of 1..32 entries, not %d' % policy.obs_dim)
    if not 1 <= policy.n_out <= 15:
        raise ValueError('the learner kernel takes 1..15 action outputs, not %d' % policy.n_out)


def flat_params(policy):
    return torch.cat([w.reshape(-1).to(torch.float32) for w in policy.weights()]).contiguous()


def unflatten_into(policy, params):
    """Copy a flat parameter vector into the policy's own tensors (asynchronous device copies)."""
    off = 0
    for w in policy.weights():
        w.copy_(params[off:off + w.numel()].view(w.shape))
        off += w.numel()


def minibatches(n_rows, size):
    """(start, n) of the minibatches of one epoch: consecutive slices of the permutation, the last one ragged."""
    return [(s, min(size, n_rows - s)) for s in range(0, n_rows, size)]


def adapt_kl(kl_coeff, kl, kl_target):
    """RLlib PPO's update_kl: x1.5 above twice the target, x0.5 below half of it."""
    if kl > 2.0 * kl_target:
        return kl_coeff * 1.5
    if kl < 0.5 * kl_target:
        return kl_coeff * 0.5
    return kl_coeff


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


class PPOLearner(object):
    """PPO over fragments of a `RolloutWorker(..., keep_logits=True)`, training `policy` (an `rollout.MlpPolicy`) in
    place: its torch tensors and, when enabled, its native act kernel's weights follow every update."""

    def __init__(self, policy, config=None):
        check_policy(policy)
        self.cfg = config if config is not None else PPOConfig()
        self.policy = policy
        self.device = torch.device(policy.device)
        if self.device.type != 'cuda':
            raise ValueError('the learner runs on a CUDA device (no CPU fallback)')
        self.obs_dim, self.n_out, self.discrete = policy.obs_dim, policy.n_out, bool(policy.discrete)
        self._lib = _capi.lib()
        self.n_params = num_params(self.obs_dim, self.n_out)
        self.params = flat_params(policy).to(self.device)
        self.m = torch.zeros_like(self.params)
        self.v = torch.zeros_like(self.params)
        self.grad = torch.zeros_like(self.params)
        self.step = 0
        self.kl_coeff = float(self.cfg.kl_coeff)
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(self.cfg.seed)
        c = self.cfg
        pc = _capi.PaintrlPpoConfig(_capi.PAINTRL_ABI_VERSION, self.obs_dim, self.n_out, int(self.discrete), c.minibatch_size,
                                    c.clip_param, c.vf_clip_param, c.vf_loss_coeff, c.entropy_coeff)
        handle = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _capi.check(self._lib.paintrl_ppo_create(ctypes.byref(pc), index, ctypes.byref(handle)))
        self._h = handle

    def close(self):
        if getattr(self, '_h', None):
            self._lib.paintrl_ppo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def forward(self, obs, idx):
        """The learner kernel's forward pass on rows `idx` (int32) of `obs` (float64 [rows, obs_dim]): float32
        [len(idx), n_out + 1], logits | means then the value (for tests: equals the act kernel's logits bit for bit)."""
        out = torch.empty(idx.numel(), self.n_out + 1, dtype=torch.float32, device=self.device)
        for s, n in minibatches(idx.numel(), self.cfg.minibatch_size):
            _capi.check(self._lib.paintrl_ppo_forward(self._h, _ptr(self.params), _ptr(idx[s:]), n, _ptr(obs), _ptr(out[s:]), self._stream()))
        return out

    def grad_into(self, rows, idx, kl_coeff, grad, stats):
        """One `paintrl_ppo_grad` call: `rows` is the dict `flatten()` returns."""
        _capi.check(self._lib.paintrl_ppo_grad(
            self._h, _ptr(self.params), _ptr(idx), idx.numel(), _ptr(rows['obs']), _ptr(rows['actions']), _ptr(rows['logp']),
            _ptr(rows['value']), _ptr(rows['logits']), _ptr(rows['adv']), _ptr(rows['vtarg']), float(kl_coeff), _ptr(grad),
            _ptr(stats), self._stream()))

    def adam(self, grad):
        self.step += 1
        c = self.cfg
        _capi.check(self._lib.paintrl_adam_step(_ptr(self.params), _ptr(grad), _ptr(self.m), _ptr(self.v), self.n_params, c.lr,
                                                c.adam_beta1, c.adam_beta2, c.adam_eps, self.step, self._stream()))

    def flatten(self, frag):
        """The fragment as T*B rows (views where the buffers allow) plus standardised advantages and value targets."""
        if getattr(frag, 'logits', None) is None:
            raise ValueError('the learner needs the fragment logits: collect with RolloutWorker(..., keep_logits=True)')
        T, B = frag.T, frag.B
        N = T * B
        adv, vtarg = gae(frag, self.cfg.gamma, self.cfg.lam)
        adv = (adv - adv.mean()) / adv.std(unbiased=False).clamp_min(1e-4)      # RLlib standardize_fields
        return {'n': N, 'obs': frag.obs[:T].reshape(N, -1), 'actions': frag.actions.reshape((N,) + tuple(frag.actions.shape[2:])),
                'logp': frag.logp.reshape(N), 'value': frag.value[:T].reshape(N), 'logits': frag.logits.reshape(N, -1),
                'adv': adv.reshape(N).contiguous(), 'vtarg': vtarg.reshape(N).contiguous()}

    @torch.no_grad()
    def update(self, frag):
        """num_sgd_iter epochs over the fragment, each a fresh device permutation cut into minibatches of
        minibatch_size (the last one ragged); grad -> Adam -> set_params per minibatch.  Returns the mean statistics
        over all minibatches (those of STAT_NAMES), the KL of the last epoch and the kl_coeff now in force."""
        rows = self.flatten(frag)
        N = rows['n']
        bounds = minibatches(N, self.cfg.minibatch_size)
        stats = torch.zeros(self.cfg.num_sgd_iter * len(bounds), 8, dtype=torch.float32, device=self.device)
        native = getattr(self.policy, 'native', None)
        k = 0
        for _ in range(self.cfg.num_sgd_iter):
            perm = torch.randperm(N, generator=self.gen, device=self.device).to(torch.int32)
            for s, n in bounds:
                self.grad_into(rows, perm[s:s + n], self.kl_coeff, self.grad, stats[k])
                self.adam(self.grad)
                if native is not None:
                    native.set_params(self.params)
                k += 1
        unflatten_into(self.policy, self.params)
        host = stats.cpu().numpy().astype('float64')
        out = {name: float(host[:, i].mean()) for i, name in enumerate(STAT_NAMES)}
        out['kl_last_epoch'] = float(host[-len(bounds):, 2].mean())
        out['kl_coeff_used'] = self.kl_coeff
        self.kl_coeff = adapt_kl(self.kl_coeff, out['kl_last_epoch'], self.cfg.kl_target)
        out['kl_coeff'] = self.kl_coeff
        out['minibatches'] = k
        out['samples'] = N
        return out

    def state_dict(self):
        return {'config': self.cfg.to_dict(), 'obs_dim': self.obs_dim, 'n_out': self.n_out, 'discrete': self.discrete,
                'params': self.params.cpu(), 'adam_m': self.m.cpu(), 'adam_v': self.v.cpu(), 'step': int(self.step),
                'kl_coeff': float(self.kl_coeff), 'generator': self.gen.get_state()}

    def load_state_dict(self, sd):
        check_state_dict(sd, self.obs_dim, self.n_out, self.discrete)
        self.params.copy_(sd['params'])
        self.m.copy_(sd['adam_m'])
        self.v.copy_(sd['adam_v'])
        self.step = int(sd['step'])
        self.kl_coeff = float(sd['kl_coeff'])
        self.gen.set_state(sd['generator'])
        unflatten_into(self.policy, self.params)
        if getattr(self.policy, 'native', None) is not None:
            self.policy.native.set_params(self.params)


def check_state_dict(sd, obs_dim, n_out, discrete):
    """Raise ValueError when a learner state does not fit a policy of this shape."""
    if (sd.get('obs_dim'), sd.get('n_out'), bool(sd.get('discrete'))) != (obs_dim, n_out, bool(discrete)):
        raise ValueError('checkpoint is for obs_dim %r, n_out %r, discrete %r' % (sd.get('obs_dim'), sd.get('n_out'), sd.get('discrete')))
    n = num_params(obs_dim, n_out)
    for k in ('params', 'adam_m', 'adam_v'):
        if tuple(sd[k].shape) != (n,):
            raise ValueError('%s has shape %s, expected (%d,)' % (k, tuple(sd[k].shape), n))
    if int(sd['step']) < 0 or not float(sd['kl_coeff']) >= 0.0:
        raise ValueError('step must be non-negative and kl_coeff non-negative')
