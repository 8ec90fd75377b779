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
import torch

from . import _capi
from .learner import Learner, LearnerConfig, _ptr, check_policy, flat_params, num_params, unflatten_into  # noqa: F401
from .learner import check_state_dict as _check_state_dict
from .rollout import gae

# RLlib PPO's loss and optimiser defaults; num_sgd_iter is paint_ppo.py's (BASELINE.md section 1: train batch 1500,
# SGD minibatch 64 x 16 iterations).  The reference's minibatch of 64 becomes a multiple of 128 here (one kernel CTA
# per 128 samples); thousands of environments give fragments of hundreds of thousands of samples.
_DEFAULTS = dict(lr=5e-5, clip_param=0.3, vf_clip_param=10.0, vf_loss_coeff=1.0, entropy_coeff=0.0, kl_coeff=0.2,
                 kl_target=0.01, gamma=0.99, lam=1.0, num_sgd_iter=16, minibatch_size=4096, adam_beta1=0.9,
                 adam_beta2=0.999, adam_eps=1e-8, seed=0)
STAT_NAMES = ('policy_loss', 'vf_loss', 'kl', 'entropy', 'clip_fraction', 'mean_ratio')


class PPOConfig(LearnerConfig):
    """Hyper-parameters of `PPOLearner`.  Defaults: RLlib PPO (clip 0.3, vf_clip 10, vf_loss_coeff 1, entropy 0,
    kl_coeff 0.2 adapted toward kl_target 0.01, gamma 0.99, lambda 1.0, Adam lr 5e-5) and paint_ppo.py's 16 SGD
    iterations; minibatch_size must be a positive multiple of 128."""
    _DEFAULTS = _DEFAULTS

    def _check(self):
        if self.num_sgd_iter <= 0:
            raise ValueError('num_sgd_iter must be positive')


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


class PPOLearner(Learner):
    """PPO over fragments of a `RolloutWorker(..., keep_logits=True)`, training `policy` (an `rollout.MlpPolicy`) in
    place: its torch tensors and, when enabled, its native act kernel's weights follow every update."""
    _CREATE, _DESTROY = 'paintrl_ppo_create', 'paintrl_ppo_destroy'

    def __init__(self, policy, config=None):
        super().__init__(policy, config if config is not None else PPOConfig())
        self.kl_coeff = float(self.cfg.kl_coeff)

    def _c_config(self):
        c = self.cfg
        return _capi.PaintrlPpoConfig(_capi.PAINTRL_ABI_VERSION, self.obs_dim, self.n_out, int(self.discrete), c.minibatch_size,
                                      c.clip_param, c.vf_clip_param, c.vf_loss_coeff, c.entropy_coeff)

    def forward(self, obs, idx):
        """The learner kernel's forward pass on rows `idx` (int32) of `obs` (float64 [rows, obs_dim]): float32
        [len(idx), n_out + 1], logits | means then the value (for tests: equals the act kernel's logits bit for bit)."""
        out = torch.empty(idx.numel(), self.n_out + 1, dtype=torch.float32, device=self.device)
        for s, n in minibatches(idx.numel(), self.cfg.minibatch_size):
            _capi.check(self._lib.paintrl_ppo_forward(self._h, _ptr(self.params), _ptr(idx[s:]), n, _ptr(obs), _ptr(out[s:]), self._stream()))
        return out

    def grad_into(self, rows, idx, kl_coeff, grad, stats):
        """One `paintrl_ppo_grad` call (`paintrl_ppo_grad_diag_gaussian` for a diagonal-Gaussian policy): `rows` is the
        dict `flatten()` returns."""
        fn = self._lib.paintrl_ppo_grad_diag_gaussian if self.dist == 'diag_gaussian' else self._lib.paintrl_ppo_grad
        _capi.check(fn(
            self._h, _ptr(self.params), _ptr(idx), idx.numel(), _ptr(rows['obs']), _ptr(rows['actions']), _ptr(rows['logp']),
            _ptr(rows['value']), _ptr(rows['logits']), _ptr(rows['adv']), _ptr(rows['vtarg']), float(kl_coeff), _ptr(grad),
            _ptr(stats), self._stream()))

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
        return dict(self._state_dict(), kl_coeff=float(self.kl_coeff), dist=self.dist)

    def load_state_dict(self, sd):
        check_state_dict(sd, self.obs_dim, self.n_out, self.discrete, self.dist)
        self.kl_coeff = float(sd['kl_coeff'])
        self._load_state_dict(sd)


def state_dist(sd):
    """The action distribution a PPO learner state was trained with; states written before `dist` was recorded hold
    the distribution every policy had then."""
    return sd.get('dist') or ('categorical' if sd.get('discrete') else 'tanh_gaussian')


def check_state_dict(sd, obs_dim, n_out, discrete, dist=None):
    """Raise ValueError when a learner state does not fit a policy of this shape (and of distribution `dist`, when
    given)."""
    _check_state_dict(sd, obs_dim, n_out, discrete, ('params', 'adam_m', 'adam_v'))
    if not float(sd['kl_coeff']) >= 0.0:
        raise ValueError('kl_coeff must be non-negative')
    if dist is not None and state_dist(sd) != dist:
        raise ValueError('checkpoint is for the %s distribution, not %s' % (state_dist(sd), dist))
