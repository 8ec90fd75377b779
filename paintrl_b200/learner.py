"""What the PPO and the DQN learners share: the flat-parameter network contract of the learner kernel
(csrc/paintrl_learn.cuh), their configuration rules, and the device state and handle lifecycle of a learner.

The network is the rollout policy's MLP (`rollout.MlpPolicy`, hidden layers 256 and 128), trained as one flat float32
vector w1 | b1 | w2 | b2 | w3 | b3, each row-major.  `ppo.PPOLearner` and `dqn.DQNLearner` subclass `Learner`.
"""
import ctypes

import torch

from . import _capi


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


def check_state_dict(sd, obs_dim, n_out, discrete, tensors):
    """Raise ValueError when a learner state does not fit a policy of this shape: its shape fields, the flat vectors
    named in `tensors` and the step count."""
    if (sd.get('obs_dim'), sd.get('n_out'), bool(sd.get('discrete'))) != (obs_dim, n_out, bool(discrete)):
        raise ValueError('checkpoint is for obs_dim %r, n_out %r, discrete %r' % (sd.get('obs_dim'), sd.get('n_out'), sd.get('discrete')))
    n = num_params(obs_dim, n_out)
    for k in tensors:
        if k not in sd or tuple(sd[k].shape) != (n,):
            raise ValueError('%s has shape %s, expected (%d,)' % (k, tuple(sd[k].shape) if k in sd else None, n))
    if int(sd['step']) < 0:
        raise ValueError('step must be non-negative')


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


class LearnerConfig(object):
    """Hyper-parameters: the subclass's _DEFAULTS, each converted to its default's type.  minibatch_size must be a
    positive multiple of 128; subclasses add their own rules in `_check`."""
    _DEFAULTS = {}

    def __init__(self, **kw):
        unknown = set(kw) - set(self._DEFAULTS)
        if unknown:
            raise TypeError('unknown %s fields: %s' % (type(self).__name__, sorted(unknown)))
        for k, v in self._DEFAULTS.items():
            setattr(self, k, type(v)(kw.get(k, v)))
        if self.minibatch_size <= 0 or self.minibatch_size % 128:
            raise ValueError('minibatch_size must be a positive multiple of 128 (one learner CTA per 128 samples)')
        self._check()

    def _check(self):
        pass

    def to_dict(self):
        return {k: getattr(self, k) for k in self._DEFAULTS}

    @classmethod
    def from_dict(cls, d):
        return cls(**d)

    def __repr__(self):
        return '%s(%s)' % (type(self).__name__, ', '.join('%s=%r' % kv for kv in self.to_dict().items()))


class Learner(object):
    """Trains `policy` (a `rollout.MlpPolicy`) in place on one CUDA device: the flat parameters, Adam's moments, a
    gradient buffer, a seeded device generator and a native learner handle.  A subclass names its handle's C create and
    destroy functions and builds their config in `_c_config`."""
    _CREATE = _DESTROY = None

    def __init__(self, policy, config):
        check_policy(policy)
        self.cfg = config
        self.policy = policy
        self.device = torch.device(policy.device)
        if self.device.type != 'cuda':
            raise ValueError('the learner runs on a CUDA device (no CPU fallback)')
        self.obs_dim, self.n_out, self.discrete = policy.obs_dim, policy.n_out, bool(policy.discrete)
        self.dist = getattr(policy, 'dist', None) or ('categorical' if self.discrete else 'tanh_gaussian')
        self._lib = _capi.lib()
        self.n_params = num_params(self.obs_dim, self.n_out)
        self.params = flat_params(policy).to(self.device)
        self.m = torch.zeros_like(self.params)
        self.v = torch.zeros_like(self.params)
        self.grad = torch.zeros_like(self.params)
        self.step = 0                              # Adam's step count
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(self.cfg.seed)
        handle = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _capi.check(getattr(self._lib, self._CREATE)(ctypes.byref(self._c_config()), index, ctypes.byref(handle)))
        self._h = handle

    def _c_config(self):
        raise NotImplementedError

    def close(self):
        if getattr(self, '_h', None):
            getattr(self._lib, self._DESTROY)(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def adam(self, grad):
        self.step += 1
        c = self.cfg
        _capi.check(self._lib.paintrl_adam_step(_ptr(self.params), _ptr(grad), _ptr(self.m), _ptr(self.v), self.n_params, c.lr,
                                                c.adam_beta1, c.adam_beta2, c.adam_eps, self.step, self._stream()))

    def _state_dict(self):
        return {'config': self.cfg.to_dict(), 'obs_dim': self.obs_dim, 'n_out': self.n_out, 'discrete': self.discrete,
                'params': self.params.cpu(), 'adam_m': self.m.cpu(), 'adam_v': self.v.cpu(), 'step': int(self.step),
                'generator': self.gen.get_state()}

    def _load_state_dict(self, sd):
        """The shared half of load_state_dict, after the subclass has checked sd and loaded its own fields: parameters,
        Adam state and generator, then the parameters pushed into the policy and its native act kernel."""
        self.params.copy_(sd['params'])
        self.m.copy_(sd['adam_m'])
        self.v.copy_(sd['adam_v'])
        self.step = int(sd['step'])
        self.gen.set_state(sd['generator'])
        unflatten_into(self.policy, self.params)
        if getattr(self.policy, 'native', None) is not None:
            self.policy.native.set_params(self.params)
