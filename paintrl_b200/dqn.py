"""Double DQN on the GPU: a device replay buffer, epsilon-greedy collection through the act kernel, and the learner
kernel's DQN loss stage (csrc/paintrl_learn.cuh), for discrete action spaces.

The network is the rollout policy's own MLP read as a dueling Q-network: the n_out head outputs are the advantages A,
the value column is V, and Q(s, a) = V + A_a - mean_o A_o (RLlib DQN's dueling combination; RLlib also adds a 256-unit
hidden layer per stream, which is left out here, so the flat parameter layout and the act kernel stay the PPO ones).

Per gradient step the learner issues, all asynchronous on the current stream: a seeded device `randint` of replay
rows, `paintrl_dqn_grad` (the head on s' under the online and the target parameters, then forward, Huber loss and
backward of the minibatch in one kernel, then the fixed-order sum of the per-CTA partials), `paintrl_clip_grad_norm`,
`paintrl_adam_step` and `paintrl_policy_set_params` -- so a `RolloutWorker` graph captured before the update acts with
the new weights on its next replay.  `update()` reads its statistics back once, at its end.

    eps = torch.ones(1, device='cuda')
    worker = RolloutWorker(env, policy, fragment_length=100, use_cuda_graph=True, epsilon=eps)
    learner = DQNLearner(policy, DQNConfig())
    eps.fill_(epsilon_at(learner.cfg, env_steps, total_samples))
    frag, rollout_stats = worker.collect()
    learn_stats = learner.update(frag)
"""
import math

import torch

from . import _capi
from .learner import Learner, LearnerConfig, _ptr, flat_params, unflatten_into  # noqa: F401
from .learner import check_state_dict as _check_state_dict

# RLlib DQN's defaults as recalled (lr 5e-4, Adam eps 1e-8, gamma 0.99, grad-norm clip 40, 1-step double-Q dueling
# targets, epsilon 1.0 -> 0.02 over the first 10 % of the sample budget); they could not be checked against an RLlib or
# reference checkout, so they are this module's chosen defaults.  The replay and minibatch sizes are scaled to
# thousands of environments and are this project's choice: minibatch 4096 (a multiple of 128, one kernel CTA per 128
# samples), 2^21 transitions, learning after 65536, 8 replayed samples per collected sample, target sync every 200
# gradient steps.
_DEFAULTS = dict(lr=5e-4, adam_beta1=0.9, adam_beta2=0.999, adam_eps=1e-8, gamma=0.99, grad_clip=40.0, minibatch_size=4096,
                 replay_capacity=1 << 21, learning_starts=65536, train_intensity=8.0, target_update_freq=200,
                 epsilon_initial=1.0, epsilon_final=0.02, epsilon_fraction=0.1, seed=0)
STAT_NAMES = ('loss', 'abs_td', 'q_mean', 'target_mean')


class DQNConfig(LearnerConfig):
    """Hyper-parameters of `DQNLearner` (see _DEFAULTS); minibatch_size must be a positive multiple of 128."""
    _DEFAULTS = _DEFAULTS

    def _check(self):
        if self.replay_capacity <= 0 or self.learning_starts < 0 or self.target_update_freq <= 0:
            raise ValueError('replay_capacity and target_update_freq must be positive, learning_starts non-negative')
        if not self.train_intensity > 0.0 or not 0.0 < self.gamma <= 1.0 or not self.grad_clip > 0.0:
            raise ValueError('train_intensity and grad_clip must be positive and gamma in (0, 1]')
        if not (0.0 <= self.epsilon_final <= 1.0 and 0.0 <= self.epsilon_initial <= 1.0 and 0.0 < self.epsilon_fraction <= 1.0):
            raise ValueError('epsilon_initial and epsilon_final must be in [0, 1] and epsilon_fraction in (0, 1]')


def epsilon_at(cfg, env_steps, total_samples):
    """The exploration schedule: linear from epsilon_initial to epsilon_final over the first epsilon_fraction of the
    sample budget, epsilon_final after it."""
    horizon = cfg.epsilon_fraction * float(total_samples)
    frac = min(1.0, float(env_steps) / horizon) if horizon > 0 else 1.0
    return cfg.epsilon_initial + frac * (cfg.epsilon_final - cfg.epsilon_initial)


def grad_steps_for(cfg, n_collected):
    """Gradient steps per update: ceil(train_intensity * collected samples / minibatch_size)."""
    return int(math.ceil(cfg.train_intensity * n_collected / cfg.minibatch_size))


class ReplayBuffer(object):
    """A ring of transitions on the device.  Fragment row (t, b) becomes ring row (pos + t * B + b) % capacity, where pos
    is where the previous insertion stopped: s = obs[t], a = actions[t], r = actual[t] (the gym reward, reward - penalty),
    s' = term_obs[t] (the terminal observation when done, not the reset observation in obs[t + 1]), done = done[t]."""

    def __init__(self, capacity, obs_dim, device):
        self.capacity, self.obs_dim, self.device = int(capacity), int(obs_dim), torch.device(device)
        f64 = torch.float64
        self.obs = torch.zeros(self.capacity, self.obs_dim, dtype=f64, device=self.device)
        self.next_obs = torch.zeros(self.capacity, self.obs_dim, dtype=f64, device=self.device)
        self.actions = torch.zeros(self.capacity, dtype=torch.int64, device=self.device)
        self.reward = torch.zeros(self.capacity, dtype=torch.float32, device=self.device)
        self.done = torch.zeros(self.capacity, dtype=torch.uint8, device=self.device)
        self.pos = 0
        self.size = 0

    def add(self, frag):
        """Insert the T * B transitions of a fragment (stream-ordered copies; no synchronisation)."""
        T, B = frag.T, frag.B
        N = T * B
        src = (frag.obs[:T].reshape(N, -1), frag.term_obs.reshape(N, -1), frag.actions.reshape(N), frag.actual.reshape(N),
               frag.done.reshape(N))
        dst = (self.obs, self.next_obs, self.actions, self.reward, self.done)
        skip = max(0, N - self.capacity)          # a fragment larger than the ring keeps its last `capacity` rows
        start = (self.pos + skip) % self.capacity
        n = N - skip
        first = min(n, self.capacity - start)
        for s, d in zip(src, dst):
            d[start:start + first].copy_(s[skip:skip + first])
            if n > first:
                d[:n - first].copy_(s[skip + first:])
        self.pos = (self.pos + N) % self.capacity
        self.size = min(self.capacity, self.size + N)

    def sample(self, n, generator):
        """n row indices (int32), uniform with replacement over the filled rows."""
        if self.size == 0:
            raise ValueError('the replay buffer is empty')
        return torch.randint(0, self.size, (n,), generator=generator, device=self.device, dtype=torch.int32)


class DQNLearner(Learner):
    """Double DQN over fragments of a `RolloutWorker`, training `policy` (a discrete `rollout.MlpPolicy`) in place: its
    torch tensors and, when enabled, its native act kernel's weights follow every update.  The target network is a
    second flat parameter vector, copied from the online one every target_update_freq gradient steps."""
    _CREATE, _DESTROY = 'paintrl_dqn_create', 'paintrl_dqn_destroy'

    def __init__(self, policy, config=None):
        if not policy.discrete:
            raise ValueError('DQN takes discrete action spaces only')
        super().__init__(policy, config if config is not None else DQNConfig())
        self.target = self.params.clone()
        self.replay = ReplayBuffer(self.cfg.replay_capacity, self.obs_dim, self.device)

    def _c_config(self):
        return _capi.PaintrlDqnConfig(_capi.PAINTRL_ABI_VERSION, self.obs_dim, self.n_out, self.cfg.minibatch_size, self.cfg.gamma)

    def grad_into(self, buf, idx, grad, stats, params=None, target=None):
        """One `paintrl_dqn_grad` call on rows `idx` (int32) of `buf` (a `ReplayBuffer` or anything with its five
        arrays); stats float32 [>= 4]."""
        _capi.check(self._lib.paintrl_dqn_grad(
            self._h, _ptr(self.params if params is None else params), _ptr(self.target if target is None else target), _ptr(idx),
            idx.numel(), _ptr(buf.obs), _ptr(buf.actions), _ptr(buf.reward), _ptr(buf.next_obs), _ptr(buf.done), _ptr(grad),
            _ptr(stats), self._stream()))

    def clip(self, grad, norm_out):
        _capi.check(self._lib.paintrl_clip_grad_norm(_ptr(grad), grad.numel(), self.cfg.grad_clip, _ptr(norm_out), self._stream()))

    def sync_target(self):
        self.target.copy_(self.params)

    @torch.no_grad()
    def train_steps(self, n_steps, buf=None):
        """n_steps gradient steps on uniform samples of `buf` (a `ReplayBuffer`, default: this learner's); returns the
        device statistics [n_steps, 8]: STAT_NAMES, then the gradient norm before clipping."""
        buf = self.replay if buf is None else buf
        stats = torch.zeros(n_steps, 8, dtype=torch.float32, device=self.device)
        native = getattr(self.policy, 'native', None)
        for k in range(n_steps):
            idx = buf.sample(self.cfg.minibatch_size, self.gen)
            self.grad_into(buf, idx, self.grad, stats[k])
            self.clip(self.grad, stats[k, 4:5])
            self.adam(self.grad)
            if native is not None:
                native.set_params(self.params)
            if self.step % self.cfg.target_update_freq == 0:
                self.sync_target()
        return stats

    @torch.no_grad()
    def update(self, frag):
        """Insert the fragment into the replay buffer; once learning_starts transitions are stored, run
        ceil(train_intensity * T * B / minibatch_size) gradient steps.  Returns the mean statistics over those steps
        (STAT_NAMES and the mean gradient norm before clipping), the number of steps and the replay size."""
        self.replay.add(frag)
        n_new = frag.T * frag.B
        out = {'grad_steps': 0, 'replay_size': self.replay.size, 'samples': n_new}
        if self.replay.size < self.cfg.learning_starts:
            return out
        n_steps = grad_steps_for(self.cfg, n_new)
        stats = self.train_steps(n_steps)
        unflatten_into(self.policy, self.params)
        host = stats.cpu().numpy().astype('float64')
        out.update({name: float(host[:, i].mean()) for i, name in enumerate(STAT_NAMES)})
        out['grad_norm'] = float(host[:, 4].mean())
        out['grad_steps'] = n_steps
        out['replayed_samples'] = n_steps * self.cfg.minibatch_size
        return out

    def state_dict(self):
        """Parameters, target parameters, Adam moments, the step count and the sampling generator.  The replay buffer
        is not part of it: a resumed run refills it (and waits for learning_starts transitions again)."""
        return dict(self._state_dict(), algo='dqn', target_params=self.target.cpu())

    def load_state_dict(self, sd):
        check_state_dict(sd, self.obs_dim, self.n_out)
        self.target.copy_(sd['target_params'])
        self._load_state_dict(sd)


def check_state_dict(sd, obs_dim, n_out):
    """Raise ValueError when a DQN learner state does not fit a discrete policy of this shape."""
    _check_state_dict(sd, obs_dim, n_out, True, ('params', 'target_params', 'adam_m', 'adam_v'))
