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

Prioritized replay and n-step returns (Ape-X DQN's replay side; the 4096 environments play its many actors) are opt-in:
`DQNConfig(prioritized_replay=True, n_step=3)`.  Then the buffer is a `PrioritizedReplayBuffer` (sum and min trees on
the device, csrc/paintrl_replay.cuh), and a gradient step samples in proportion to priority (`paintrl_prio_sample`),
runs the importance-weighted loss (`paintrl_dqn_grad_weighted`), and writes the minibatch's TD errors back as
priorities (`paintrl_prio_update`) before the clip, Adam and the weight pack.  The n-step transitions are built in
`ReplayBuffer.add`, so the kernel bootstraps with the handle's discount gamma^n.
"""
import ctypes
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
#
# Prioritized replay and n-step returns, off by default: RLlib DQN's prioritized-replay values as recalled (alpha 0.6,
# beta 0.4, eps 1e-6) and Ape-X's n_step = 3 (for `--n-step 3`), not checked against an RLlib checkout either, so they too
# are this module's chosen defaults.  beta stays constant.
_DEFAULTS = dict(lr=5e-4, adam_beta1=0.9, adam_beta2=0.999, adam_eps=1e-8, gamma=0.99, grad_clip=40.0, minibatch_size=4096,
                 replay_capacity=1 << 21, learning_starts=65536, train_intensity=8.0, target_update_freq=200,
                 epsilon_initial=1.0, epsilon_final=0.02, epsilon_fraction=0.1, seed=0,
                 prioritized_replay=False, prioritized_replay_alpha=0.6, prioritized_replay_beta=0.4, prioritized_replay_eps=1e-6,
                 n_step=1)
STAT_NAMES = ('loss', 'abs_td', 'q_mean', 'target_mean')
PER_STAT_NAMES = STAT_NAMES + ('weight_mean',)    # with prioritized replay: loss is the importance-weighted Huber loss


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
        if not (0.0 <= self.prioritized_replay_alpha < math.inf and 0.0 <= self.prioritized_replay_beta <= 1.0
                and 0.0 < self.prioritized_replay_eps < math.inf):
            raise ValueError('prioritized_replay_alpha must be finite and >= 0, prioritized_replay_beta in [0, 1] and '
                             'prioritized_replay_eps finite and > 0')
        if self.n_step < 1:
            raise ValueError('n_step must be 1 or more')


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
    """A ring of transitions on the device.  With n_step = 1, fragment row (t, b) becomes ring row (pos + t * B + b) %
    capacity, where pos is where the previous insertion stopped: s = obs[t], a = actions[t], r = actual[t] (the gym
    reward, reward - penalty), s' = term_obs[t] (the terminal observation when done, not the reset observation in
    obs[t + 1]), done = done[t].

    With n_step = n > 1, transition t covers steps t .. t + m - 1, m = n or fewer when the episode ends inside the
    window: r = fl32(sum_{k < m} gamma^k actual[t + k]) summed in FP64 in increasing k, s' = term_obs[t + m - 1], done =
    done[t + m - 1].  A done transition never bootstraps, so the learner's discount is gamma^n for every other one.  The
    last n - 1 steps of a fragment wait in a device carry and complete with the next fragment's first steps, so no
    transition is cut at a fragment boundary: every insertion after the first n - 1 steps writes T * B rows."""

    def __init__(self, capacity, obs_dim, device, n_step=1, gamma=1.0):
        self.capacity, self.obs_dim, self.device = int(capacity), int(obs_dim), torch.device(device)
        self.n_step, self.gamma = int(n_step), float(gamma)
        if self.n_step < 1:
            raise ValueError('n_step must be 1 or more')
        f64 = torch.float64
        self.obs = torch.zeros(self.capacity, self.obs_dim, dtype=f64, device=self.device)
        self.next_obs = torch.zeros(self.capacity, self.obs_dim, dtype=f64, device=self.device)
        self.actions = torch.zeros(self.capacity, dtype=torch.int64, device=self.device)
        self.reward = torch.zeros(self.capacity, dtype=torch.float32, device=self.device)
        self.done = torch.zeros(self.capacity, dtype=torch.uint8, device=self.device)
        self.pos = 0
        self.size = 0
        self._carry = None                         # n_step > 1: the last < n steps, time-major (obs, term_obs, actions, actual, done)

    def add(self, frag):
        """Insert a fragment's transitions (stream-ordered copies; no synchronisation).  Returns (start, count): the
        ring rows [start, start + count) mod capacity that were written (count 0 when none was)."""
        T, B = frag.T, frag.B
        steps = (frag.obs[:T], frag.term_obs, frag.actions, frag.actual, frag.done)
        if self.n_step == 1:
            N = T * B
            return self._write(N, (steps[0].reshape(N, -1), steps[1].reshape(N, -1), steps[2].reshape(N), steps[3].reshape(N),
                                   steps[4].reshape(N)))
        if self._carry is not None:
            if self._carry[0].shape[1] != B:
                raise ValueError('a fragment of %d environments follows one of %d' % (B, self._carry[0].shape[1]))
            steps = tuple(torch.cat([c, x]) for c, x in zip(self._carry, steps))
        n = self.n_step
        C = steps[0].shape[0]
        E = max(0, C - (n - 1))                    # steps whose whole n-step window is here
        self._carry = tuple(x[E:].clone() for x in steps)
        if E == 0:
            return self.pos, 0
        obs, term_obs, actions, actual, done = steps
        d = done.bool()
        ret = torch.zeros(E, B, dtype=torch.float64, device=actual.device)
        alive = torch.ones(E, B, dtype=torch.bool, device=actual.device)
        last = torch.full((E, B), n - 1, dtype=torch.int64, device=actual.device)
        for k in range(n):
            ret = ret + torch.where(alive, (self.gamma ** k) * actual[k:k + E], torch.zeros_like(ret))
            if k < n - 1:
                last = torch.where(alive & d[k:k + E], torch.full_like(last, k), last)
                alive = alive & ~d[k:k + E]
        t_end = torch.arange(E, device=actual.device).unsqueeze(1) + last          # t + m - 1
        b_idx = torch.arange(B, device=actual.device).unsqueeze(0).expand(E, B)
        N = E * B
        return self._write(N, (obs[:E].reshape(N, -1), term_obs[t_end, b_idx].reshape(N, -1), actions[:E].reshape(N),
                               ret.reshape(N), done[t_end, b_idx].reshape(N)))

    def _write(self, N, src):
        """Copy N transitions (s, s', a, r, done) into the ring at pos; a batch larger than the ring keeps its last
        `capacity` rows."""
        dst = (self.obs, self.next_obs, self.actions, self.reward, self.done)
        skip = max(0, N - self.capacity)
        start = (self.pos + skip) % self.capacity
        n = N - skip
        first = min(n, self.capacity - start)
        for s, d in zip(src, dst):
            d[start:start + first].copy_(s[skip:skip + first])
            if n > first:
                d[:n - first].copy_(s[skip + first:])
        self.pos = (self.pos + N) % self.capacity
        self.size = min(self.capacity, self.size + N)
        return start, n

    def sample(self, n, generator):
        """n row indices (int32), uniform with replacement over the filled rows."""
        if self.size == 0:
            raise ValueError('the replay buffer is empty')
        return torch.randint(0, self.size, (n,), generator=generator, device=self.device, dtype=torch.int32)


def tree_leaves(capacity):
    """L, the sum and min trees' leaf count: the smallest power of two at or above capacity."""
    return 1 << (int(capacity) - 1).bit_length()


class PrioritizedReplayBuffer(ReplayBuffer):
    """The ring with RLlib's proportional prioritization: priorities p^alpha in a device sum tree and min tree (FP64
    [2L], root at 1, row r at leaf L + r, see include/paintrl.h), and max_priority, the largest |td| + eps so far
    (starting at 1), which new rows receive.  Every operation is a stream-ordered native call."""

    def __init__(self, capacity, obs_dim, device, alpha=0.6, eps=1e-6, n_step=1, gamma=1.0):
        super().__init__(capacity, obs_dim, device, n_step, gamma)
        self.alpha, self.eps = float(alpha), float(eps)
        self.L = tree_leaves(self.capacity)
        self.sum_tree = torch.zeros(2 * self.L, dtype=torch.float64, device=self.device)
        self.min_tree = torch.full((2 * self.L,), math.inf, dtype=torch.float64, device=self.device)
        self.max_priority = torch.ones(1, dtype=torch.float64, device=self.device)
        self._lib = _capi.lib()

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def add(self, frag):
        start, count = super().add(frag)
        if count:
            _capi.check(self._lib.paintrl_prio_fill(_ptr(self.sum_tree), _ptr(self.min_tree), self.L, self.capacity, start, count,
                                                    _ptr(self.max_priority), self.alpha, self._stream()))
        return start, count

    def sample(self, n, generator, beta=0.4):
        """(idx int32 [n], weights float32 [n]): rows drawn in proportion to priority from n FP64 uniforms of
        `generator`, and their importance weights (p_i / p_min)^(-beta)."""
        if self.size == 0:
            raise ValueError('the replay buffer is empty')
        u = torch.rand(n, generator=generator, dtype=torch.float64, device=self.device)
        idx = torch.empty(n, dtype=torch.int32, device=self.device)
        w = torch.empty(n, dtype=torch.float32, device=self.device)
        _capi.check(self._lib.paintrl_prio_sample(_ptr(self.sum_tree), _ptr(self.min_tree), self.L, self.capacity, self.size, _ptr(u),
                                                  n, float(beta), _ptr(idx), _ptr(w), self._stream()))
        return idx, w

    def update_priorities(self, idx, td):
        """Rows idx (int32) get priority |td| + eps (td float32, as the weighted loss writes it)."""
        _capi.check(self._lib.paintrl_prio_update(_ptr(self.sum_tree), _ptr(self.min_tree), self.L, self.capacity, _ptr(idx), _ptr(td),
                                                  idx.numel(), _ptr(self.max_priority), self.alpha, self.eps, self._stream()))


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
        c = self.cfg
        if c.prioritized_replay:
            self.replay = PrioritizedReplayBuffer(c.replay_capacity, self.obs_dim, self.device, c.prioritized_replay_alpha,
                                                  c.prioritized_replay_eps, c.n_step, c.gamma)
            self.td = torch.zeros(c.minibatch_size, dtype=torch.float32, device=self.device)
        else:
            self.replay = ReplayBuffer(c.replay_capacity, self.obs_dim, self.device, c.n_step, c.gamma)

    def _c_config(self):
        # n-step transitions carry their own discounted return; the bootstrap discount is gamma^n (rounded to float32)
        return _capi.PaintrlDqnConfig(_capi.PAINTRL_ABI_VERSION, self.obs_dim, self.n_out, self.cfg.minibatch_size,
                                      self.cfg.gamma ** self.cfg.n_step)

    def grad_into(self, buf, idx, grad, stats, params=None, target=None):
        """One `paintrl_dqn_grad` call on rows `idx` (int32) of `buf` (a `ReplayBuffer` or anything with its five
        arrays); stats float32 [>= 4]."""
        _capi.check(self._lib.paintrl_dqn_grad(
            self._h, _ptr(self.params if params is None else params), _ptr(self.target if target is None else target), _ptr(idx),
            idx.numel(), _ptr(buf.obs), _ptr(buf.actions), _ptr(buf.reward), _ptr(buf.next_obs), _ptr(buf.done), _ptr(grad),
            _ptr(stats), self._stream()))

    def grad_weighted_into(self, buf, idx, weight, td_out, grad, stats, params=None, target=None):
        """One `paintrl_dqn_grad_weighted` call: `grad_into` with importance weights (float32 [n]) and the TD errors
        written to td_out (float32 [n]); stats float32 [>= 5] (PER_STAT_NAMES)."""
        _capi.check(self._lib.paintrl_dqn_grad_weighted(
            self._h, _ptr(self.params if params is None else params), _ptr(self.target if target is None else target), _ptr(idx),
            idx.numel(), _ptr(buf.obs), _ptr(buf.actions), _ptr(buf.reward), _ptr(buf.next_obs), _ptr(buf.done), _ptr(weight),
            _ptr(td_out), _ptr(grad), _ptr(stats), self._stream()))

    def clip(self, grad, norm_out):
        _capi.check(self._lib.paintrl_clip_grad_norm(_ptr(grad), grad.numel(), self.cfg.grad_clip, _ptr(norm_out), self._stream()))

    def sync_target(self):
        self.target.copy_(self.params)

    @torch.no_grad()
    def train_steps(self, n_steps, buf=None):
        """n_steps gradient steps on uniform samples of `buf` (a `ReplayBuffer`, default: this learner's); returns the
        device statistics [n_steps, 8]: STAT_NAMES, then the gradient norm before clipping.  With prioritized_replay the
        samples are prioritized (`buf` a `PrioritizedReplayBuffer`) and the columns are PER_STAT_NAMES, then the norm."""
        buf = self.replay if buf is None else buf
        if self.cfg.prioritized_replay:
            return self._train_steps_prioritized(n_steps, buf)
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

    def _train_steps_prioritized(self, n_steps, buf):
        stats = torch.zeros(n_steps, 8, dtype=torch.float32, device=self.device)
        native = getattr(self.policy, 'native', None)
        nst = len(PER_STAT_NAMES)
        for k in range(n_steps):
            idx, w = buf.sample(self.cfg.minibatch_size, self.gen, self.cfg.prioritized_replay_beta)
            self.grad_weighted_into(buf, idx, w, self.td, self.grad, stats[k])
            buf.update_priorities(idx, self.td)
            self.clip(self.grad, stats[k, nst:nst + 1])
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
        (STAT_NAMES, or PER_STAT_NAMES with prioritized replay, and the mean gradient norm before clipping), the number
        of steps and the replay size."""
        self.replay.add(frag)
        n_new = frag.T * frag.B
        out = {'grad_steps': 0, 'replay_size': self.replay.size, 'samples': n_new}
        if self.replay.size < self.cfg.learning_starts:
            return out
        n_steps = grad_steps_for(self.cfg, n_new)
        stats = self.train_steps(n_steps)
        unflatten_into(self.policy, self.params)
        host = stats.cpu().numpy().astype('float64')
        names = PER_STAT_NAMES if self.cfg.prioritized_replay else STAT_NAMES
        out.update({name: float(host[:, i].mean()) for i, name in enumerate(names)})
        out['grad_norm'] = float(host[:, len(names)].mean())
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
