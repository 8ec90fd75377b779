"""On-GPU rollout collection against the batched paint environment (BASELINE config C5).

The reference collects PPO experience with RLlib: 15 CPU rollout workers, one PaintGymEnv each,
`sample_batch_size` = 100 steps per fragment, `batch_mode` = truncate_episodes, a fully connected
policy with hidden layers [256, 128] and a shared value branch (paint_ppo.py:170-195), and
per-episode totals of reward / penalty / return gathered by callbacks (paint_ppo.py:36-72).  Ray and
TensorFlow are absent here, so this module is the built-in torch stand-in SURVEY.md section 8(d) C5
asks for: the same fragment shape and statistics, with the policy evaluated and sampled on the GPU
the environments live on -- observations and actions never visit the host.

One process per GPU owns a shard of the environments (`sharding.shard_range`); the step path has no
collective; `iteration_stats` reduces the per-iteration statistics with one small all-reduce.
The policy runs as ONE kernel of this repository per environment step (`paintrl_policy_act`, csrc/paintrl_policy.cuh:
layer 2 on the tcgen05 tensor cores, sampling included); a plain torch evaluation of the same weights is kept as the
FP32 reference the tests compare against and as the path for shapes the kernel does not take (obs_dim > 32).
"""
import ctypes
import math

import numpy as np
import torch

from . import _capi, sharding


def _fptr(t):
    return t.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


class NativePolicy(object):
    """`paintrl_policy_*` (include/paintrl.h): the MLP of paint_ppo.py:179-183 evaluated and sampled in one launch."""

    def __init__(self, obs_dim, n_out, discrete, weights, capacity, device, seed=0):
        self._lib = _capi.lib()
        self.device = torch.device(device)
        self.obs_dim, self.n_out, self.discrete, self.capacity, self.seed = int(obs_dim), int(n_out), bool(discrete), int(capacity), int(seed)
        host = [np.ascontiguousarray(w.detach().cpu().numpy(), dtype=np.float32) for w in weights]    # w1 b1 w2 b2 w3 b3
        cfg = _capi.PaintrlPolicyConfig(_capi.PAINTRL_ABI_VERSION, self.obs_dim, self.n_out, int(self.discrete), self.capacity, self.seed,
                                        *[_fptr(a) for a in host])
        handle = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _capi.check(self._lib.paintrl_policy_create(ctypes.byref(cfg), index, ctypes.byref(handle)))
        self._h = handle

    def close(self):
        if getattr(self, '_h', None):
            self._lib.paintrl_policy_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def act_into(self, obs, actions, logp, value, logits=None, sample=True):
        """obs float64 [B, obs_dim] -> actions (int64 [B] | float64 [B, n_out]), logp / value float32 [B], all contiguous
        CUDA tensors of this device, written in place by one kernel launch on the current stream."""
        B = obs.shape[0]
        p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        _capi.check(self._lib.paintrl_policy_act(self._h, p(obs), B, p(actions), p(logp), p(value), p(logits), int(bool(sample)),
                                                 ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def act_epsilon_into(self, obs, actions, value, epsilon, logits=None):
        """Epsilon-greedy actions over the head read as a dueling Q-network (`paintrl_policy_act_epsilon`, discrete
        engines only): `epsilon` is a one-element float32 CUDA tensor the kernel reads on every launch."""
        if not self.discrete:
            raise ValueError('epsilon-greedy actions need a discrete policy')
        B = obs.shape[0]
        p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        _capi.check(self._lib.paintrl_policy_act_epsilon(self._h, p(obs), B, p(actions), p(value), p(logits), p(epsilon),
                                                         ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def act_diag_gaussian_into(self, obs, actions, logp, value, logits=None):
        """Sample the diagonal-Gaussian head (`paintrl_policy_act_diag_gaussian`, continuous engines with an even n_out):
        head columns [0, A) are the means and [A, 2A) the log-stds, A = n_out / 2; actions float64 [B, A] hold the FP32
        values mean + std * noise, and logp is their log-probability as the learner computes it."""
        if self.discrete or self.n_out % 2:
            raise ValueError('diagonal-Gaussian actions need a continuous policy with an even n_out')
        B = obs.shape[0]
        p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        _capi.check(self._lib.paintrl_policy_act_diag_gaussian(self._h, p(obs), B, p(actions), p(logp), p(value), p(logits),
                                                               ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def set_params(self, params):
        """Pack a flat FP32 parameter vector (w1 | b1 | w2 | b2 | w3 | b3, a contiguous CUDA tensor of this device) into
        this engine's device weights, in place and on the current stream: a captured rollout graph samples with the new
        weights on its next replay."""
        _capi.check(self._lib.paintrl_policy_set_params(self._h, ctypes.c_void_p(params.data_ptr()),
                                                        ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))


DISTS = ('categorical', 'tanh_gaussian', 'diag_gaussian')


def default_dist(discrete):
    """The distribution of a policy built without `dist`: what every policy was before `dist` existed."""
    return 'categorical' if discrete else 'tanh_gaussian'


class MlpPolicy(object):
    """Fully connected policy of paint_ppo.py:179-183: obs -> 256 -> 128 -> {logits | mean, value},
    tanh activations (RLlib's fcnet default), value branch sharing the hidden layers
    (`vf_share_layers`).  Random-init FP32 weights.  `dist` names the action distribution:
    'categorical' (discrete; Gumbel-max sampling of n_out logits), 'tanh_gaussian' (continuous; unit-variance
    Gaussian around tanh(mean), n_out means) or 'diag_gaussian' (continuous; RLlib's DiagGaussian, mean + exp(log_std)
    noise with a learned log-std: `n_out` is then the action dimension A, and the head has 2A outputs, means then
    log-stds, so `self.n_out` is 2A and `self.action_dim` is A)."""

    def __init__(self, obs_dim, n_out, hiddens=(256, 128), device=None, seed=0, discrete=True, dist=None):
        dist = default_dist(discrete) if dist is None else dist
        if dist not in DISTS or (dist == 'categorical') != bool(discrete):
            raise ValueError('dist %r does not fit discrete=%r (categorical is the discrete one)' % (dist, discrete))
        self.dist = dist
        self.action_dim = int(n_out) if not discrete else 1
        if dist == 'diag_gaussian':
            n_out = 2 * int(n_out)
        gen = torch.Generator(device='cpu')
        gen.manual_seed(seed)
        dims = [obs_dim] + list(hiddens)
        self.layers = []
        for i in range(len(hiddens)):
            bound = 1.0 / math.sqrt(dims[i])
            w = (torch.rand(dims[i], dims[i + 1], generator=gen) * 2 - 1) * bound
            b = torch.zeros(dims[i + 1])
            self.layers.append((w.to(device), b.to(device)))
        bound = 1.0 / math.sqrt(dims[-1])
        self.head_w = ((torch.rand(dims[-1], n_out + 1, generator=gen) * 2 - 1) * bound * 0.1).to(device)
        self.head_b = torch.zeros(n_out + 1, device=device)
        self.n_out = n_out
        self.discrete = discrete
        if torch.cuda.is_available():
            torch.backends.cuda.matmul.allow_tf32 = True     # the policy's three small GEMMs on the tensor cores
        self.device = device
        self.gen = torch.Generator(device=device)
        self.gen.manual_seed(seed + 1)
        self.obs_dim, self.seed = obs_dim, seed
        self.native = None

    def weights(self):
        (w1, b1), (w2, b2) = self.layers
        return [w1, b1, w2, b2, self.head_w, self.head_b]

    def enable_native(self, capacity):
        """Evaluate and sample with the repository's own kernel (one launch per step) for batches up to `capacity`.
        Returns False when the shape is outside what the kernel takes (the torch path stays)."""
        if self.native is not None and self.native.capacity >= capacity:
            return True
        if not (self.obs_dim <= 32 and self.n_out + 1 <= 16 and len(self.layers) == 2 and
                tuple(self.layers[0][0].shape) == (self.obs_dim, 256) and tuple(self.layers[1][0].shape) == (256, 128)):
            return False
        self.native = NativePolicy(self.obs_dim, self.n_out, self.discrete, self.weights(), capacity, self.device, seed=self.seed)
        return True

    def describe(self):
        return ('one paintrl_policy_act kernel per step: layer 2 on tcgen05 tensor cores (BF16 x BF16 -> FP32), FP32 elsewhere'
                if self.native is not None else 'torch addmm (TF32) + elementwise kernels')

    def forward(self, obs):
        """obs [B, obs_dim] (any float dtype) -> (logits or means [B, n_out], value [B]) in FP32."""
        h = obs.to(torch.float32)
        for w, b in self.layers:
            h = torch.tanh(torch.addmm(b, h, w))
        out = torch.addmm(self.head_b, h, self.head_w)
        return out[:, :self.n_out], out[:, self.n_out]

    def act(self, obs):
        """Sample one action per environment: (actions, log-probability, value)."""
        out, value = self.forward(obs)
        if self.dist == 'diag_gaussian':
            A = self.action_dim
            mean, log_std = out[:, :A], out[:, A:]
            noise = torch.randn(mean.shape, generator=self.gen, device=out.device)
            a = mean + torch.exp(log_std) * noise
            logp = (-0.5 * noise * noise - log_std).sum(dim=1) - A * 0.5 * math.log(2 * math.pi)
            return a.to(torch.float64), logp, value
        if self.discrete:
            logp_all = torch.log_softmax(out, dim=1)
            u = torch.rand(out.shape, generator=self.gen, device=out.device).clamp_(1e-10, 1.0)
            a = torch.argmax(logp_all - torch.log(-torch.log(u)), dim=1)
            return a, logp_all.gather(1, a[:, None])[:, 0], value
        mean = torch.tanh(out)
        noise = torch.randn(out.shape, generator=self.gen, device=out.device)
        a = mean + noise
        logp = (-0.5 * noise * noise - 0.5 * math.log(2 * math.pi)).sum(dim=1)
        return a.to(torch.float64), logp, value


class RolloutFragment(object):
    """Time-major buffers of one fragment: T steps of B environments, all on the device."""

    def __init__(self, T, B, obs_dim, action_shape, device, logits_dim=None):
        f64, f32 = torch.float64, torch.float32
        self.T, self.B = T, B
        self.obs = torch.zeros(T + 1, B, obs_dim, dtype=f64, device=device)     # obs[t] is what the policy saw at step t
        self.term_obs = torch.zeros(T, B, obs_dim, dtype=f64, device=device)    # observation returned with step t (terminal if done)
        self.actions = torch.zeros((T, B) + tuple(action_shape), dtype=torch.int64 if not action_shape else f64,
                                   device=device)
        self.reward = torch.zeros(T, B, dtype=f64, device=device)               # info['reward']   (robot_gym_env.py:368)
        self.penalty = torch.zeros(T, B, dtype=f64, device=device)              # info['penalty']
        self.actual = torch.zeros(T, B, dtype=f64, device=device)               # the gym reward = reward - penalty
        self.done = torch.zeros(T, B, dtype=torch.uint8, device=device)
        self.new_texels = torch.zeros(T, B, dtype=torch.int32, device=device)
        self.logp = torch.zeros(T, B, dtype=f32, device=device)
        self.value = torch.zeros(T + 1, B, dtype=f32, device=device)
        # the policy's logits | means and value at step t (the PPO learner's KL term); only with keep_logits
        self.logits = torch.zeros(T, B, logits_dim, dtype=f32, device=device) if logits_dim else None


class RolloutWorker(object):
    """Collects fragments from a `BatchedPaintEnv` created with `auto_reset=True`."""

    def __init__(self, env, policy, fragment_length=100, use_cuda_graph=False, use_native_policy=True, keep_logits=False,
                 epsilon=None):
        """`use_cuda_graph`: after one eager fragment, capture the whole T-step loop (policy kernels and the
        two step kernels per step, ~25 launches each) into one CUDA graph and replay it per fragment -- the
        fragment buffers are persistent, so every address in the loop is static.  Small batches are
        launch-bound without it.
        `keep_logits`: the policy kernel also writes its logits | means and value into `fragment.logits`
        [T, B, n_out + 1] (what `ppo.PPOLearner` needs for the KL term); needs the native policy.
        `epsilon`: a one-element float32 CUDA tensor; the native policy then acts epsilon-greedily on its head read as a
        dueling Q-network (`dqn.DQNLearner`), reading epsilon on every step, inside a captured graph too, and
        `fragment.logp` is not written.  Needs the native policy and discrete actions."""
        if not env.cfg.auto_reset:
            raise ValueError('RolloutWorker needs an environment created with auto_reset=True')
        self.diag = getattr(policy, 'dist', None) == 'diag_gaussian'
        if self.diag and (env.cfg.action_mode != 'continuous' or policy.action_dim != env.action_dim):
            raise ValueError('a diagonal-Gaussian policy of %d action dimensions does not fit this environment (%s, %d)'
                             % (policy.action_dim, env.cfg.action_mode, env.action_dim))
        self.env, self.policy, self.T = env, policy, int(fragment_length)
        if use_native_policy and hasattr(policy, 'enable_native'):
            policy.enable_native(env.num_envs)
        self.keep_logits = bool(keep_logits)
        if self.keep_logits and getattr(policy, 'native', None) is None:
            raise ValueError('keep_logits needs the native policy kernel (obs_dim <= 32, n_out <= 15, hidden layers 256, 128)')
        self.epsilon = epsilon
        if epsilon is not None:
            if getattr(policy, 'native', None) is None or env.cfg.action_mode != 'discrete':
                raise ValueError('epsilon-greedy collection needs the native policy kernel and discrete actions')
            if not (torch.is_tensor(epsilon) and epsilon.is_cuda and epsilon.dtype == torch.float32 and epsilon.numel() == 1):
                raise ValueError('epsilon must be a one-element float32 CUDA tensor')
        self.use_cuda_graph = bool(use_cuda_graph)
        self._graph, self._eager_fragments, self.graph_error = None, 0, None
        shape = () if env.cfg.action_mode == 'discrete' else (env.action_dim,)
        self.frag = RolloutFragment(self.T, env.num_envs, env.obs_dim, shape, env.device,
                                    logits_dim=policy.n_out + 1 if self.keep_logits else None)
        dev, B = env.device, env.num_envs
        # running per-episode totals (the reference's on_episode_step / on_episode_end callbacks)
        self.ep_reward = torch.zeros(B, dtype=torch.float64, device=dev)
        self.ep_penalty = torch.zeros(B, dtype=torch.float64, device=dev)
        self.ep_len = torch.zeros(B, dtype=torch.int64, device=dev)
        # the observation the next fragment starts from: written by start() and at the end of every fragment,
        # read at the top of every fragment -- inside the captured loop, so back-to-back collect() calls are
        # always consistent (no separate advance() step to forget)
        self._carry = torch.zeros(B, env.obs_dim, dtype=torch.float64, device=dev)
        self._started = False

    def start(self, start_index=None):
        """Reset every environment; the first observation of the first fragment."""
        self._carry.copy_(self.env.reset(start_index))
        self.frag.obs[0].copy_(self._carry)
        self.ep_reward.zero_(); self.ep_penalty.zero_(); self.ep_len.zero_()
        self._started = True

    def _run_steps(self):
        f, env, pol = self.frag, self.env, self.policy
        f.obs[0].copy_(self._carry)
        native = pol.native
        for t in range(self.T):
            if native is not None and self.epsilon is not None:
                native.act_epsilon_into(f.obs[t], f.actions[t], f.value[t], self.epsilon, logits=None if f.logits is None else f.logits[t])
            elif native is not None and self.diag:
                native.act_diag_gaussian_into(f.obs[t], f.actions[t], f.logp[t], f.value[t], logits=None if f.logits is None else f.logits[t])
            elif native is not None:
                # one launch: obs[t] -> actions[t], logp[t], value[t] written in place (no torch kernels in the loop)
                native.act_into(f.obs[t], f.actions[t], f.logp[t], f.value[t], logits=None if f.logits is None else f.logits[t])
            else:
                a, logp, value = pol.act(f.obs[t])
                f.actions[t].copy_(a)
                f.logp[t].copy_(logp)
                f.value[t].copy_(value)
            env.step_into(f.actions[t], f.term_obs[t], f.reward[t], f.penalty[t], f.actual[t], f.done[t],
                          next_obs=f.obs[t + 1], new_texels=f.new_texels[t])
        if native is not None:
            native.act_into(f.obs[self.T], None, None, f.value[self.T], sample=False)     # bootstrap value of the truncated episodes
        else:
            f.value[self.T].copy_(pol.forward(f.obs[self.T])[1])
        self._carry.copy_(f.obs[self.T])

    def _capture(self):
        try:
            torch.cuda.synchronize(self.env.device)
            graph = torch.cuda.CUDAGraph()
            if hasattr(graph, 'register_generator_state'):
                graph.register_generator_state(self.policy.gen)
            with torch.cuda.graph(graph):
                self._run_steps()
            self._graph = graph
        except Exception as exc:                   # noqa: BLE001 - stay on the eager loop, keep the reason
            self._graph = None
            self.graph_error = '%s: %s' % (type(exc).__name__, exc)
            torch.cuda.synchronize(self.env.device)

    @torch.no_grad()
    def collect(self):
        """One fragment of T steps (truncate_episodes: episodes continue across fragments).
        Returns (fragment, stats) where stats holds this rank's sums for `iteration_stats`; the
        only host synchronisation is the read of those eight numbers at the end."""
        if not self._started:
            self.start()
        f, env = self.frag, self.env
        if self.use_cuda_graph and self._graph is None and self._eager_fragments >= 1 and self.graph_error is None:
            self._capture()
        if self._graph is not None:
            self._graph.replay()
        else:
            self._run_steps()
            self._eager_fragments += 1
        # per-episode totals (the reference's on_episode_step / on_episode_end callbacks), once per fragment:
        # running sums over time; an episode's total is the running sum at its `done` minus the running sum at
        # the previous `done` (rewards, penalties and step counts are non-negative, so that is a running maximum)
        done = f.done.bool()
        ones = torch.ones_like(f.reward)
        totals = []
        carries = []
        for carry, x in ((self.ep_reward, f.reward), (self.ep_penalty, f.penalty), (self.ep_len.to(torch.float64), ones)):
            cs = carry.unsqueeze(0) + torch.cumsum(x, dim=0)
            at_done = torch.where(done, cs, torch.zeros_like(cs))
            seen = torch.cummax(at_done, dim=0).values                      # running sum at the latest done <= t
            prev = torch.cat([torch.zeros_like(seen[:1]), seen[:-1]], dim=0)
            totals.append(torch.where(done, cs - prev, torch.zeros_like(cs)))
            carries.append(cs[-1] - seen[-1])
        self.ep_reward, self.ep_penalty = carries[0], carries[1]
        self.ep_len = carries[2].round().to(torch.int64)
        acc = torch.stack([done.sum().to(torch.float64), totals[0].sum(), totals[1].sum(), totals[0].sum() - totals[1].sum(),
                           f.new_texels.sum().to(torch.float64), totals[2].max()])
        host = acc.cpu()
        stats = {'env_steps': float(self.T * env.num_envs), 'episodes': float(host[0]), 'sum_reward': float(host[1]),
                 'sum_penalty': float(host[2]), 'sum_return': float(host[3]), 'new_texels': float(host[4]),
                 'max_episode_len': float(host[5])}
        return f, stats

    def advance(self):
        """Kept for callers of the first version: the hand-over of the last observation to the next fragment now
        happens inside `collect()` itself (`_carry`), so this is a no-op."""
        return None


def gae(frag, gamma=0.99, lam=1.0):
    """Generalised advantage estimates over a fragment (RLlib PPO defaults gamma 0.99, lambda 1.0):
    advantages and value targets [T, B] in FP32; `done` cuts the bootstrap."""
    T = frag.T
    adv = torch.zeros(T, frag.B, dtype=torch.float32, device=frag.value.device)
    last = torch.zeros(frag.B, dtype=torch.float32, device=frag.value.device)
    r = frag.actual.to(torch.float32)
    nd = 1.0 - frag.done.to(torch.float32)
    for t in range(T - 1, -1, -1):
        delta = r[t] + gamma * frag.value[t + 1] * nd[t] - frag.value[t]
        last = delta + gamma * lam * nd[t] * last
        adv[t] = last
    return adv, adv + frag.value[:T]


def iteration_stats(stats, device=None):
    """All-reduce one iteration's rollout statistics over the ranks (sums; maxima for `max_*`)."""
    return sharding.allreduce_stats(stats, device=device)
