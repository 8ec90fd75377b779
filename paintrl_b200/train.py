"""Train the rollout policy with PPO or double DQN on one GPU: collection and learning both on the device.

    python -m paintrl_b200.train --part 0 --envs 4096 --fragment 100 --samples 8000000 --seed 0 --checkpoint door.pt
    python -m paintrl_b200.train --algo dqn --envs 4096 --samples 2000000 --checkpoint door_dqn.pt
    python -m paintrl_b200.train --algo dqn --prioritized-replay --n-step 3 --samples 2000000 --checkpoint door_apex.pt
    python -m paintrl_b200.train --action-mode continuous --action-shape 2 --samples 20000000 --checkpoint door_cont.pt

Environment: BASELINE config C2 (RGB, section-4 observation, discrete-4 actions, late termination, anchor start points,
auto-reset) on the chosen part; --action-mode, --action-shape, --granularity, --obs-mode and --obs-grad change the
spaces.  Discrete actions give the policy one logit per action (n_out = granularity); continuous PPO trains RLlib's
diagonal-Gaussian head (a mean and a learned log-std per action dimension).  Shapes the kernels do not take
(observations of more than 32 entries, more than 15 discrete actions) and DQN with continuous actions are refused
before any work starts.  Policy: paint_ppo.py's [256, 128] MLP, sampled by the act kernel inside a captured
CUDA graph; the learner (`ppo.PPOLearner`) refreshes the kernel's weights in place after every minibatch.

Per iteration one JSON line: env-steps so far, the ended episodes' mean return, mean coverage ratio (episode `reward`
total x 100 / the part's max points; RGB) and mean length / 235 (the zigzag baseline's steps to full coverage), and the
collection and learner times (host clock around work that ends in a device synchronisation).  With --algo dqn
(`dqn.DQNLearner`) the act kernel is epsilon-greedy on the head read as a dueling Q-network, epsilon follows the
schedule of `dqn.epsilon_at` over the --samples budget and is written before every collection, and each line also
carries epsilon and the learner's DQN statistics.  --prioritized-replay and --n-step turn on `dqn.DQNConfig`'s
prioritized replay and n-step returns (Ape-X DQN's replay side); the statistics then include the mean importance
weight, weight_mean.
"""
import argparse
import json
import time

import torch

from .config import DEFAULT_EXTRA_CONFIG

C2_SETTINGS = dict(DEFAULT_EXTRA_CONFIG)        # robot_gym_env.py's defaults are BASELINE config C2
ZIGZAG_STEPS = 235.0


class EpisodeLengths(object):
    """Lengths of the episodes that end inside each fragment (running step counts cut at `done`)."""

    def __init__(self, B, device):
        self.carry = torch.zeros(B, dtype=torch.float64, device=device)

    def update(self, done):
        d = done.bool()
        T = d.shape[0]
        cs = self.carry.unsqueeze(0) + torch.arange(1, T + 1, dtype=torch.float64, device=d.device).unsqueeze(1)
        at_done = torch.where(d, cs, torch.zeros_like(cs))
        seen = torch.cummax(at_done, dim=0).values
        prev = torch.cat([torch.zeros_like(seen[:1]), seen[:-1]], dim=0)
        self.carry = cs[-1] - seen[-1]
        return torch.where(d, cs - prev, torch.zeros_like(cs)).sum()


# C2's spaces (robot_gym_env.py's class defaults): what every run used before the spaces could be chosen
C2_SPACES = dict(action_mode='discrete', action_shape=1, granularity=4, obs_mode='section', obs_grad=4)


def check_spaces(algo, action_mode, action_shape, granularity, obs_mode, obs_grad):
    """Raise ValueError for spaces this trainer cannot train: shapes the act and learner kernels do not take (obs_dim
    <= 32, n_out <= 15), and DQN with continuous actions.  Returns (obs_dim, n_out)."""
    from .config import _OBS_MODES, obs_dim
    if algo not in ('ppo', 'dqn'):
        raise ValueError('algo must be ppo or dqn, not %r' % (algo,))
    if action_mode not in ('discrete', 'continuous'):
        raise ValueError('action mode must be discrete or continuous, not %r' % (action_mode,))
    if obs_mode not in _OBS_MODES:
        raise ValueError('obs mode must be one of %s, not %r' % (sorted(_OBS_MODES), obs_mode))
    if obs_grad < 1:
        raise ValueError('obs grad must be positive, not %d' % obs_grad)
    od = obs_dim(obs_mode, obs_grad)
    if od > 32:
        raise ValueError('the %s observation with grad %d has %d entries; the policy kernels take at most 32' % (obs_mode, obs_grad, od))
    if action_mode == 'continuous':
        if algo == 'dqn':
            raise ValueError('DQN takes discrete actions only; train continuous actions with --algo ppo')
        if action_shape not in (1, 2):
            raise ValueError('action shape must be 1 or 2, not %r' % (action_shape,))
        return od, 2 * action_shape
    if not 1 <= granularity <= 15:
        raise ValueError('granularity %d: the policy kernels take 1..15 discrete actions' % granularity)
    return od, granularity


def make_env(part, num_envs, seed, device, spaces=None):
    from .batched_env import BatchedPaintEnv
    from .config import EnvConfig
    sp = dict(C2_SPACES, **(spaces or {}))
    cfg = EnvConfig(dict(C2_SETTINGS, Part_NO=int(part)), action_mode=sp['action_mode'], action_shape=sp['action_shape'],
                    discrete_granularity=sp['granularity'], obs_mode=sp['obs_mode'], obs_grad=sp['obs_grad'], auto_reset=True,
                    seed=seed)
    return BatchedPaintEnv(num_envs, cfg, device=device)


def max_points(env):
    return env.cfg.max_possible_point if env.cfg.max_possible_point is not None else env.pack.max_points


class Trainer(object):
    """One environment batch, one policy, one worker, one learner; `iteration()` collects a fragment and learns on it.
    `spaces` overrides C2_SPACES.  `dist` is the continuous policy's distribution: 'diag_gaussian' (the default, RLlib's
    DiagGaussian with a learned log-std) or 'tanh_gaussian' (unit variance around tanh(mean))."""

    def __init__(self, part=0, num_envs=4096, fragment_length=100, seed=0, device='cuda:0', config=None, use_cuda_graph=True,
                 algo='ppo', total_samples=2000000, spaces=None, dist=None):
        from .rollout import MlpPolicy, RolloutWorker
        self.spaces = dict(C2_SPACES, **(spaces or {}))
        unknown = set(self.spaces) - set(C2_SPACES)
        if unknown:
            raise ValueError('unknown spaces: %s' % sorted(unknown))
        check_spaces(algo, **self.spaces)
        discrete = self.spaces['action_mode'] == 'discrete'
        dist = dist or ('categorical' if discrete else 'diag_gaussian')
        self.algo, self.total_samples = algo, int(total_samples)
        self.device = torch.device(device)
        self.env = make_env(part, num_envs, seed, self.device, self.spaces)
        self.policy = MlpPolicy(self.env.obs_dim, self.spaces['granularity'] if discrete else self.env.action_dim,
                                device=self.device, seed=seed, discrete=discrete, dist=dist)
        if algo == 'ppo':
            from .ppo import PPOConfig, PPOLearner
            self.epsilon = None
            self.worker = RolloutWorker(self.env, self.policy, fragment_length=fragment_length, use_cuda_graph=use_cuda_graph, keep_logits=True)
            self.learner = PPOLearner(self.policy, config if config is not None else PPOConfig(seed=seed))
        else:
            from .dqn import DQNConfig, DQNLearner
            self.epsilon = torch.ones(1, dtype=torch.float32, device=self.device)
            self.worker = RolloutWorker(self.env, self.policy, fragment_length=fragment_length, use_cuda_graph=use_cuda_graph,
                                        epsilon=self.epsilon)
            self.learner = DQNLearner(self.policy, config if config is not None else DQNConfig(seed=seed))
        self.lengths = EpisodeLengths(num_envs, self.device)
        self.max_points = max_points(self.env)
        self.env_steps = 0
        self.worker.start((torch.arange(num_envs) % self.env.n_starts).numpy().astype('int32'))

    def iteration(self):
        eps = None
        if self.algo == 'dqn':
            from .dqn import epsilon_at
            eps = epsilon_at(self.learner.cfg, self.env_steps, self.total_samples)
            self.epsilon.fill_(eps)
        torch.cuda.synchronize(self.device)
        t0 = time.perf_counter()
        frag, st = self.worker.collect()
        ep_len = float(self.lengths.update(frag.done))            # host read: synchronises the collection
        t1 = time.perf_counter()
        ls = self.learner.update(frag)                            # ends in the read of its statistics
        t2 = time.perf_counter()
        self.env_steps += int(st['env_steps'])
        n_ep = st['episodes']
        r = dict(env_steps=self.env_steps, episodes=int(n_ep),
                 mean_return=st['sum_return'] / n_ep if n_ep else None,
                 coverage=st['sum_reward'] * 100.0 / self.max_points / n_ep if n_ep else None,
                 length_ratio=ep_len / n_ep / ZIGZAG_STEPS if n_ep else None,
                 collect_s=t1 - t0, learn_s=t2 - t1, learner=ls)
        if eps is not None:
            r['epsilon'] = eps
        return r

    def save(self, path):
        ck = {'learner': self.learner.state_dict(), 'obs_dim': self.policy.obs_dim, 'n_out': self.policy.n_out,
              'discrete': self.policy.discrete, 'env_settings': dict(C2_SETTINGS, Part_NO=self.env.cfg.part_no),
              'spaces': dict(self.spaces), 'dist': self.policy.dist}
        if self.algo != 'ppo':
            ck['algo'] = self.algo
        torch.save(ck, path)

    def close(self):
        self.learner.close()
        self.env.close()


def checkpoint_spaces(ck):
    """The spaces a checkpoint of this script was trained in (C2's for checkpoints that predate recording them)."""
    return dict(C2_SPACES, **ck.get('spaces', {}))


def load_policy(path, device):
    """A trained `rollout.MlpPolicy` from a checkpoint of this script (PPO, or DQN when it records algo 'dqn').  For a
    DQN policy the argmax of the head outputs' first n_out columns is the greedy action: Q differs from them by a
    per-state constant, so only the tie rule can differ (the first maximum of the advantages vs. of Q).  A
    diagonal-Gaussian policy's mean action is its head's first `action_dim` columns; `checkpoint_spaces` gives the
    environment spaces to drive it in."""
    from .ppo import check_state_dict, state_dist, unflatten_into
    from .rollout import MlpPolicy
    ck = torch.load(path, map_location='cpu', weights_only=False)
    dist = ck.get('dist') or state_dist(ck['learner'])
    n_out = ck['n_out'] // 2 if dist == 'diag_gaussian' else ck['n_out']
    pol = MlpPolicy(ck['obs_dim'], n_out, device=device, discrete=ck['discrete'], dist=dist)
    if ck.get('algo', 'ppo') == 'dqn':
        from .dqn import check_state_dict as check_dqn_state_dict
        check_dqn_state_dict(ck['learner'], ck['obs_dim'], ck['n_out'])
    else:
        check_state_dict(ck['learner'], ck['obs_dim'], ck['n_out'], ck['discrete'], dist)
    unflatten_into(pol, ck['learner']['params'].to(device))
    return pol


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--part', type=int, default=0, help='Part_NO (0: door, 1: sheet)')
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--fragment', type=int, default=100, help='steps per fragment (sample_batch_size)')
    ap.add_argument('--iters', type=int, default=None, help='iterations (default: as many as --samples needs)')
    ap.add_argument('--samples', type=int, default=2000000, help='env-step budget when --iters is not given')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--minibatch', type=int, default=None, help='SGD minibatch (multiple of 128)')
    ap.add_argument('--sgd-iters', type=int, default=None)
    ap.add_argument('--lr', type=float, default=None, help='Adam learning rate; PPO: 1e-3 (RLlib default 5e-5; 1e-3 learns faster on '
                    'the door, profiles/ppo_door_b200.json); DQN: DQNConfig\'s 5e-4')
    ap.add_argument('--checkpoint', default=None, help='write the learner state here at the end')
    ap.add_argument('--algo', choices=('ppo', 'dqn'), default='ppo', help='learner: PPO (default) or double DQN with a dueling head')
    ap.add_argument('--prioritized-replay', action='store_true', help='DQN: proportional prioritized replay (alpha 0.6, beta 0.4)')
    ap.add_argument('--n-step', type=int, default=None, help='DQN: n-step returns (default 1; Ape-X uses 3)')
    ap.add_argument('--action-mode', choices=('discrete', 'continuous'), default=C2_SPACES['action_mode'],
                    help='continuous: PPO with a diagonal-Gaussian head (learned log-std)')
    ap.add_argument('--action-shape', type=int, choices=(1, 2), default=None, help='continuous action dimensions (default 2)')
    ap.add_argument('--granularity', type=int, default=None, help='discrete actions (default 4; 1..15)')
    ap.add_argument('--obs-mode', choices=('section', 'grid', 'simple', 'discrete'), default=C2_SPACES['obs_mode'])
    ap.add_argument('--obs-grad', type=int, default=C2_SPACES['obs_grad'], help='observation granularity (default 4)')
    args = ap.parse_args(argv)
    if args.algo != 'dqn' and (args.prioritized_replay or args.n_step is not None):
        ap.error('--prioritized-replay and --n-step apply to --algo dqn')
    continuous = args.action_mode == 'continuous'
    if args.action_shape is not None and not continuous:
        ap.error('--action-shape applies to --action-mode continuous')
    if args.granularity is not None and continuous:
        ap.error('--granularity applies to --action-mode discrete')
    spaces = dict(action_mode=args.action_mode, action_shape=args.action_shape or (2 if continuous else 1),
                  granularity=args.granularity or C2_SPACES['granularity'], obs_mode=args.obs_mode, obs_grad=args.obs_grad)
    try:
        check_spaces(args.algo, **spaces)
    except ValueError as exc:
        ap.error(str(exc))
    if args.algo == 'dqn':
        from .dqn import DQNConfig
        kw = {k: v for k, v in (('minibatch_size', args.minibatch), ('lr', args.lr), ('n_step', args.n_step)) if v is not None}
        if args.prioritized_replay:
            kw['prioritized_replay'] = True
        tr = Trainer(args.part, args.envs, args.fragment, args.seed, config=DQNConfig(seed=args.seed, **kw), algo='dqn',
                     total_samples=args.samples, spaces=spaces)
    else:
        from .ppo import PPOConfig
        lr = args.lr if args.lr is not None else 1e-3
        kw = {k: v for k, v in (('minibatch_size', args.minibatch), ('num_sgd_iter', args.sgd_iters), ('lr', lr)) if v is not None}
        tr = Trainer(args.part, args.envs, args.fragment, args.seed, config=PPOConfig(seed=args.seed, **kw), spaces=spaces)
    iters = args.iters if args.iters is not None else -(-args.samples // (args.envs * args.fragment))
    t0 = time.perf_counter()
    for it in range(iters):
        r = tr.iteration()
        r['iteration'] = it
        r['wall_s'] = time.perf_counter() - t0
        print(json.dumps(r), flush=True)
    if args.checkpoint:
        tr.save(args.checkpoint)
    tr.close()


if __name__ == '__main__':
    main()
