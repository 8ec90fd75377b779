"""Train the rollout policy with PPO on one GPU: collection and learning both on the device.

    python -m paintrl_b200.train --part 0 --envs 4096 --fragment 100 --samples 8000000 --seed 0 --checkpoint door.pt

Environment: BASELINE config C2 (RGB, section-4 observation, discrete-4 actions, late termination, anchor start points,
auto-reset) on the chosen part.  Policy: paint_ppo.py's [256, 128] MLP, sampled by the act kernel inside a captured
CUDA graph; the learner (`ppo.PPOLearner`) refreshes the kernel's weights in place after every minibatch.

Per iteration one JSON line: env-steps so far, the ended episodes' mean return, mean coverage ratio (episode `reward`
total x 100 / the part's max points; RGB) and mean length / 235 (the zigzag baseline's steps to full coverage), and the
collection and learner times (host clock around work that ends in a device synchronisation).
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


def make_env(part, num_envs, seed, device):
    from .batched_env import BatchedPaintEnv
    from .config import EnvConfig
    cfg = EnvConfig(dict(C2_SETTINGS, Part_NO=int(part)), auto_reset=True, seed=seed)
    return BatchedPaintEnv(num_envs, cfg, device=device)


def max_points(env):
    return env.cfg.max_possible_point if env.cfg.max_possible_point is not None else env.pack.max_points


class Trainer(object):
    """One environment batch, one policy, one worker, one learner; `iteration()` collects a fragment and learns on it."""

    def __init__(self, part=0, num_envs=4096, fragment_length=100, seed=0, device='cuda:0', config=None, use_cuda_graph=True):
        from .ppo import PPOConfig, PPOLearner
        from .rollout import MlpPolicy, RolloutWorker
        self.device = torch.device(device)
        self.env = make_env(part, num_envs, seed, self.device)
        self.policy = MlpPolicy(self.env.obs_dim, 4 if self.env.cfg.action_mode == 'discrete' else self.env.action_dim,
                                device=self.device, seed=seed, discrete=self.env.cfg.action_mode == 'discrete')
        self.worker = RolloutWorker(self.env, self.policy, fragment_length=fragment_length, use_cuda_graph=use_cuda_graph, keep_logits=True)
        self.learner = PPOLearner(self.policy, config if config is not None else PPOConfig(seed=seed))
        self.lengths = EpisodeLengths(num_envs, self.device)
        self.max_points = max_points(self.env)
        self.env_steps = 0
        self.worker.start((torch.arange(num_envs) % self.env.n_starts).numpy().astype('int32'))

    def iteration(self):
        torch.cuda.synchronize(self.device)
        t0 = time.perf_counter()
        frag, st = self.worker.collect()
        ep_len = float(self.lengths.update(frag.done))            # host read: synchronises the collection
        t1 = time.perf_counter()
        ls = self.learner.update(frag)                            # ends in the read of its statistics
        t2 = time.perf_counter()
        self.env_steps += int(st['env_steps'])
        eps = st['episodes']
        return dict(env_steps=self.env_steps, episodes=int(eps),
                    mean_return=st['sum_return'] / eps if eps else None,
                    coverage=st['sum_reward'] * 100.0 / self.max_points / eps if eps else None,
                    length_ratio=ep_len / eps / ZIGZAG_STEPS if eps else None,
                    collect_s=t1 - t0, learn_s=t2 - t1, learner=ls)

    def save(self, path):
        torch.save({'learner': self.learner.state_dict(), 'obs_dim': self.policy.obs_dim, 'n_out': self.policy.n_out,
                    'discrete': self.policy.discrete, 'env_settings': dict(C2_SETTINGS, Part_NO=self.env.cfg.part_no)}, path)

    def close(self):
        self.learner.close()
        self.env.close()


def load_policy(path, device):
    """A trained `rollout.MlpPolicy` from a checkpoint of this script."""
    from .ppo import check_state_dict, unflatten_into
    from .rollout import MlpPolicy
    ck = torch.load(path, map_location='cpu', weights_only=False)
    pol = MlpPolicy(ck['obs_dim'], ck['n_out'], device=device, discrete=ck['discrete'])
    check_state_dict(ck['learner'], ck['obs_dim'], ck['n_out'], ck['discrete'])
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
    ap.add_argument('--lr', type=float, default=1e-3, help='Adam learning rate (RLlib default 5e-5; 1e-3 learns faster on the door, '
                    'profiles/ppo_door_b200.json)')
    ap.add_argument('--checkpoint', default=None, help='write the learner state here at the end')
    args = ap.parse_args(argv)
    from .ppo import PPOConfig
    kw = {k: v for k, v in (('minibatch_size', args.minibatch), ('num_sgd_iter', args.sgd_iters), ('lr', args.lr)) if v is not None}
    tr = Trainer(args.part, args.envs, args.fragment, args.seed, config=PPOConfig(seed=args.seed, **kw))
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
