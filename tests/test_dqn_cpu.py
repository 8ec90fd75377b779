"""CPU: host-side logic of the double-DQN learner (paintrl_b200.dqn) -- configuration, the exploration schedule, the
replay ring's arithmetic on CPU tensors, checkpoint fields -- and the argument checks of its C ABI entry points.
The kernels themselves need the GPU: tests/test_gpu_dqn.py."""
import ctypes

import pytest
import torch

from paintrl_b200 import dqn, ppo
from paintrl_b200.rollout import RolloutFragment


def _lib():
    from paintrl_b200 import _capi, build
    build.build()
    return _capi.lib()


_FAKE = ctypes.c_void_p(256)     # a non-null pointer the argument checks reject before any launch


def test_config_defaults_validation_and_unknown_fields():
    c = dqn.DQNConfig()
    assert (c.lr, c.adam_eps, c.gamma, c.grad_clip) == (5e-4, 1e-8, 0.99, 40.0)
    assert (c.minibatch_size, c.replay_capacity, c.learning_starts, c.train_intensity, c.target_update_freq) == \
        (4096, 1 << 21, 65536, 8.0, 200)
    assert (c.epsilon_initial, c.epsilon_final, c.epsilon_fraction) == (1.0, 0.02, 0.1)
    assert dqn.DQNConfig.from_dict(c.to_dict()).to_dict() == c.to_dict()
    with pytest.raises(TypeError, match='unknown DQNConfig fields'):
        dqn.DQNConfig(learning_rate=1e-3)
    for bad in (dict(minibatch_size=1000), dict(minibatch_size=0), dict(replay_capacity=0), dict(target_update_freq=0),
                dict(learning_starts=-1), dict(train_intensity=0.0), dict(gamma=0.0), dict(gamma=1.5), dict(grad_clip=0.0),
                dict(epsilon_final=1.5), dict(epsilon_fraction=0.0)):
        with pytest.raises(ValueError):
            dqn.DQNConfig(**bad)
    assert dqn.DQNConfig(gamma=1.0).gamma == 1.0


def test_epsilon_schedule():
    c = dqn.DQNConfig()
    total = 2000000
    assert dqn.epsilon_at(c, 0, total) == 1.0
    assert dqn.epsilon_at(c, 100000, total) == pytest.approx(1.0 - 0.5 * 0.98)
    assert dqn.epsilon_at(c, 200000, total) == pytest.approx(0.02)
    assert dqn.epsilon_at(c, 10 ** 9, total) == pytest.approx(0.02)
    vals = [dqn.epsilon_at(c, s, total) for s in range(0, 400000, 409600 // 8)]
    assert all(a >= b for a, b in zip(vals, vals[1:]))
    c2 = dqn.DQNConfig(epsilon_initial=0.5, epsilon_final=0.1, epsilon_fraction=0.5)
    assert dqn.epsilon_at(c2, 250, 1000) == pytest.approx(0.3)


def test_grad_steps_per_update():
    c = dqn.DQNConfig()
    assert dqn.grad_steps_for(c, 409600) == 800                   # 8 x 409600 / 4096
    assert dqn.grad_steps_for(dqn.DQNConfig(minibatch_size=128, train_intensity=1.0), 129) == 2
    assert dqn.grad_steps_for(dqn.DQNConfig(minibatch_size=128, train_intensity=0.5), 256) == 1


def _fragment(T, B, obs_dim, base):
    """A fragment whose every entry encodes (t, b): obs = base + 1000 t + b (+ 0.25 per column), term_obs the negation."""
    f = RolloutFragment(T, B, obs_dim, (), torch.device('cpu'))
    t = torch.arange(T + 1, dtype=torch.float64)[:, None]
    b = torch.arange(B, dtype=torch.float64)[None, :]
    code = base + 1000.0 * t + b
    f.obs.copy_(code[:, :, None] + 0.25 * torch.arange(obs_dim, dtype=torch.float64))
    f.term_obs.copy_(-f.obs[:T])
    f.actions.copy_((code[:T] % 4).to(torch.int64))
    f.actual.copy_(code[:T] * 0.5)
    f.done.copy_((code[:T].to(torch.int64) % 3 == 0).to(torch.uint8))
    return f


def test_replay_ring_rows_wraparound_and_next_obs():
    T, B, obs_dim = 3, 4, 2
    buf = dqn.ReplayBuffer(20, obs_dim, 'cpu')
    frags = [_fragment(T, B, obs_dim, 100000.0 * k) for k in range(3)]
    expect = {}                                   # ring row -> (fragment, t, b) of the latest writer
    pos = 0
    for k, f in enumerate(frags):
        buf.add(f)
        for t in range(T):
            for b in range(B):
                expect[(pos + t * B + b) % 20] = (k, t, b)
        pos = (pos + T * B) % 20
        assert buf.pos == pos and buf.size == min(20, (k + 1) * T * B)
    assert buf.pos == 16 and buf.size == 20       # 36 rows into 20: the second fragment wrapped at row 20
    for row, (k, t, b) in expect.items():
        f = frags[k]
        assert torch.equal(buf.obs[row], f.obs[t, b])
        assert torch.equal(buf.next_obs[row], f.term_obs[t, b])           # s' is term_obs[t] ...
        assert not torch.equal(buf.next_obs[row], f.obs[t + 1, b])        # ... not the reset observation obs[t + 1]
        assert buf.actions[row] == f.actions[t, b]
        assert buf.reward[row] == torch.tensor(float(f.actual[t, b]), dtype=torch.float32)
        assert buf.done[row] == f.done[t, b]
    # the second fragment went to rows 12..19 and 0..3, the third to rows 4..15
    assert expect[16] == (1, 1, 0) and expect[0] == (1, 2, 0) and expect[3] == (1, 2, 3)
    assert expect[4] == (2, 0, 0) and expect[15] == (2, 2, 3)


def test_replay_fragment_larger_than_the_ring_keeps_its_last_rows():
    T, B = 4, 4
    buf = dqn.ReplayBuffer(10, 1, 'cpu')
    buf.add(_fragment(1, 3, 1, 0.0))              # pos 3
    f = _fragment(T, B, 1, 5000.0)
    buf.add(f)
    assert buf.size == 10 and buf.pos == (3 + 16) % 10
    flat = f.obs[:T].reshape(-1)
    for i in range(6, 16):                        # the last 10 rows land at (3 + i) % 10
        assert buf.obs[(3 + i) % 10, 0] == flat[i]


def test_replay_sampling_covers_only_filled_rows():
    buf = dqn.ReplayBuffer(1000, 1, 'cpu')
    gen = torch.Generator().manual_seed(0)
    with pytest.raises(ValueError):
        buf.sample(8, gen)
    buf.add(_fragment(5, 7, 1, 0.0))             # 35 rows
    idx = buf.sample(20000, gen)
    assert idx.dtype == torch.int32 and int(idx.min()) == 0 and int(idx.max()) == 34
    assert torch.bincount(idx.long()).numel() == 35


def test_state_dict_round_trip_and_shape_checks(tmp_path):
    n = ppo.num_params(6, 4)
    cfg = dqn.DQNConfig(lr=1e-4, minibatch_size=1024, seed=3)
    sd = {'algo': 'dqn', 'config': cfg.to_dict(), 'obs_dim': 6, 'n_out': 4, 'discrete': True,
          'params': torch.arange(n, dtype=torch.float32), 'target_params': -torch.arange(n, dtype=torch.float32),
          'adam_m': torch.zeros(n), 'adam_v': torch.ones(n), 'step': 77, 'generator': torch.Generator().manual_seed(5).get_state()}
    path = tmp_path / 'dqn.pt'
    torch.save(sd, path)
    back = torch.load(path, weights_only=False)
    dqn.check_state_dict(back, 6, 4)
    assert back['step'] == 77 and back['config'] == cfg.to_dict() and back['algo'] == 'dqn'
    assert torch.equal(back['target_params'], sd['target_params']) and torch.equal(back['generator'], sd['generator'])
    with pytest.raises(ValueError):
        dqn.check_state_dict(back, 6, 3)
    with pytest.raises(ValueError):
        dqn.check_state_dict(dict(back, discrete=False), 6, 4)
    with pytest.raises(ValueError):
        dqn.check_state_dict(dict(back, target_params=torch.zeros(n + 1)), 6, 4)
    with pytest.raises(ValueError):
        dqn.check_state_dict({k: v for k, v in back.items() if k != 'target_params'}, 6, 4)
    with pytest.raises(ValueError):
        dqn.check_state_dict(dict(back, step=-1), 6, 4)


def test_learner_refuses_continuous_policies_and_cpu_devices():
    from paintrl_b200.rollout import MlpPolicy
    with pytest.raises(ValueError, match='discrete'):
        dqn.DQNLearner(MlpPolicy(6, 2, device=torch.device('cpu'), discrete=False))
    with pytest.raises(ValueError, match='CUDA'):
        dqn.DQNLearner(MlpPolicy(6, 4, device=torch.device('cpu')))


def test_entry_points_check_their_arguments():
    lib = _lib()
    from paintrl_b200 import _capi
    F = _FAKE
    # epsilon-greedy act
    assert lib.paintrl_policy_act_epsilon(None, F, 128, F, F, None, F, None) == -1 and b'null handle' in lib.paintrl_last_error()
    # grad
    assert lib.paintrl_dqn_grad(None, F, F, F, 128, F, F, F, F, F, F, F, None) == -1 and b'null handle' in lib.paintrl_last_error()
    lib.paintrl_dqn_destroy(None)
    # clipping
    assert lib.paintrl_clip_grad_norm(None, 10, 1.0, F, None) == -1 and b'null' in lib.paintrl_last_error()
    assert lib.paintrl_clip_grad_norm(F, 10, 1.0, None, None) == -1 and b'null' in lib.paintrl_last_error()
    assert lib.paintrl_clip_grad_norm(F, 0, 1.0, F, None) == -1 and b'n must be positive' in lib.paintrl_last_error()
    for bad in (0.0, -1.0, float('nan')):
        assert lib.paintrl_clip_grad_norm(F, 10, bad, F, None) == -1 and b'max_norm' in lib.paintrl_last_error()
    # create
    out = ctypes.c_void_p()
    assert lib.paintrl_dqn_create(None, 0, ctypes.byref(out)) == -1
    good = dict(abi_version=_capi.PAINTRL_ABI_VERSION, obs_dim=6, n_out=4, max_minibatch=4096, gamma=0.99)
    for bad, msg in ((dict(abi_version=1), b'ABI'), (dict(obs_dim=33), b'observations'), (dict(obs_dim=0), b'observations'),
                     (dict(n_out=16), b'action outputs'), (dict(n_out=0), b'action outputs'), (dict(max_minibatch=0), b'max_minibatch'),
                     (dict(gamma=0.0), b'gamma'), (dict(gamma=1.01), b'gamma'), (dict(gamma=float('nan')), b'gamma')):
        cfg = _capi.PaintrlDqnConfig(**dict(good, **bad))
        assert lib.paintrl_dqn_create(ctypes.byref(cfg), 0, ctypes.byref(out)) == -1, bad
        assert msg in lib.paintrl_last_error(), (bad, lib.paintrl_last_error())
        assert not out.value
    if not torch.cuda.is_available():
        cfg = _capi.PaintrlDqnConfig(**dict(good, gamma=1.0))
        assert lib.paintrl_dqn_create(ctypes.byref(cfg), 0, ctypes.byref(out)) == -2
        assert b'no CPU fallback' in lib.paintrl_last_error()
        assert not out.value
