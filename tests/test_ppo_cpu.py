"""CPU: host-side logic of the PPO learner (paintrl_b200.ppo) and the argument checks of its C ABI entry points.
The kernels themselves need the GPU: tests/test_gpu_ppo.py."""
import ctypes

import pytest
import torch

from paintrl_b200 import ppo
from paintrl_b200.rollout import MlpPolicy


def _lib():
    from paintrl_b200 import _capi, build
    build.build()
    return _capi.lib()


_FAKE = ctypes.c_void_p(256)     # a non-null pointer the argument checks reject before any launch


def test_flat_parameter_layout():
    lib = _lib()
    for obs_dim, n_out in ((6, 4), (16, 2), (32, 15), (1, 1)):
        assert lib.paintrl_policy_num_params(obs_dim, n_out) == ppo.num_params(obs_dim, n_out)
    for obs_dim, n_out in ((0, 4), (33, 4), (6, 0), (6, 16)):
        assert lib.paintrl_policy_num_params(obs_dim, n_out) == -1
    pol = MlpPolicy(6, 4, device=torch.device('cpu'), seed=3)
    flat = ppo.flat_params(pol)
    assert flat.shape == (ppo.num_params(6, 4),) and flat.dtype == torch.float32
    w1, b1, w2, b2, w3, b3 = pol.weights()
    # w1 | b1 | w2 | b2 | w3 | b3, each row-major
    assert torch.equal(flat[:6 * 256].view(6, 256), w1)
    assert torch.equal(flat[6 * 256 + 256 + 3 * 128:6 * 256 + 256 + 4 * 128], w2[3])
    assert torch.equal(flat[-5:], b3) and torch.equal(flat[-5 - 128 * 5:-5].view(128, 5), w3)
    other = MlpPolicy(6, 4, device=torch.device('cpu'), seed=4)
    ppo.unflatten_into(other, flat)
    assert all(torch.equal(a, b) for a, b in zip(other.weights(), pol.weights()))


def test_shapes_the_kernel_does_not_take_are_refused():
    with pytest.raises(ValueError, match='observations'):
        ppo.check_policy(MlpPolicy(33, 4, device=torch.device('cpu')))
    with pytest.raises(ValueError, match='action outputs'):
        ppo.check_policy(MlpPolicy(6, 16, device=torch.device('cpu')))
    with pytest.raises(ValueError, match='hidden'):
        ppo.check_policy(MlpPolicy(6, 4, hiddens=(128, 128), device=torch.device('cpu')))
    ppo.check_policy(MlpPolicy(32, 15, device=torch.device('cpu')))
    with pytest.raises(ValueError):
        ppo.PPOConfig(minibatch_size=1000)
    with pytest.raises(TypeError):
        ppo.PPOConfig(learning_rate=1.0)


def test_kl_coeff_schedule():
    # RLlib PPO's update_kl around kl_target 0.01
    assert ppo.adapt_kl(0.2, 0.0201, 0.01) == pytest.approx(0.3)
    assert ppo.adapt_kl(0.2, 0.02, 0.01) == 0.2
    assert ppo.adapt_kl(0.2, 0.005, 0.01) == 0.2
    assert ppo.adapt_kl(0.2, 0.0049, 0.01) == pytest.approx(0.1)
    k = 0.2
    for _ in range(3):
        k = ppo.adapt_kl(k, 1.0, 0.01)
    assert k == pytest.approx(0.2 * 1.5 ** 3)


def test_minibatch_partitioning():
    assert ppo.minibatches(1024, 512) == [(0, 512), (512, 512)]
    assert ppo.minibatches(1000, 256) == [(0, 256), (256, 256), (512, 256), (768, 232)]
    assert ppo.minibatches(100, 4096) == [(0, 100)]
    for n_rows, size in ((409600, 4096), (12345, 1024), (1, 128)):
        mb = ppo.minibatches(n_rows, size)
        covered = [s + k for s, n in mb for k in range(n)] if n_rows < 20000 else None
        assert sum(n for _, n in mb) == n_rows and all(0 < n <= size for _, n in mb)
        assert all(mb[i][0] + mb[i][1] == mb[i + 1][0] for i in range(len(mb) - 1))
        if covered is not None:
            assert covered == list(range(n_rows))


def test_state_dict_host_fields_round_trip(tmp_path):
    cfg = ppo.PPOConfig(lr=3e-4, minibatch_size=2048, num_sgd_iter=4, seed=7)
    assert ppo.PPOConfig.from_dict(cfg.to_dict()).to_dict() == cfg.to_dict()
    n = ppo.num_params(6, 4)
    sd = {'config': cfg.to_dict(), 'obs_dim': 6, 'n_out': 4, 'discrete': True, 'params': torch.arange(n, dtype=torch.float32),
          'adam_m': torch.zeros(n), 'adam_v': torch.ones(n), 'step': 123, 'kl_coeff': 0.45,
          'generator': torch.Generator().manual_seed(5).get_state()}
    path = tmp_path / 'learner.pt'
    torch.save(sd, path)
    back = torch.load(path, weights_only=False)
    ppo.check_state_dict(back, 6, 4, True)
    assert back['step'] == 123 and back['kl_coeff'] == 0.45 and back['config'] == cfg.to_dict()
    assert torch.equal(back['params'], sd['params']) and torch.equal(back['generator'], sd['generator'])
    with pytest.raises(ValueError):
        ppo.check_state_dict(back, 6, 3, True)
    with pytest.raises(ValueError):
        ppo.check_state_dict(dict(back, params=torch.zeros(n - 1)), 6, 4, True)
    with pytest.raises(ValueError):
        ppo.check_state_dict(dict(back, step=-1), 6, 4, True)


def test_entry_points_check_their_arguments():
    lib = _lib()
    from paintrl_b200 import _capi
    F = _FAKE
    # null handles
    assert lib.paintrl_policy_set_params(None, F, None) == -1 and b'null handle' in lib.paintrl_last_error()
    assert lib.paintrl_ppo_grad(None, F, F, 128, F, F, F, F, F, F, F, 0.2, F, F, None) == -1
    assert b'null handle' in lib.paintrl_last_error()
    assert lib.paintrl_ppo_forward(None, F, F, 128, F, F, None) == -1 and b'null handle' in lib.paintrl_last_error()
    lib.paintrl_ppo_destroy(None)
    # create
    out = ctypes.c_void_p()
    assert lib.paintrl_ppo_create(None, 0, ctypes.byref(out)) == -1
    good = dict(abi_version=_capi.PAINTRL_ABI_VERSION, obs_dim=6, n_out=4, discrete=1, max_minibatch=4096, clip_param=0.3,
                vf_clip_param=10.0, vf_loss_coeff=1.0, entropy_coeff=0.0)
    for bad, msg in ((dict(abi_version=1), b'ABI'), (dict(obs_dim=33), b'observations'), (dict(n_out=16), b'action outputs'),
                     (dict(max_minibatch=0), b'max_minibatch'), (dict(clip_param=0.0), b'clip_param'),
                     (dict(vf_clip_param=-1.0), b'clip_param'), (dict(entropy_coeff=-0.1), b'entropy_coeff')):
        cfg = _capi.PaintrlPpoConfig(**dict(good, **bad))
        assert lib.paintrl_ppo_create(ctypes.byref(cfg), 0, ctypes.byref(out)) == -1, bad
        assert msg in lib.paintrl_last_error(), (bad, lib.paintrl_last_error())
        assert not out.value
    if not torch.cuda.is_available():
        cfg = _capi.PaintrlPpoConfig(**good)
        assert lib.paintrl_ppo_create(ctypes.byref(cfg), 0, ctypes.byref(out)) == -2
        assert b'no CPU fallback' in lib.paintrl_last_error()
    # Adam
    assert lib.paintrl_adam_step(None, F, F, F, 10, 1e-3, 0.9, 0.999, 1e-8, 1, None) == -1
    assert lib.paintrl_adam_step(F, F, F, F, 0, 1e-3, 0.9, 0.999, 1e-8, 1, None) == -1
    assert lib.paintrl_adam_step(F, F, F, F, 10, 1e-3, 0.9, 0.999, 1e-8, 0, None) == -1
    assert b'step' in lib.paintrl_last_error()
    assert lib.paintrl_adam_step(F, F, F, F, 10, 1e-3, 1.0, 0.999, 1e-8, 1, None) == -1
    assert lib.paintrl_adam_step(F, F, F, F, 10, 1e-3, 0.9, 0.999, 0.0, 1, None) == -1
