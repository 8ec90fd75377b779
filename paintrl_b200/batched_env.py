"""`BatchedPaintEnv` -- thousands of independent PaintRL environments resident on one GPU.

Host-side mirror of the reference's per-environment interface
(PaintRLEnv/robot_gym_env.py:207-422, PaintRLEnv/bullet_paint_wrapper.py:1327-1400) over the C ABI
of include/paintrl.h.  PyTorch is used for device memory and streams only; every result comes
from the CUDA library (there is no CPU fallback -- construction fails without it).
"""
import ctypes

import numpy as np
import torch

from . import _capi
from .config import EnvConfig
from .partpack import PartPack


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def check_subset(ids_or_range, num_envs):
    """Validate a subset of a batch of `num_envs` environments once, so that stepping it needs no further check.

    `ids_or_range` is a `range` with step 1 (a contiguous group: returns (None, lo, n)) or a list / array / tensor of
    environment ids (returns (ids, 0, n), ids an int32 NumPy array, or an int32 tensor on the given CUDA tensor's
    device).  Ids must be integers, in [0, num_envs) and unique, and the subset must not be empty: the kernels index
    per-environment state with them, so a duplicate would race and an id out of range would touch no environment.
    A CUDA tensor is checked with one reduction and one synchronisation."""
    if isinstance(ids_or_range, range):
        r = ids_or_range
        if r.step != 1:
            raise ValueError('a subset range must have step 1, got %d' % r.step)
        if len(r) == 0:
            raise ValueError('the subset range is empty')
        if r.start < 0 or r.stop > num_envs:
            raise IndexError('subset range [%d, %d) outside [0, %d)' % (r.start, r.stop, num_envs))
        return None, r.start, len(r)
    if isinstance(ids_or_range, torch.Tensor) and ids_or_range.is_cuda:
        if ids_or_range.dtype.is_floating_point or ids_or_range.dtype.is_complex or ids_or_range.dtype == torch.bool:
            raise ValueError('env ids must be integers')
        ids = ids_or_range.reshape(-1)
        n = int(ids.numel())
        if n == 0:
            raise ValueError('the subset is empty')
        srt = torch.sort(ids.to(torch.int64)).values
        lo, hi, dup = torch.stack([srt[0], srt[-1], (srt[1:] == srt[:-1]).sum()]).tolist()
        host = None
    else:
        host = np.asarray(ids_or_range.cpu() if isinstance(ids_or_range, torch.Tensor) else ids_or_range).reshape(-1)
        n = int(host.size)
        if n == 0:
            raise ValueError('the subset is empty')
        if host.dtype.kind not in 'iu':
            raise ValueError('env ids must be integers')
        lo, hi = int(host.min()), int(host.max())
        dup = n - np.unique(host).size
    if lo < 0 or hi >= num_envs:
        raise IndexError('env ids out of range [0, %d): min %d, max %d' % (num_envs, lo, hi))
    if dup:
        raise ValueError('env ids must be unique')
    if host is None:
        return ids_or_range.reshape(-1).to(torch.int32).contiguous(), 0, n
    return host.astype(np.int32), 0, n


class EnvSubset(object):
    """A fixed subset of one `BatchedPaintEnv`'s environments (`BatchedPaintEnv.subset`): the device id list, or the
    range lo .. lo + n - 1 (`ids` None), and compact output tensors of n rows of its own, row k = the k-th listed
    environment, so that two subsets in flight never share buffers.  `env_ids` is the id of every row (int32, on the
    environment's device)."""

    def __init__(self, owner, ids, lo, n):
        self.owner = owner
        self.ids, self.lo, self.n = ids, lo, n
        dev, f64 = owner.device, torch.float64
        self.env_ids = ids if ids is not None else torch.arange(lo, lo + n, dtype=torch.int32, device=dev)
        self.obs = torch.zeros(n, owner.obs_dim, dtype=f64, device=dev)
        self.next_obs = torch.zeros(n, owner.obs_dim, dtype=f64, device=dev)
        self.reward = torch.zeros(n, dtype=f64, device=dev)
        self.penalty = torch.zeros(n, dtype=f64, device=dev)
        self.actual = torch.zeros(n, dtype=f64, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.new_texels = torch.zeros(n, dtype=torch.int32, device=dev)

    @property
    def is_range(self):
        return self.ids is None

    def __len__(self):
        return self.n


class BatchedPaintEnv(object):
    """`num_envs` PaintGymEnv instances sharing one part and one configuration.

    Args mirror PaintGymEnv (robot_gym_env.py:207-208, 126-157): `extra_config` carries the same
    keys; the class attributes ACTION_MODE/ACTION_SHAPE/DISCRETE_GRANULARITY/OBS_MODE/OBS_GRAD are
    keyword arguments here because one process can hold several configurations.
    """

    def __init__(self, num_envs, extra_config=None, action_mode='discrete', action_shape=1,
                 discrete_granularity=4, obs_mode='section', obs_grad=4, device=None,
                 auto_reset=False, seed=0, pack=None, texture_size=(240, 240), max_possible_point=None, urdf_root=None):
        if not torch.cuda.is_available():
            raise RuntimeError('paintrl_b200 needs a CUDA device: there is no CPU fallback')
        self.cfg = extra_config if isinstance(extra_config, EnvConfig) else EnvConfig(
            extra_config, action_mode=action_mode, action_shape=action_shape,
            discrete_granularity=discrete_granularity, obs_mode=obs_mode, obs_grad=obs_grad,
            auto_reset=auto_reset, seed=seed, max_possible_point=max_possible_point)
        self.device = torch.device(device if device is not None else 'cuda:%d' % torch.cuda.current_device())
        if self.device.type != 'cuda':
            raise RuntimeError('paintrl_b200 runs on CUDA devices only')
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.pack = pack if pack is not None else PartPack.for_part(self.cfg.part_no, *texture_size, device=dev_index,
                                                                          urdf_root=urdf_root)
        self.num_envs = int(num_envs)
        self._lib = _capi.lib()
        cpack, keep_pack = self.pack.to_c(self.cfg.start_point_mode, self.cfg.color_mode, with_nn_rep=self.cfg.paint_method == 'normal')
        ccfg, keep_cfg = self.cfg.to_c(self.pack.max_points, density=self.pack.meta.get('density'))
        handle = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        with torch.cuda.device(index):
            _capi.check(self._lib.paintrl_create(ctypes.byref(cpack), ctypes.byref(ccfg), self.num_envs,
                                                 index, ctypes.byref(handle)))
        del keep_pack, keep_cfg     # paintrl_create copied everything it needs
        self._h = handle
        self.obs_dim = int(self._lib.paintrl_obs_dim(self._h))
        self.action_dim = int(self._lib.paintrl_action_dim(self._h))
        self.n_texels = int(self._lib.paintrl_num_texels(self._h))
        self.state_bytes_per_env = int(self._lib.paintrl_state_bytes_per_env(self._h))
        self.n_starts = self.pack.start_points(self.cfg.start_point_mode).shape[0]
        B, f64 = self.num_envs, torch.float64
        dev = self.device
        self.obs = torch.zeros(B, self.obs_dim, dtype=f64, device=dev)
        self.next_obs = torch.zeros(B, self.obs_dim, dtype=f64, device=dev)
        self.reward = torch.zeros(B, dtype=f64, device=dev)
        self.penalty = torch.zeros(B, dtype=f64, device=dev)
        self.actual = torch.zeros(B, dtype=f64, device=dev)
        self.done = torch.zeros(B, dtype=torch.uint8, device=dev)
        self.new_texels = torch.zeros(B, dtype=torch.int32, device=dev)

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, '_h', None):
            self._lib.paintrl_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _ids(self, env_ids):
        """Device list of environment indices for the by-index entry points, validated on the host by
        `check_subset`: in range and unique (the kernels index states / planes with them; a duplicate would race,
        an out-of-range id corrupt another environment -- the device code also ignores ids out of range)."""
        if env_ids is None:
            return None, self.num_envs
        ids, _, n = check_subset(list(env_ids) if isinstance(env_ids, range) else env_ids, self.num_envs)
        return torch.as_tensor(ids, device=self.device).to(torch.int32).contiguous(), n

    # ------------------------------------------------------------------ reference call mirror
    def reset(self, start_index=None, env_ids=None):
        """PaintGymEnv.reset (robot_gym_env.py:370-387).  `start_index` plays the role of the
        reference's `randint(0, len(start_points) - 1)` draw (0 in rollout mode); None uses the
        library's seeded stream.  Returns the first observations [n, obs_dim]."""
        ids, n = self._ids(env_ids)
        si = None
        if start_index is not None:
            si = torch.as_tensor(start_index, dtype=torch.int32, device=self.device)
            si = si.expand(n).contiguous() if si.dim() == 0 else si.contiguous()
            if si.numel() != n:
                raise ValueError('start_index must have one entry per reset environment')
        out = self.obs if ids is None else torch.zeros(n, self.obs_dim, dtype=torch.float64, device=self.device)
        _capi.check(self._lib.paintrl_reset(self._h, _ptr(ids), n, _ptr(si), _ptr(out), self._stream()))
        if ids is None:
            self.next_obs.copy_(out)
        return out

    def set_pose(self, pos, normal, env_ids=None):
        """Robot.reset(pose) (robot.py:366-372) as spiral.py:28-38 uses it."""
        ids, n = self._ids(env_ids)
        pos = torch.as_tensor(pos, dtype=torch.float64, device=self.device).expand(n, 3).contiguous()
        normal = torch.as_tensor(normal, dtype=torch.float64, device=self.device).expand(n, 3).contiguous()
        out = torch.zeros(n, self.obs_dim, dtype=torch.float64, device=self.device)
        _capi.check(self._lib.paintrl_set_pose(self._h, _ptr(ids), n, _ptr(pos), _ptr(normal), _ptr(out),
                                               self._stream()))
        return out

    def subset(self, ids_or_range):
        """An `EnvSubset` of this batch to pass as `subset=` to `step`, `step_into` and (ranges only)
        `step_host_submit`: a `range` with step 1, or a list / array / tensor of unique environment ids.  Validated
        here, once (see `check_subset`); stepping a fixed subset needs no host synchronisation, so it can be captured
        in a CUDA graph."""
        ids, lo, n = check_subset(ids_or_range, self.num_envs)
        if ids is not None:
            ids = torch.as_tensor(ids, device=self.device).to(torch.int32).contiguous()
        return EnvSubset(self, ids, lo, n)

    def _rows(self, subset):
        if subset is None:
            return self.num_envs
        if not isinstance(subset, EnvSubset) or subset.owner is not self:
            raise ValueError('subset must be an EnvSubset made by this environment\'s subset()')
        return subset.n

    def _step_call(self, subset, actions, obs, reward, penalty, actual, done, new_texels, next_obs, rs):
        nxt = _ptr(next_obs) if self.cfg.auto_reset else None
        if subset is None:
            rc = self._lib.paintrl_step(self._h, _ptr(actions), _ptr(obs), _ptr(reward), _ptr(penalty), _ptr(actual),
                                        _ptr(done), _ptr(new_texels), nxt, _ptr(rs), self._stream())
        else:
            rc = self._lib.paintrl_step_subset(self._h, _ptr(subset.ids), subset.lo, subset.n, _ptr(actions), _ptr(obs),
                                               _ptr(reward), _ptr(penalty), _ptr(actual), _ptr(done), _ptr(new_texels),
                                               nxt, _ptr(rs), self._stream())
        _capi.check(rc)

    def step(self, actions, reset_start_index=None, subset=None):
        """PaintGymEnv.step for all environments (robot_gym_env.py:349-368), device tensors in and
        out, asynchronous on the current stream.  Returns (obs, actual_reward, done, info) where
        info = {'reward', 'penalty'} like robot_gym_env.py:368 plus 'next_obs' / 'new_texels'.
        With `subset` (an `EnvSubset`) only its n environments step: actions, reset_start_index and every output
        have n rows, row k = the k-th environment of the subset (info['env_ids'])."""
        B = self._rows(subset)
        if self.cfg.action_mode == 'discrete':
            a = torch.as_tensor(actions, device=self.device).to(torch.int64).contiguous()
            if a.numel() != B:
                raise ValueError('expected %d discrete actions' % B)
        else:
            a = torch.as_tensor(actions, device=self.device).to(torch.float64).contiguous()
            if a.numel() != B * self.action_dim:
                raise ValueError('expected actions of shape [%d, %d]' % (B, self.action_dim))
        rs = None
        if reset_start_index is not None:
            rs = torch.as_tensor(reset_start_index, dtype=torch.int32, device=self.device).contiguous()
            if rs.numel() != B:
                raise ValueError('reset_start_index must have one entry per environment (%d), got %d' % (B, rs.numel()))
        o = self if subset is None else subset
        self._step_call(subset, a, o.obs, o.reward, o.penalty, o.actual, o.done, o.new_texels, o.next_obs, rs)
        info = {'reward': o.reward, 'penalty': o.penalty, 'new_texels': o.new_texels,
                'next_obs': o.next_obs if self.cfg.auto_reset else o.obs}
        if subset is not None:
            info['env_ids'] = subset.env_ids
        return o.obs, o.actual, o.done, info

    def step_into(self, actions, obs, reward, penalty, actual, done, next_obs=None, new_texels=None, subset=None):
        """`step` writing straight into caller tensors (e.g. row t of a rollout fragment): contiguous
        CUDA tensors of this environment's device, float64 [B, obs_dim] / [B], uint8 [B], int32 [B];
        `actions` int64 [B] or float64 [B, action_dim].  Nothing is returned and nothing is copied.
        With `subset`, B is the subset's size and row k belongs to its k-th environment."""
        B = self._rows(subset)
        want = (torch.int64, B) if self.cfg.action_mode == 'discrete' else (torch.float64, B * self.action_dim)
        for t, (dt, n) in ((actions, want), (obs, (torch.float64, B * self.obs_dim)), (reward, (torch.float64, B)),
                           (penalty, (torch.float64, B)), (actual, (torch.float64, B)), (done, (torch.uint8, B)),
                           (next_obs, (torch.float64, B * self.obs_dim)), (new_texels, (torch.int32, B))):
            if t is None:
                continue
            if t.dtype != dt or t.numel() != n or not t.is_contiguous() or t.device != self.device:
                raise ValueError('step_into: expected a contiguous %s tensor of %d elements on %s' % (dt, n, self.device))
        self._step_call(subset, actions, obs, reward, penalty, actual, done, new_texels, next_obs, None)
        if next_obs is not None and not self.cfg.auto_reset:
            next_obs.copy_(obs)

    def step_host(self, actions, out=None):
        """The same step through HOST buffers (paintrl_step_host): actions are copied host->device
        and obs / reward / penalty / actual / done (/ next_obs) device->host inside the call."""
        B = self.num_envs
        discrete = self.cfg.action_mode == 'discrete'
        want = np.int64 if discrete else np.float64
        a = actions
        if not (isinstance(a, np.ndarray) and a.dtype == want and a.flags.c_contiguous):
            a = np.ascontiguousarray(actions, dtype=want)
        if a.size != (B if discrete else B * self.action_dim):
            raise ValueError('expected %d actions' % B)
        if out is None:
            out = self.host_buffers()
        ptrs = out.get('_ptrs')
        if ptrs is None:       # buffers not made by host_buffers(): resolve the addresses every call
            nxt = out.get('next_obs')
            ptrs = tuple(out[k].ctypes.data for k in ('obs', 'reward', 'penalty', 'actual', 'done')) + (
                nxt.ctypes.data if nxt is not None else None,)
        rc = self._lib.paintrl_step_host(self._h, a.ctypes.data, ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5],
                                         torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            _capi.check(rc)
        return out

    def step_host_submit(self, actions, out, slot=0, subset=None):
        """First half of `step_host` (paintrl_step_host_submit): queue the copy-in of `actions`, the step and the
        copy-out into `out` (from `host_buffers`) on staging slot 0 or 1 and return at once.  `actions` must stay
        untouched (and should be pinned) until `step_host_wait(slot)`.  Submitting step t + 1 on the other slot
        before waiting for step t overlaps its copy-in and kernels with step t's copy-out and the host's wake-up.
        With `subset` (a range `EnvSubset`, paintrl_step_host_submit_range) only that group steps; `actions` and
        `out` (`host_buffers(n=subset.n)`) have its n rows.  Two groups on the two slots let a closed-loop policy
        compute one group's actions while the other steps."""
        B = self._rows(subset)
        if subset is not None and not subset.is_range:
            raise ValueError('step_host_submit takes range subsets only (BatchedPaintEnv.subset(range(lo, hi)))')
        discrete = self.cfg.action_mode == 'discrete'
        want = np.int64 if discrete else np.float64
        a = actions
        if not (isinstance(a, np.ndarray) and a.dtype == want and a.flags.c_contiguous):
            a = np.ascontiguousarray(actions, dtype=want)
        if a.size != (B if discrete else B * self.action_dim):
            raise ValueError('expected %d actions' % B)
        if subset is not None and out['obs'].shape[0] != B:
            raise ValueError('host buffers of %d rows for a step of %d environments' % (out['obs'].shape[0], B))
        ptrs = out.get('_ptrs')
        if ptrs is None:
            nxt = out.get('next_obs')
            ptrs = tuple(out[k].ctypes.data for k in ('obs', 'reward', 'penalty', 'actual', 'done')) + (
                nxt.ctypes.data if nxt is not None else None,)
        self._inflight = getattr(self, '_inflight', {})
        self._inflight[slot] = (a, out)          # keep the buffers alive until the wait
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if subset is None:
            rc = self._lib.paintrl_step_host_submit(self._h, int(slot), a.ctypes.data, ptrs[0], ptrs[1], ptrs[2], ptrs[3],
                                                    ptrs[4], ptrs[5], stream)
        else:
            rc = self._lib.paintrl_step_host_submit_range(self._h, int(slot), subset.lo, subset.n, a.ctypes.data, ptrs[0],
                                                          ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5], stream)
        if rc != 0:
            _capi.check(rc)

    def step_host_wait(self, slot=0):
        """Second half: block until the results of `slot` have landed in its host buffers; returns them."""
        rc = self._lib.paintrl_step_host_wait(self._h, int(slot))
        if rc != 0:
            _capi.check(rc)
        return self._inflight.pop(slot)[1]

    def host_buffers(self, pinned=True, next_obs=True, n=None):
        """Host result buffers for `step_host`: views into ONE (pinned) allocation laid out
        obs | reward | penalty | actual | [next_obs] | done, the order `paintrl_step_host` stages its
        results in, so that they come back with a single device->host copy.  `n`: rows (a group of
        `step_host_submit(subset=...)`); default the whole batch."""
        B, od = (self.num_envs if n is None else int(n)), self.obs_dim
        n_f64 = B * (od * (2 if next_obs else 1) + 3)
        raw = torch.zeros(n_f64 * 8 + B, dtype=torch.uint8, pin_memory=pinned)
        f64 = raw[:n_f64 * 8].view(torch.float64).numpy()
        out = {'obs': f64[:B * od].reshape(B, od), 'reward': f64[B * od:B * od + B],
               'penalty': f64[B * od + B:B * od + 2 * B], 'actual': f64[B * od + 2 * B:B * od + 3 * B]}
        if next_obs:
            out['next_obs'] = f64[B * od + 3 * B:].reshape(B, od)
        out['done'] = raw[n_f64 * 8:].numpy()
        out['_storage'] = raw
        out['_ptrs'] = tuple(out[k].ctypes.data for k in ('obs', 'reward', 'penalty', 'actual', 'done')) + (
            out['next_obs'].ctypes.data if next_obs else None,)
        return out

    # ------------------------------------------------------------------ state
    def get_state(self, env_ids=None, status=True):
        ids, n = self._ids(env_ids)
        dev = self.device
        st = torch.zeros(n, self.n_texels, dtype=torch.int16, device=dev) if status else None
        pose = torch.zeros(n, 3, dtype=torch.float64, device=dev)
        quat = torch.zeros(n, 4, dtype=torch.float64, device=dev)
        scal = torch.zeros(n, _capi.PAINTRL_STATE_SCALARS, dtype=torch.float64, device=dev)
        _capi.check(self._lib.paintrl_get_state(self._h, _ptr(ids), n, _ptr(st), _ptr(pose), _ptr(quat),
                                                _ptr(scal), self._stream()))
        keys = ('total_reward', 'total_return', 'step_counter', 'term_counter', 'last_on_part',
                'terminate', 'last_angle', 'angle_diff', 'has_overlap_reference')
        out = {'status': st, 'pose': pose, 'quat': quat, 'scalars': scal}
        out.update({k: scal[:, i] for i, k in enumerate(keys)})
        out['overlap_reference_centre'] = scal[:, 9:12]
        return out

    def set_state(self, env_ids=None, status=None, pose=None, quat=None, scalars=None):
        """Import per-environment state (the tensors `get_state` returns).  `scalars` [n, 12] carries the overlap
        reference (Part._last_painted_pixels as the last shot's centre), so a mid-episode checkpoint restored
        into another engine continues bit for bit; a status plane without scalars clears that reference."""
        ids, n = self._ids(env_ids)

        def prep(t, dtype, shape):
            if t is None:
                return None
            t = torch.as_tensor(t, device=self.device).to(dtype).contiguous()
            if tuple(t.shape) != shape:
                raise ValueError('expected shape %s, got %s' % (shape, tuple(t.shape)))
            return t
        st = prep(status, torch.int16, (n, self.n_texels))
        po = prep(pose, torch.float64, (n, 3))
        qu = prep(quat, torch.float64, (n, 4))
        sc = prep(scalars, torch.float64, (n, _capi.PAINTRL_STATE_SCALARS))
        _capi.check(self._lib.paintrl_set_state(self._h, _ptr(ids), n, _ptr(st), _ptr(po), _ptr(qu), _ptr(sc),
                                                self._stream()))

    def job_status(self):
        """get_job_status per env (bullet_paint_wrapper.py:727-732)."""
        out = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        _capi.check(self._lib.paintrl_job_status(self._h, _ptr(out), self._stream()))
        return out

    def job_limit(self):
        """get_job_limit (bullet_paint_wrapper.py:734-735)."""
        return self.n_texels

    def stats(self):
        s = _capi.PaintrlStats()
        torch.cuda.synchronize(self.device)
        _capi.check(self._lib.paintrl_stats(self._h, ctypes.byref(s)))
        return {'env_steps': int(s.env_steps), 'episodes_ended': int(s.episodes_ended),
                'footprint_texels': int(s.footprint_texels), 'kernel_launches': int(s.kernel_launches),
                'ray_full_scans': int(s.ray_full_scans), 'move_bailouts': int(s.move_bailouts)}
