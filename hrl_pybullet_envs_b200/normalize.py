"""Running observation and reward normalization (Stable-Baselines3 ``VecNormalize``) on the device.

The statistics are kept by the kernels of include/hrl_b200.h (``hrl_obs_moments``, ``hrl_reward_scale``) in float64; torch
only holds the buffers.  ``VecEnv.rollout_mlp(..., obs_norm=norm)`` feeds the in-kernel policy the normalized observation
(``hrl_rollout_mlp_norm``).
"""
import ctypes as C

import torch

from . import _cabi


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class RunningNormalizer:
    """SB3 ``VecNormalize`` statistics for N envs with D-dimensional observations.

    ``env_or_dims``: a ``VecEnv`` (its N, D and device) or a tuple ``(N, D)`` / ``(N, D, device)``.
    Holds the observation moments ``obs_moments`` f64[1 + 2D] = {count, mean[D], var[D]} with the float32 ``mean`` and
    ``rstd`` = 1 / sqrt(var + epsilon) the rollout reads, the return moments ``ret_moments`` f64[3] = {count, mean, var},
    the per-env discounted returns ``returns`` f64[N] and a work buffer; all allocated once.  Initial state as SB3:
    count = 1e-4, mean = 0, var = 1, returns = 0.  No method synchronises with the host.

    The one difference from SB3: the observation statistics are frozen for a rollout (``update_obs`` after it), where
    SB3 updates them every step.  Reward scaling follows SB3 step by step."""

    def __init__(self, env_or_dims, gamma=0.99, clip_obs=10.0, clip_reward=10.0, epsilon=1e-8):
        if isinstance(env_or_dims, tuple):
            N, D = int(env_or_dims[0]), int(env_or_dims[1])
            dev = torch.device(env_or_dims[2]) if len(env_or_dims) > 2 else torch.device("cuda", torch.cuda.current_device())
        else:
            N, D, dev = env_or_dims.N, env_or_dims.D, env_or_dims.device
        if N < 1 or not 1 <= D <= 64:
            raise ValueError("RunningNormalizer needs N >= 1 and 1 <= D <= 64, got N = %d, D = %d" % (N, D))
        if not 0.0 <= gamma <= 1.0:
            raise ValueError("gamma must lie in [0, 1], got %r" % (gamma,))
        for name, v in (("clip_obs", clip_obs), ("clip_reward", clip_reward), ("epsilon", epsilon)):
            if not (v > 0.0 and v < float("inf")):
                raise ValueError("%s must be finite and > 0, got %r" % (name, v))
        self.N, self.D, self.device = N, D, dev
        self.gamma, self.clip_obs, self.clip_reward, self.epsilon = float(gamma), float(clip_obs), float(clip_reward), float(epsilon)
        f64 = dict(dtype=torch.float64, device=dev)
        self.obs_moments = torch.zeros(1 + 2 * D, **f64)
        self.mean = torch.zeros(D, dtype=torch.float32, device=dev)
        self.rstd = torch.zeros(D, dtype=torch.float32, device=dev)
        self.ret_moments = torch.zeros(3, **f64)
        self.returns = torch.zeros(N, **f64)
        self._work = torch.zeros(0, **f64)
        self._clip32 = torch.tensor(self.clip_obs, dtype=torch.float32).item()
        self.reset_statistics()

    def reset_statistics(self):
        """SB3's initial state: count = 1e-4, mean = 0, var = 1 for observations and returns; returns = 0."""
        D = self.D
        self.obs_moments.zero_()
        self.obs_moments[0] = 1e-4
        self.obs_moments[1 + D:] = 1.0
        self.mean.zero_()
        self.rstd.copy_((1.0 / torch.sqrt(torch.ones(D, dtype=torch.float64) + torch.tensor(self.epsilon, dtype=torch.float32).double()))
                        .to(torch.float32))
        self.ret_moments.copy_(torch.tensor([1e-4, 0.0, 1.0], dtype=torch.float64))
        self.returns.zero_()

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, name, t, shape=None, dtypes=(torch.float32,)):
        if not isinstance(t, torch.Tensor) or t.dtype not in dtypes or not t.is_contiguous() or t.device != self.device \
                or (shape is not None and tuple(t.shape) != tuple(shape)):
            what = "[%s]" % ", ".join(map(str, shape)) if shape is not None else "[..., %d]" % self.D
            raise ValueError("%s must be a contiguous %s tensor %s on %s" % (name, "/".join(str(d).replace("torch.", "") for d in dtypes),
                                                                         what, self.device))

    def update_obs(self, x):
        """Merge the observations ``x`` (contiguous float32 CUDA tensor [..., D]) into the statistics, in one launch
        (``hrl_obs_moments``), and refresh ``mean`` and ``rstd``.  Call it with the ``vec.reset()`` output once, then with
        ``buf.obs[1:]`` after each rollout: SB3 counts reset and post-step observations, not terminal ones."""
        self._check("x", x)
        if x.dim() < 1 or x.shape[-1] != self.D or x.numel() == 0:
            raise ValueError("x must be a non-empty tensor [..., %d], got shape %s" % (self.D, tuple(x.shape)))
        M = x.numel() // self.D
        if M >= 2 ** 31:
            raise ValueError("x holds %d rows; at most 2^31 - 1 per call" % M)
        with torch.cuda.device(self.device):
            _cabi.check(_cabi.lib().hrl_obs_moments(M, self.D, _ptr(x), _ptr(self.obs_moments), self.epsilon, _ptr(self.mean),
                                                    _ptr(self.rstd), self._stream()))

    def normalize(self, obs):
        """clamp((obs - mean) * rstd, -clip_obs, clip_obs) in float32: bit for bit the input the in-kernel policy of
        ``rollout_mlp(..., obs_norm=self)`` saw (for finite observations)."""
        return torch.clamp((obs - self.mean) * self.rstd, -self._clip32, self._clip32)

    def scale_rewards(self, rew, done, out=None):
        """SB3's reward normalization over a [T, N] buffer, in three launches (``hrl_reward_scale``): per step, the
        discounted returns are updated, their moments merged, and the rewards divided by sqrt(var + epsilon) and clipped
        to +-clip_reward.  The returns carry over to the next call and restart where ``done``.  ``rew`` float32 [T, N],
        ``done`` bool / uint8 [T, N], ``out`` float32 [T, N] (allocated when None; must not overlap ``rew``).  Returns out."""
        self._check("rew", rew)
        if rew.dim() != 2 or rew.shape[1] != self.N or rew.shape[0] < 1:
            raise ValueError("rew must be a [T, %d] tensor, got shape %s" % (self.N, tuple(rew.shape)))
        T = rew.shape[0]
        self._check("done", done, (T, self.N), (torch.bool, torch.uint8))
        if out is None:
            out = torch.empty_like(rew)
        else:
            self._check("out", out, (T, self.N))
            if out.data_ptr() == rew.data_ptr():
                raise ValueError("out must not overlap rew")
        if self._work.numel() < 2 * T:
            self._work = torch.zeros(2 * T, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(_cabi.lib().hrl_reward_scale(T, self.N, self.gamma, self.clip_reward, self.epsilon, _ptr(rew), _ptr(done),
                                                     _ptr(self.returns), _ptr(self.ret_moments), _ptr(self._work), _ptr(out),
                                                     self._stream()))
        return out

    def reset_returns(self, mask=None):
        """Zero the discounted returns of all envs, or of those where ``mask`` (bool [N]) is set: for an explicit
        ``vec.reset()``, which SB3 treats like a done."""
        if mask is None:
            self.returns.zero_()
        else:
            m = torch.as_tensor(mask, device=self.device)
            if m.shape != (self.N,):
                raise ValueError("mask must have %d entries, got shape %s" % (self.N, tuple(m.shape)))
            self.returns.masked_fill_(m.to(torch.bool), 0.0)

    def state_dict(self):
        """Everything needed to resume: the moments, the per-env returns and the settings (tensors are copies)."""
        return dict(obs_moments=self.obs_moments.clone(), ret_moments=self.ret_moments.clone(), returns=self.returns.clone(),
                    gamma=self.gamma, clip_obs=self.clip_obs, clip_reward=self.clip_reward, epsilon=self.epsilon)

    def load_state_dict(self, sd):
        for k in ("gamma", "clip_obs", "clip_reward", "epsilon"):
            if float(sd[k]) != getattr(self, k):
                raise ValueError("state_dict has %s = %r, this normalizer %r" % (k, sd[k], getattr(self, k)))
        for k, shape in (("obs_moments", (1 + 2 * self.D,)), ("ret_moments", (3,)), ("returns", (self.N,))):
            if tuple(sd[k].shape) != shape:
                raise ValueError("state_dict %s has shape %s, expected %s" % (k, tuple(sd[k].shape), shape))
            getattr(self, k).copy_(sd[k])
        D = self.D
        self.mean.copy_(self.obs_moments[1:1 + D].to(torch.float32))
        self.rstd.copy_((1.0 / torch.sqrt(self.obs_moments[1 + D:] + torch.tensor(self.epsilon, dtype=torch.float32).double()))
                        .to(torch.float32))
