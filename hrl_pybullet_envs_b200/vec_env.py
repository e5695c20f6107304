"""Vectorised env: ``step(actions[N, A]) -> (obs[N, D], rew[N], done[N], info)`` as torch tensors.

Host-side mirror of the reference's gym surface for N envs at once.  All arithmetic happens in
the sm_100a kernels behind the C-ABI (``_cabi``); torch only supplies device memory and streams.
"""
import ctypes as C
from collections.abc import Mapping

import numpy as np
import torch

from . import _cabi
import os

from .config import (ENV_IDS, HRL_STATE_F, HRL_STATE_I, HRL_ANT_FLAGRUN, HRL_ANT_GATHER, HRL_POINT_GATHER, HrlConfig, SF_TARGET, SI_GOALS_LEFT,
                     SI_GOAL_GEN, apply_kwargs)

_NVTX = bool(int(os.environ.get("HRL_NVTX", "0")))   # NVTX ranges around reset / step (SURVEY.md section 5), off by default


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class LazyInfo(Mapping):
    """The step's ``info`` as a read-only mapping over the raw ``info[N, 4]`` array the kernel wrote
    (food_rew | inner reward, dead_rew | goals_left, TimeLimit.truncated, episode length).  Entries
    are materialised on access, so a stepping loop that never looks at ``info`` launches nothing
    besides the env kernel.  Keys follow the reference: ant_gather_env.py:119 ('food_rew',
    'dead_rew'), gym TimeLimit ('TimeLimit.truncated')."""

    def __init__(self, raw, kind, term=None, env=None):
        self.raw, self._kind, self._term, self._env = raw, kind, term, env
        keys = ["TimeLimit.truncated", "episode_length"]
        keys += ["food_rew", "dead_rew"] if kind in (HRL_ANT_GATHER, HRL_POINT_GATHER) else ["inner_rew"]
        if kind == HRL_ANT_FLAGRUN:
            # ant_flagrun_env.py:188-191,199: the reference sets i['target'] = self.goal only in a step that switched goals;
            # 'target_switched' is that condition per env, 'target' the current goal of every env (read on access)
            keys += ["goals_left", "target_switched"]
            if env is not None:
                keys.append("target")
        if term is not None:
            keys.append("terminal_obs")
        self._keys = keys

    def __getitem__(self, k):
        if k not in self._keys:
            raise KeyError(k)
        r = self.raw
        if k == "TimeLimit.truncated":   # info[:, 2] holds flag bits: 1 = truncated, 2 = Flagrun goal switched
            return (r[:, 2] % 2) > 0
        if k == "target_switched":
            return r[:, 2] >= 2
        if k == "episode_length":
            return r[:, 3]
        if k in ("food_rew", "inner_rew"):
            return r[:, 0]
        if k in ("dead_rew", "goals_left"):
            return r[:, 1]
        if k == "target":  # read from the state on access (one small kernel + copy, only when somebody looks)
            f, _ = self._env.get_state()
            t = f[:, SF_TARGET:SF_TARGET + 2]
            return t.cpu().numpy() if isinstance(r, np.ndarray) else t
        return self._term

    def __iter__(self):
        return iter(self._keys)

    def __len__(self):
        return len(self._keys)


class HostLazyInfo(LazyInfo):
    """`info` of the host (numpy) path: the raw columns live on the device and are copied to the host when an entry is
    read - a stepping loop that never looks at `info` moves 16 bytes per env less over PCIe every step."""

    def __init__(self, dev_raw, kind, env=None):
        super().__init__(dev_raw, kind, None, env)
        self._dev, self._seq, self._copy = dev_raw, -1, None

    def __getitem__(self, k):
        """Entries describe the MOST RECENT step (one device copy per step, made on first access)."""
        if k not in self._keys:
            raise KeyError(k)
        seq = self._env._host_seq
        if seq != self._seq:
            self._copy, self._seq = self._dev.cpu().numpy(), seq
        self.raw = self._copy
        return super().__getitem__(k)


class RolloutBuffer:
    """[T, N, ...] CUDA tensors the env kernel writes into directly (SURVEY.md 8f-4: the consumer side keeps the
    observations on the device; a trainer reads obs[t] / rew[t] / done[t] without any copy in between).
    obs has T + 1 slots: slot 0 takes the reset observation, step t writes obs[t + 1], rew[t], done[t].
    With ``info=True`` it also holds info[T, N, 4] (the four columns of ``step()``'s info per step), with
    ``terminal_obs=True`` terminal_obs[T, N, D]: row e of slot t is the observation before the auto-reset of an env that
    finished in step t (other rows are stale) - what a value bootstrap at a TimeLimit truncation needs."""

    def __init__(self, env, horizon, info=False, terminal_obs=False):
        d = env.device
        self.T = int(horizon)
        self.kind = env.kind
        self.obs = torch.zeros(self.T + 1, env.N, env.D, device=d)
        self.act = torch.zeros(self.T, env.N, env.A, device=d)
        self.rew = torch.zeros(self.T, env.N, device=d)
        self.done = torch.zeros(self.T, env.N, dtype=torch.bool, device=d)
        self.info = torch.zeros(self.T, env.N, 4, device=d) if info else None
        self.terminal_obs = torch.zeros(self.T, env.N, env.D, device=d) if terminal_obs else None

    def slot(self, t):
        return self.obs[t + 1], self.rew[t], self.done[t]

    @property
    def truncated(self):
        """bool [T, N]: the episode ended in step t by the TimeLimit, not by the env (``info["TimeLimit.truncated"]``)."""
        if self.info is None:
            raise ValueError("this RolloutBuffer holds no info (create it with info=True)")
        return (self.info[..., 2] % 2) > 0

    def infos(self, t):
        """``info`` of step t, the mapping ``step()`` returns (with "terminal_obs" when the buffer holds them)."""
        if self.info is None:
            raise ValueError("this RolloutBuffer holds no info (create it with info=True)")
        return LazyInfo(self.info[t], self.kind, None if self.terminal_obs is None else self.terminal_obs[t])

    def gae(self, values, gamma=0.99, lam=0.95, terminal_values=None, out=None, rew=None):
        """GAE(lambda) advantages and returns of the T steps in this buffer, in ONE kernel launch (include/hrl_b200.h
        `hrl_gae`).  ``values``: float32 [T + 1, N], V(obs[0..T]).  ``terminal_values``: float32 [T, N], typically
        ``critic(buf.terminal_obs)`` over the whole tensor (stale rows included: a row is read only where it is selected);
        it needs a buffer made with ``info=True``.  With it, an episode ended by the TimeLimit bootstraps from
        ``terminal_values[t]`` and one ended by the env from 0; without it, every done is a termination.  ``obs[t + 1]`` of
        an env that finished in step t is the reset observation, so its value never bootstraps step t.
        ``out=(adv, ret)``: float32 [T, N] tensors written in place (no allocation, so the call can be captured in a CUDA
        graph).  ``rew``: float32 [T, N] rewards used instead of ``self.rew`` (e.g. ``RunningNormalizer.scale_rewards``).
        No host synchronisation.  Returns ``(adv, ret)``."""
        T, N = self.rew.shape
        dev = self.rew.device

        def check(name, t, shape):
            if not isinstance(t, torch.Tensor) or tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous() \
                    or t.device != dev:
                raise ValueError("%s must be a contiguous float32 tensor [%s] on %s" % (name, ", ".join(map(str, shape)), dev))

        check("values", values, (T + 1, N))
        if rew is not None:
            check("rew", rew, (T, N))
        else:
            rew = self.rew
        if terminal_values is not None:
            if self.info is None:
                raise ValueError("terminal_values need the truncation flags: create the RolloutBuffer with info=True")
            check("terminal_values", terminal_values, (T, N))
        if not (0.0 <= gamma <= 1.0 and 0.0 <= lam <= 1.0):
            raise ValueError("gamma and lam must lie in [0, 1], got %r, %r" % (gamma, lam))
        if out is None:
            adv, ret = torch.empty_like(self.rew), torch.empty_like(self.rew)
        else:
            if len(out) != 2:
                raise ValueError("out must be (adv, ret)")
            adv, ret = out
            check("out[0] (adv)", adv, (T, N))
            check("out[1] (ret)", ret, (T, N))
        info = self.info if terminal_values is not None else None
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib().hrl_gae(T, N, float(gamma), float(lam), _ptr(rew), _ptr(self.done), _ptr(info), _ptr(values),
                                            _ptr(terminal_values), _ptr(adv), _ptr(ret),
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        return adv, ret


class VecEnv:
    """N independent envs of one reference id on one GPU.

    Parameters mirror ``gym.make(id, **kwargs)`` of the reference plus ``num_envs``, ``device``,
    ``seed`` and ``env_index_offset`` (global index of env 0, for multi-GPU shards).
    """

    def __init__(self, env_id, num_envs, device=0, seed=None, env_index_offset=0, auto_reset=True,
                 max_episode_steps=2000, config_overrides=None, env_seed=None, **kwargs):
        """``seed`` keys the per-env RNG streams (joint noise, item placement, maze goal choice: what ``env.seed(s)``
        and the Maze ctor's ``seed`` kwarg feed in the reference, ant_maze_bullet_env.py:48,99-102).  For
        AntFlagrunBulletEnv an explicit ``seed`` is ALSO the ctor kwarg of the reference (ant_flagrun_env.py:16,39): it
        seeds the goal stream shared by all envs (default 123).  ``env_seed`` overrides the per-env key alone."""
        if env_id not in ENV_IDS:
            raise KeyError("unknown env id %r; known: %s" % (env_id, sorted(ENV_IDS)))
        if not torch.cuda.is_available():
            raise _cabi.HrlError("no CUDA device: hrl_pybullet_envs_b200 has no CPU fallback")
        self.env_id = env_id
        self.kind = ENV_IDS[env_id]
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        cfg = _cabi.default_config(self.kind, num_envs)
        apply_kwargs(cfg, self.kind, kwargs)
        cfg.seed = int(seed or 0)
        if self.kind == HRL_ANT_FLAGRUN and seed is not None:
            cfg.flag_seed = int(seed)
        if env_seed is not None:
            cfg.seed = int(env_seed)
        cfg.env_index_offset = int(env_index_offset)
        cfg.auto_reset = int(bool(auto_reset))
        cfg.max_episode_steps = int(max_episode_steps)
        known = {f[0] for f in HrlConfig._fields_}
        for k, v in (config_overrides or {}).items():
            if k not in known:
                raise KeyError("config_overrides: hrl_config has no field %r" % k)
            setattr(cfg, k, v)
        self.cfg = cfg
        self.L = _cabi.lib()
        self.h = C.c_void_p()
        _cabi.check(self.L.hrl_create(C.byref(cfg), self.device.index, C.byref(self.h)))
        self.num_envs = self.N = num_envs
        self.obs_dim = self.D = self.L.hrl_obs_dim(C.byref(cfg))
        self.act_dim = self.A = self.L.hrl_act_dim(C.byref(cfg))
        d = self.device
        self._obs = torch.zeros(self.N, self.D, device=d)
        self._rew = torch.zeros(self.N, device=d)
        self._done = torch.zeros(self.N, dtype=torch.uint8, device=d)
        self._info = torch.zeros(self.N, 4, device=d)
        self._term = None
        self._host = None
        self._host_seq = 0

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, "h", None):
            self.L.hrl_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ gym-like API
    def seed(self, seed=None):
        """Re-seeding happens at construction (counter RNG keyed by (seed, env index))."""
        return [self.cfg.seed]

    def _mask(self, mask):
        if mask is None:
            return None
        m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        if m.numel() != self.N:
            raise ValueError("mask must have %d entries, got %d" % (self.N, m.numel()))
        return m

    def reset(self, mask=None):
        """Reset all envs (or the masked ones) and return obs[N, D]; rows of envs outside the mask hold the observation
        of their CURRENT state (refreshed, so the returned tensor is always a consistent batch)."""
        m = self._mask(mask)
        if _NVTX:
            torch.cuda.nvtx.range_push("hrl.reset")
        if m is not None:
            _cabi.check(self.L.hrl_observe(self.h, _ptr(self._obs), self._stream()))
        _cabi.check(self.L.hrl_reset(self.h, _ptr(m), _ptr(self._obs), self._stream()))
        if _NVTX:
            torch.cuda.nvtx.range_pop()
        return self._obs

    def step(self, actions, want_terminal_obs=False, out=None):
        """actions: float32 CUDA tensor [N, A] (device path) or numpy array (host path).
        ``out=(obs[N, D] f32, rew[N] f32, done[N] u8/bool)``: the kernel writes this step's results straight into
        those CUDA tensors (e.g. slot t of a ``RolloutBuffer``) instead of the env's own buffers - no copy.  A fourth
        tensor ``info[N, 4] f32`` takes the raw info columns the same way."""
        if isinstance(actions, np.ndarray):
            return self.step_host(actions)
        a = actions
        if a.dtype != torch.float32 or not a.is_contiguous() or a.device != self.device:
            a = a.to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(a.shape) != (self.N, self.A):
            raise ValueError("actions must have shape (%d, %d), got %s" % (self.N, self.A, tuple(a.shape)))
        term = None
        if want_terminal_obs:
            if self._term is None:
                self._term = torch.zeros(self.N, self.D, device=self.device)
            term = self._term
        obs, rew, done, info = self._obs, self._rew, self._done, self._info
        if out is not None:
            if len(out) not in (3, 4):
                raise ValueError("out must be (obs, rew, done) or (obs, rew, done, info)")
            obs, rew, done = out[:3]
            info = out[3] if len(out) == 4 else info
            for t, shape, dts in ((obs, (self.N, self.D), (torch.float32,)), (rew, (self.N,), (torch.float32,)),
                                  (done, (self.N,), (torch.uint8, torch.bool)), (info, (self.N, 4), (torch.float32,))):
                if tuple(t.shape) != shape or t.dtype not in dts or not t.is_contiguous() or t.device != self.device:
                    raise ValueError("out tensors must be contiguous CUDA tensors obs[%d,%d] f32, rew[%d] f32, done[%d] u8/bool"
                                     ", info[%d,4] f32" % (self.N, self.D, self.N, self.N, self.N))
        if _NVTX:
            torch.cuda.nvtx.range_push("hrl.step")
        _cabi.check(self.L.hrl_step(self.h, _ptr(a), _ptr(obs), _ptr(rew), _ptr(done),
                                    _ptr(info), _ptr(term), self._stream()))
        if _NVTX:
            torch.cuda.nvtx.range_pop()
        return obs, rew, done.view(torch.bool), self._info_dict(info, term)

    def capture_rollout(self, actions, buf=None):
        """CUDA-graph launch (SURVEY.md section 7 step 5): capture ``T = actions.shape[0]`` consecutive steps, step t
        reading ``actions[t]`` (a [T, N, A] CUDA tensor the caller refills between replays) and writing slot t of
        ``buf`` (a ``RolloutBuffer``; created when None), its ``info[t]`` too when the buffer holds info (terminal
        observations are not recorded here).  Returns ``(graph, buf)``; ``graph.replay()`` runs the T
        steps with ONE launch from the host.  ``step()`` itself is capture-safe (no allocation, no synchronisation),
        so a caller can equally capture its own policy + ``env.step`` loop with ``torch.cuda.graph``."""
        a = actions
        if a.dtype != torch.float32 or not a.is_contiguous() or a.device != self.device or tuple(a.shape[1:]) != (self.N, self.A):
            raise ValueError("actions must be a contiguous float32 CUDA tensor [T, %d, %d]" % (self.N, self.A))
        T = a.shape[0]
        buf = buf or RolloutBuffer(self, T)
        if buf.T < T:
            raise ValueError("rollout buffer holds %d steps, need %d" % (buf.T, T))
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for t in range(T):
                self.step(a[t], out=buf.slot(t) if buf.info is None else buf.slot(t) + (buf.info[t],))
        return g, buf

    @staticmethod
    def pack_mlp(layers):
        """Pack ((W1, b1), (W2, b2), (W3, b3)) in torch.nn.Linear layout (W[out, in]) into the input-major float32 vector
        `hrl_rollout_mlp` reads: W1^T b1 W2^T b2 W3^T b3.  Batched layers (W[P, out, in], b[P, out]: one policy per member
        of a population) pack into [P, nw], one such vector per row (`hrl_evaluate_mlp`)."""
        parts = []
        for W, b in layers:
            W, b = W.detach().to(torch.float32), b.detach().to(torch.float32)
            if W.dim() == 3:
                parts += [W.transpose(1, 2).reshape(W.shape[0], -1), b.reshape(b.shape[0], -1)]
            else:
                parts += [W.t().contiguous().reshape(-1), b.reshape(-1)]
        return torch.cat(parts, dim=-1).contiguous()

    def _mlp_width(self, layers, batched=False):
        """Hidden width H of ((W1[H, D], b1[H]), (W2[H, H], b2[H]), (W3[A, H], b3[A])), with a leading member dimension P
        on every tensor when `batched`; returns (H, P) (P = None unbatched).  ValueError on any other shape."""
        (W1, b1), (W2, b2), (W3, b3) = layers
        lead = tuple(W1.shape[:1]) if batched else ()
        H = W1.shape[len(lead)] if W1.dim() == len(lead) + 2 else -1
        want = ((H, self.D), (H,), (H, H), (H,), (self.A, H), (self.A,))
        if H not in (32, 64) or (batched and lead[0] < 1) or any(tuple(t.shape) != lead + s for t, s in zip((W1, b1, W2, b2, W3, b3), want)):
            p = "P," if batched else ""
            raise ValueError("layers must be ((W1[{p}H,{D}], b1[{p}H]), (W2[{p}H,H], b2[{p}H]), (W3[{p}{A},H], b3[{p}{A}])) with H = 32 or 64, "
                             "got W1 of shape {s}".format(p=p, D=self.D, A=self.A, s=tuple(W1.shape)))
        return H, (lead[0] if batched else None)

    def _noise_scale(self, sigma):
        """(scalar sigma, per-component scale tensor or None) for the C-ABI, from a float or a length-A tensor."""
        if not isinstance(sigma, torch.Tensor):
            return sigma, None
        sig_v = sigma.detach().to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(sig_v.shape) != (self.A,):
            raise ValueError("sigma must be a float or a tensor of %d entries, got shape %s" % (self.A, tuple(sig_v.shape)))
        if not bool((torch.isfinite(sig_v) & (sig_v >= 0)).all()):
            raise ValueError("sigma entries must be finite and >= 0")
        return 0.0, sig_v

    def _check_obs_norm(self, obs_norm):
        if obs_norm is not None and (getattr(obs_norm, "D", None) != self.D or getattr(obs_norm, "device", None) != self.device):
            raise ValueError("obs_norm must be a RunningNormalizer of obs_dim %d on %s" % (self.D, self.device))

    def rollout_mlp(self, layers, horizon, buf=None, sigma=0.0, noise_seed=0, want_info=False, want_terminal_obs=False,
                    obs_norm=None):
        """Fused rollout (include/hrl_b200.h `hrl_rollout_mlp_ex`): `horizon` steps in ONE kernel launch, actions from the
        3-layer tanh MLP `layers` = ((W1[H, D], b1), (W2[H, H], b2), (W3[A, H], b3)) evaluated inside the kernel (H = 32 or
        64), plus N(0, sigma^2) exploration noise.  `sigma` is a float or a length-A tensor (one scale per action
        component, e.g. exp(log_std) of a Gaussian policy).  Fills and returns a RolloutBuffer: obs[0..T], act, rew,
        done, and with `want_info` / `want_terminal_obs` also info / terminal_obs (allocated when `buf` is None).
        `obs_norm`: a `RunningNormalizer` of this env's obs_dim; the policy then reads `obs_norm.normalize(obs)`, with the
        statistics frozen for the launch (`hrl_rollout_mlp_norm`).  The buffer still receives the raw observations."""
        (W1, b1), (W2, b2), (W3, b3) = layers
        H = W1.shape[0]
        if H not in (32, 64) or tuple(W1.shape) != (H, self.D) or tuple(W2.shape) != (H, H) or tuple(W3.shape) != (self.A, H):
            raise ValueError("layers must be ((W1[H,%d], b1[H]), (W2[H,H], b2[H]), (W3[%d,H], b3[%d])) with H = 32 or 64" % (self.D, self.A, self.A))
        w = self.pack_mlp(layers).to(self.device)
        sigma, sig_v = self._noise_scale(sigma)
        self._check_obs_norm(obs_norm)
        buf = buf or RolloutBuffer(self, horizon, info=want_info, terminal_obs=want_terminal_obs)
        if buf.T < horizon:
            raise ValueError("rollout buffer holds %d steps, need %d" % (buf.T, horizon))
        if (want_info and buf.info is None) or (want_terminal_obs and buf.terminal_obs is None):
            raise ValueError("rollout buffer has no room for info / terminal_obs: create it with info=True / terminal_obs=True")
        info = buf.info if want_info else None
        term = buf.terminal_obs if want_terminal_obs else None
        if _NVTX:
            torch.cuda.nvtx.range_push("hrl.rollout_mlp")
        if obs_norm is None:
            _cabi.check(self.L.hrl_rollout_mlp_ex(self.h, int(horizon), _ptr(w), int(H), float(sigma), _ptr(sig_v), int(noise_seed),
                                                  _ptr(buf.obs), _ptr(buf.act), _ptr(buf.rew), _ptr(buf.done), _ptr(info), _ptr(term),
                                                  self._stream()))
        else:
            _cabi.check(self.L.hrl_rollout_mlp_norm(self.h, int(horizon), _ptr(w), int(H), float(sigma), _ptr(sig_v), int(noise_seed),
                                                    _ptr(obs_norm.mean), _ptr(obs_norm.rstd), obs_norm.clip_obs, _ptr(buf.obs),
                                                    _ptr(buf.act), _ptr(buf.rew), _ptr(buf.done), _ptr(info), _ptr(term),
                                                    self._stream()))
        if _NVTX:
            torch.cuda.nvtx.range_pop()
        self._keep = (w, sig_v)   # the launch is asynchronous: keep the packed weights and noise scales alive
        return buf

    def evaluate_mlp(self, layers, horizon, sigma=0.0, noise_seed=0, obs_norm=None, out=None):
        """Score MLP policies by their episodes in ONE kernel launch (include/hrl_b200.h `hrl_evaluate_mlp`), writing no
        per-step buffers.  `layers`: the layers of `rollout_mlp` (one policy for all envs, P = 1) or batched, every tensor
        with a leading member dimension P (W1[P, H, D], b1[P, H], ...).  Env e runs member e // M, M = N / P; for P > 1, N
        must be a multiple of P and M a multiple of 16 (Ant) or 8 (PointGather).  `sigma`, `noise_seed` and `obs_norm` act as
        in `rollout_mlp`, the same for every member.
        Runs `horizon` steps from the current state, with auto-reset.  Returns `(ret, length, finished)`, [P, M] views of [N]
        tensors (row m: member m's envs): the float32 sum of each env's rewards from the first step up to and including its
        first done, the number of those steps, and whether a done came within `horizon` steps (if not, the sum covers all of
        them).  Call `reset()` first to score whole episodes: an env started mid-episode is scored on the rest of it.
        `out=(ret f32, length i32, finished bool)`, each [N] or [P, M]: written in place (no allocation, so the call can be
        captured in a CUDA graph).  No host synchronisation, except to check a sigma tensor's entries."""
        H, P = self._mlp_width(layers, batched=layers[0][0].dim() == 3)
        P = P or 1
        T = int(horizon)
        if T < 1:
            raise ValueError("horizon must be >= 1, got %d" % T)
        epc = 8 if self.kind == HRL_POINT_GATHER else 16
        if self.N % P:
            raise ValueError("num_envs %d is not a multiple of the member count %d" % (self.N, P))
        M = self.N // P
        if P > 1 and M % epc:
            raise ValueError("envs per member (num_envs / P = %d) must be a multiple of %d for %s" % (M, epc, self.env_id))
        sigma, sig_v = self._noise_scale(sigma)
        if sig_v is None and not float(sigma) >= 0.0:
            raise ValueError("sigma must be >= 0, got %r" % (sigma,))
        self._check_obs_norm(obs_norm)
        if out is None:
            ret = torch.empty(self.N, device=self.device)
            length = torch.empty(self.N, dtype=torch.int32, device=self.device)
            finished = torch.empty(self.N, dtype=torch.bool, device=self.device)
        else:
            if len(out) != 3:
                raise ValueError("out must be (ret, length, finished)")
            ret, length, finished = out
            for t, dt in ((ret, torch.float32), (length, torch.int32), (finished, torch.bool)):
                if not isinstance(t, torch.Tensor) or tuple(t.shape) not in ((self.N,), (P, M)) or t.dtype != dt or not t.is_contiguous() \
                        or t.device != self.device:
                    raise ValueError("out must be contiguous tensors on %s of shape [%d] or [%d, %d]: ret float32, length int32, finished "
                                     "bool" % (self.device, self.N, P, M))
        w = self.pack_mlp(layers).to(self.device)
        if _NVTX:
            torch.cuda.nvtx.range_push("hrl.evaluate_mlp")
        norm = (None, None, 0.0) if obs_norm is None else (obs_norm.mean, obs_norm.rstd, obs_norm.clip_obs)
        _cabi.check(self.L.hrl_evaluate_mlp(self.h, T, P, _ptr(w), int(H), float(sigma), _ptr(sig_v), int(noise_seed), _ptr(norm[0]),
                                            _ptr(norm[1]), float(norm[2]), _ptr(ret), _ptr(length), _ptr(finished), self._stream()))
        if _NVTX:
            torch.cuda.nvtx.range_pop()
        self._keep = (w, sig_v)   # the launch is asynchronous: keep the packed weights and noise scales alive
        return ret.view(P, M), length.view(P, M), finished.view(P, M)

    def rollout_buffer(self, horizon):
        """Device-resident storage for ``horizon`` steps; ``step(a, out=buf.slot(t))`` fills slot t in place."""
        return RolloutBuffer(self, horizon)

    def _info_dict(self, info, term=None):
        return LazyInfo(info, self.kind, term, env=self)

    HOST_MODES = {"auto": 0, "copy": 1, "zerocopy": 2}

    def set_host_mode(self, mode):
        """'zerocopy' (kernel reads/writes pinned host memory over PCIe while it computes), 'copy'
        (H2D, kernel, one packed D2H) or 'auto' (zero-copy when the buffers are pinned)."""
        _cabi.check(self.L.hrl_set_host_mode(self.h, self.HOST_MODES[mode]))

    def _host_buffers(self):
        """Two packed pinned output sets [obs | rew | info | done] (hrl_host_layout) + one action buffer;
        the sets alternate so that the arrays returned by the previous step stay valid for one more step."""
        o_rew, o_info, o_done, total = (C.c_size_t() for _ in range(4))
        _cabi.check(self.L.hrl_host_layout(C.byref(self.cfg), C.byref(o_rew), C.byref(o_info), C.byref(o_done), C.byref(total)))
        sets = []
        for _ in range(2):
            raw = torch.zeros(total.value, dtype=torch.uint8, pin_memory=True)
            base = raw.data_ptr()
            v = raw.numpy()
            sets.append(dict(
                raw=raw,
                obs=v[:self.N * self.D * 4].view(np.float32).reshape(self.N, self.D),
                rew=v[o_rew.value:o_rew.value + self.N * 4].view(np.float32),
                info=v[o_info.value:o_info.value + self.N * 16].view(np.float32).reshape(self.N, 4),
                done=v[o_done.value:o_done.value + self.N].view(np.bool_),
                p_obs=C.c_void_p(base), p_rew=C.c_void_p(base + o_rew.value), p_info=C.c_void_p(base + o_info.value),
                p_done=C.c_void_p(base + o_done.value)))
        for S in sets:
            # info stays on the device (self._info) and is fetched when somebody looks: 16 of the 205 bytes per env
            S["info_map"] = HostLazyInfo(self._info, self.kind, env=self)
            S["ret"] = (S["obs"], S["rew"], S["done"], S["info_map"])
        act = torch.zeros(self.N, self.A, pin_memory=True)
        return dict(sets=sets, act=act, act_np=act.numpy(), p_act=C.c_void_p(act.data_ptr()), flip=0, p_info=_ptr(self._info),
                    n_act=self.N * self.A, step=self.L.hrl_step_host)

    def step_host(self, actions):
        """numpy in / numpy out through ``hrl_step_host``: the call a gym-style user makes.  The
        returned arrays are views of pinned memory, valid until the step after the next one."""
        H = self._host
        if H is None:
            H = self._host = self._host_buffers()
        if type(actions) is np.ndarray and actions.dtype == np.float32 and actions.size == H["n_act"] and actions.flags.c_contiguous:
            p_act = actions.ctypes.data   # used in place: read over PCIe when pinned, copied H2D by the library when not
        else:
            if np.size(actions) != H["n_act"]:
                raise ValueError("actions must have shape (%d, %d)" % (self.N, self.A))
            np.copyto(H["act_np"], np.asarray(actions).reshape(self.N, self.A), casting="same_kind")
            p_act = H["p_act"]
        S = H["sets"][H["flip"]]
        H["flip"] ^= 1
        self._host_seq += 1
        rc = H["step"](self.h, p_act, S["p_obs"], S["p_rew"], S["p_done"], H["p_info"], torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            _cabi.check(rc)
        return S["ret"]

    def observe(self):
        _cabi.check(self.L.hrl_observe(self.h, _ptr(self._obs), self._stream()))
        return self._obs

    def substeps(self, actions, n_sub):
        a = actions.to(device=self.device, dtype=torch.float32).contiguous()
        _cabi.check(self.L.hrl_substeps(self.h, _ptr(a), int(n_sub), self._stream()))

    # ------------------------------------------------------------------ Flagrun goal API (ant_flagrun_env.py:91-120)
    def _flagrun_only(self):
        if self.kind != HRL_ANT_FLAGRUN:
            raise TypeError("only AntFlagrunBulletEnv has walk targets to set")

    @property
    def goal(self):
        """Current walk target of every env, [N, 2] (ant_flagrun_env.py:57 `goal`)."""
        self._flagrun_only()
        return self.get_state()[0][:, SF_TARGET:SF_TARGET + 2]

    def set_target(self, xy, env_ids=None):
        """set_target(x, y) (ant_flagrun_env.py:98-110) for all envs or `env_ids`: moves the walk target only - like the
        reference it neither touches the potential nor `_rewarded` (next_target does)."""
        self._flagrun_only()
        f, i = self.get_state()
        xy = torch.as_tensor(xy, dtype=torch.float32, device=self.device)
        if env_ids is None:
            f[:, SF_TARGET:SF_TARGET + 2] = xy
        else:
            f[torch.as_tensor(env_ids, device=self.device), SF_TARGET:SF_TARGET + 2] = xy
        self.set_state(f, i)

    def create_targets(self, n=None):
        """create_targets(n) (ant_flagrun_env.py:91-96): refill every env's goal list with n (default max_targets) goals
        of the shared stream; the step pops them on reach / timeout, `next_target()` pops one now."""
        self._flagrun_only()
        n = self.cfg.flag_max_targets if n is None else int(n)
        if not 0 <= n <= 127:
            raise ValueError("n must be in [0, 127]")
        f, i = self.get_state()
        i[:, SI_GOALS_LEFT] = n
        i[:, SI_GOAL_GEN] += 1     # every call draws fresh goals from the shared stream, like the reference
        self.set_state(f, i)

    def next_target(self, mask=None):
        """next_target() (ant_flagrun_env.py:112-120) for all envs or the masked ones; returns the fresh observation."""
        self._flagrun_only()
        m = self._mask(mask)
        _cabi.check(self.L.hrl_flagrun_next_target(self.h, _ptr(m), self._stream()))
        return self.observe()

    # ------------------------------------------------------------------ checkpoint / resume
    def get_state(self):
        f = torch.zeros(self.N, HRL_STATE_F, device=self.device)
        i = torch.zeros(self.N, HRL_STATE_I, dtype=torch.int32, device=self.device)
        _cabi.check(self.L.hrl_get_state(self.h, _ptr(f), _ptr(i), self._stream()))
        return f, i

    def set_state(self, f, i):
        f = torch.as_tensor(f).to(device=self.device, dtype=torch.float32).contiguous()
        i = torch.as_tensor(i).to(device=self.device, dtype=torch.int32).contiguous()
        if f.shape != (self.N, HRL_STATE_F) or i.shape != (self.N, HRL_STATE_I):
            raise ValueError("state tensors must be [N,%d] f32 and [N,%d] i32" % (HRL_STATE_F, HRL_STATE_I))
        _cabi.check(self.L.hrl_set_state(self.h, _ptr(f), _ptr(i), self._stream()))

    def episode_stats(self, aggregate=False):
        """Episode statistics kept by the kernels (SURVEY.md section 5): finished episodes, their mean
        return and mean length, env-steps taken.  ``aggregate=True`` sums the counters over all ranks of the
        default process group (NCCL over NVLink on GPUs) - the only collective this package ever issues, and
        never on the step path."""
        from .sharding import sum_episode_stats
        f, i = self.get_state()
        finished = (i[:, 1] - 1).clamp(min=0).sum().item()          # resets so far minus the running episode
        ret_sum = f[:, 71].double().sum().item()                    # HRL_SF_RETURN_SUM
        steps = i[:, 2].sum().item()
        len_sum = (i[:, 2] - i[:, 0]).sum().item()                  # steps that belong to finished episodes
        if aggregate:
            finished, steps, ret_sum, len_sum = sum_episode_stats(finished, steps, (ret_sum, len_sum), device=self.device)
        n = max(finished, 1)
        return {"episodes": int(finished), "env_steps": int(steps), "mean_return": ret_sum / n, "mean_length": len_sum / n}

    def stats(self, reset=True):
        """In-kernel counters feeding the FLOP model: mean contacts / limit rows per env-substep."""
        out = (C.c_ulonglong * 4)()
        _cabi.check(self.L.hrl_get_stats(self.h, out, int(reset)))
        n = max(int(out[2]), 1)
        return {"contacts_per_substep": out[0] / n, "limit_rows_per_substep": out[1] / n, "env_substeps": int(out[2])}


# ---- stand-alone sensors (parity entry points) ------------------------------------------
def gather_sensor(xy, yaw, items, n_bins=10, sensor_range=20.0, sensor_span=np.pi):
    """ant_gather_env.py:128-177 for M poses: returns (food[M,n], poison[M,n], bins[M,16])."""
    L = _cabi.lib()
    dev = xy.device
    M = xy.shape[0]
    xy = xy.to(torch.float32).contiguous(); yaw = yaw.to(torch.float32).contiguous()
    items = items.to(torch.float32).contiguous()
    food = torch.zeros(M, n_bins, device=dev); poison = torch.zeros(M, n_bins, device=dev)
    bins = torch.full((M, 16), -1, dtype=torch.int32, device=dev)
    _cabi.check(L.hrl_gather_sensor(M, n_bins, float(sensor_range), float(sensor_span), _ptr(xy), _ptr(yaw), _ptr(items),
                                    _ptr(food), _ptr(poison), _ptr(bins),
                                    C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return food, poison, bins


def sense_walls(xy, yaw, bounds, n_bins=10, span=2 * np.pi, rng=5.0):
    """sizeable_enclosed_scene.py:63-97 for M poses: returns out[M, n_bins]."""
    L = _cabi.lib()
    dev = xy.device
    M = xy.shape[0]
    xy = xy.to(torch.float32).contiguous(); yaw = yaw.to(torch.float32).contiguous()
    bounds = bounds.to(device=dev, dtype=torch.float32).contiguous()
    out = torch.zeros(M, n_bins, device=dev)
    _cabi.check(L.hrl_sense_walls(M, n_bins, float(span), float(rng), bounds.shape[0], _ptr(bounds), _ptr(xy), _ptr(yaw),
                                  _ptr(out), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return out
