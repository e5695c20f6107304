"""Normalization workload for the bounds-checked build (-DHRL_BOUNDS=1 -> libhrl_b200_chk.so; run with HRL_B200_LIB pointing
at it): the normalized fused rollout of every env family at N = 203 (ragged last CTA) with both hidden widths, resets and a
binding clip; hrl_obs_moments at ragged M and D; hrl_reward_scale at ragged T and N.  A device-side assert aborts the
process; the statistics are also checked against the float64 references.  Used by tests/test_gpu_normalize.py."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
from hrl_pybullet_envs_b200 import RunningNormalizer, VecEnv, _cabi
from test_normalize import obs_moments_ref, reward_scale_ref

assert b"HRL_BOUNDS" in _cabi.lib().hrl_version(), "not the bounds-checked build: set HRL_B200_LIB=.../libhrl_b200_chk.so"
N, T = 203, 12
CASES = [("AntGatherBulletEnv-v0", {}), ("AntMazeBulletEnv-v0", dict(sense_target=True)), ("AntFlagrunBulletEnv-v0", dict(timeout=4)),
         ("AntMjBulletEnv-v0", {}), ("PointGatherBulletEnv-v0", {}), ("PointGatherBulletEnv-v0", dict(use_sensor=False, n_bins=16))]
g = torch.Generator().manual_seed(5)
for env_id, kw in CASES:
    for H in (32, 64):
        env = VecEnv(env_id, N, seed=1, max_episode_steps=5, **kw)
        norm = RunningNormalizer(env, clip_obs=3.0)
        norm.update_obs(env.reset())
        norm.rstd[1] *= 1e3                   # the clip binds
        layers = tuple((((torch.rand(o, i, generator=g) * 2 - 1) * 0.5).cuda(), (torch.rand(o, generator=g) * 0.2 - 0.1).cuda())
                       for o, i in ((H, env.D), (H, H), (env.A, H)))
        clipped = False
        for i in range(2):
            buf = env.rollout_mlp(layers, T, sigma=0.3, noise_seed=i, want_info=True, want_terminal_obs=True, obs_norm=norm)
            clipped = clipped or bool((norm.normalize(buf.obs).abs() == 3.0).any())
            norm.update_obs(buf.obs[1:])
            norm.rstd[1] *= 1e3
        torch.cuda.synchronize()
        assert bool(buf.done.any()) and clipped
        print("ok rollout", env_id, kw, "H", H, flush=True)
        env.close()
for M, D in ((1, 1), (3, 64), (1031, 7), (20000, 45)):
    n = RunningNormalizer((1, D))
    x = np.random.default_rng(M).normal(3, 2, (M, D)).astype(np.float32)
    n.update_obs(torch.from_numpy(x).cuda())
    _, m, v, mf, rf = obs_moments_ref((1e-4, np.zeros(D), np.ones(D)), x, 1e-8)
    assert np.allclose(n.obs_moments.cpu().numpy()[1:], np.concatenate([m, v]), rtol=1e-9, atol=1e-12)
    print("ok obs_moments", M, D, flush=True)
for T_, N_ in ((1, 1), (33, 17), (70, 5001)):
    n = RunningNormalizer((N_, 1))
    rng = np.random.default_rng(T_ + N_)
    rew, done = rng.normal(0, 1, (T_, N_)).astype(np.float32), rng.random((T_, N_)) < 0.1
    out = n.scale_rewards(torch.from_numpy(rew).cuda(), torch.from_numpy(done).cuda())
    ref, R, _, _ = reward_scale_ref(rew, done, np.zeros(N_), (1e-4, 0.0, 1.0), 0.99, 10.0, 1e-8)
    assert np.allclose(out.cpu().numpy(), ref, rtol=1e-6, atol=0) and np.array_equal(n.returns.cpu().numpy(), R)
    print("ok reward_scale", T_, N_, flush=True)
print("bounds normalize run complete")
