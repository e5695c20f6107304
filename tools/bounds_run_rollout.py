"""Fused-rollout workload for the bounds-checked build (-DHRL_BOUNDS=1 -> libhrl_b200_chk.so; run with HRL_B200_LIB pointing
at it): every env family, both hidden widths, ragged batch, short episodes (resets and terminal observations inside the
launch), per-step info, per-action noise scales.  A device-side assert aborts the process.  Used by
tests/test_gpu_rollout_training.py."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from hrl_pybullet_envs_b200 import VecEnv, _cabi

assert b"HRL_BOUNDS" in _cabi.lib().hrl_version(), "not the bounds-checked build: set HRL_B200_LIB=.../libhrl_b200_chk.so"
N, T = 203, 16   # ragged last CTA of both kernels
CASES = [("AntGatherBulletEnv-v0", {}), ("AntGatherBulletEnv-v0", dict(use_sensor=False)), ("AntMazeBulletEnv-v0", dict(sense_target=True)),
         ("AntFlagrunBulletEnv-v0", dict(timeout=4)), ("AntMjBulletEnv-v0", {}), ("AntMazeMjEnv-v0", {}),
         ("AntMazeMjEnv-v0", dict(n_bins=11)), ("AntGatherBulletEnv-v0", dict(robot_coll_dist=0)),
         ("PointGatherBulletEnv-v0", {}), ("PointGatherBulletEnv-v0", dict(use_sensor=False, n_bins=16))]
g = torch.Generator().manual_seed(5)
for env_id, kw in CASES:
    for H in (32, 64):
        env = VecEnv(env_id, N, seed=1, max_episode_steps=7, **kw)
        env.reset()
        layers = tuple((((torch.rand(o, i, generator=g) * 2 - 1) * 0.5).cuda(), (torch.rand(o, generator=g) * 0.2 - 0.1).cuda())
                       for o, i in ((H, env.D), (H, H), (env.A, H)))
        sigma = torch.linspace(0.1, 0.8, env.A, device="cuda")
        for i in range(2):
            buf = env.rollout_mlp(layers, T, sigma=sigma if i else 0.3, noise_seed=i, want_info=True, want_terminal_obs=True)
        torch.cuda.synchronize()
        assert bool(buf.done.any())
        print("ok", env_id, kw, "H", H)
        env.close()
print("bounds rollout run complete")
