"""Population-evaluation workload for the bounds-checked build (-DHRL_BOUNDS=1 -> libhrl_b200_chk.so; run with HRL_B200_LIB
pointing at it): every env family, both hidden widths, one policy on a ragged batch (P = 1, N = 203) and four members
(P = 4, one or two CTAs each), short episodes (resets inside the launch), scalar and per-action noise, a normalized input.
A device-side assert aborts the process.  Used by tests/test_gpu_evaluate.py."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from hrl_pybullet_envs_b200 import RunningNormalizer, VecEnv, _cabi

assert b"HRL_BOUNDS" in _cabi.lib().hrl_version(), "not the bounds-checked build: set HRL_B200_LIB=.../libhrl_b200_chk.so"
T = 16
CASES = [("AntGatherBulletEnv-v0", {}), ("AntGatherBulletEnv-v0", dict(use_sensor=False)), ("AntMazeBulletEnv-v0", dict(sense_target=True)),
         ("AntFlagrunBulletEnv-v0", dict(timeout=4)), ("AntMjBulletEnv-v0", {}), ("AntMazeMjEnv-v0", {}),
         ("AntMazeMjEnv-v0", dict(n_bins=11)), ("AntGatherBulletEnv-v0", dict(robot_coll_dist=0)),
         ("PointGatherBulletEnv-v0", {}), ("PointGatherBulletEnv-v0", dict(use_sensor=False, n_bins=16))]
g = torch.Generator().manual_seed(5)
for env_id, kw in CASES:
    for H in (32, 64):
        for P in (1, 4):
            N = 203 if P == 1 else P * (8 if env_id.startswith("Point") else 16)
            env = VecEnv(env_id, N, seed=1, max_episode_steps=7, **kw)
            env.reset()
            layers = tuple((((torch.rand(P, o, i, generator=g) * 2 - 1) * 0.5).cuda(), (torch.rand(P, o, generator=g) * 0.2 - 0.1).cuda())
                           for o, i in ((H, env.D), (H, H), (env.A, H)))
            if P == 1:
                layers = tuple((W[0], b[0]) for W, b in layers)
            norm = RunningNormalizer(env)
            norm.update_obs(env.observe())
            sigma = torch.linspace(0.1, 0.8, env.A, device="cuda")
            for i in range(2):
                ret, length, fin = env.evaluate_mlp(layers, T, sigma=sigma if i else 0.3, noise_seed=i, obs_norm=norm if i else None)
            torch.cuda.synchronize()
            assert bool(fin.all()) and int(length.max()) <= 7
            print("ok", env_id, kw, "H", H, "P", P)
            env.close()
print("bounds evaluate run complete")
