"""Workload for the bounds-checked build (-DHRL_BOUNDS=1 -> libhrl_b200_chk.so; run with HRL_B200_LIB pointing at it):
every env family and Ant kernel variant (4 lanes per env with 14-wide or compact solver rows, 8 and 16 lanes), ragged
batch, short episodes (resets inside the run), saturated actions, and ants thrown at walls / dropped upside down so
that the contact-slot, row and candidate indices reach their largest values.  A device-side assert aborts the process.
Used by tests/test_gpu_bounds_build.py (compute-sanitizer is closed on the pool)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from hrl_pybullet_envs_b200 import VecEnv, _cabi, config as K

assert b"HRL_BOUNDS" in _cabi.lib().hrl_version(), "not the bounds-checked build: set HRL_B200_LIB=.../libhrl_b200_chk.so"
N = 203   # ragged last warp
CASES = [("AntGatherBulletEnv-v0", {}), ("AntGatherBulletEnv-v0", dict(use_sensor=False, robot_coll_dist=0)),
         ("AntGatherBulletEnv-v0", dict(n_bins=16, respawn=False)),
         ("AntMazeBulletEnv-v0", dict(sense_target=True)), ("AntMazeBulletEnv-v0", {}), ("AntFlagrunBulletEnv-v0", dict(use_sensor=True)),
         ("AntFlagrunBulletEnv-v0", dict(max_targets=0, max_target_dist=2.0)), ("AntMjBulletEnv-v0", {}), ("AntMazeMjEnv-v0", {}),
         ("PointGatherBulletEnv-v0", {}), ("PointGatherBulletEnv-v0", dict(use_sensor=False))]
g = torch.Generator(device="cuda").manual_seed(5)
# (lanes per env, compact rows): at N = 203 hrl_create picks the 14-wide rows, so the compact ones are forced here
ANT_VARIANTS = ((4, 0), (4, 1), (8, 0), (16, 0))
for env_id, kw in CASES:
    for lanes, compact in (ANT_VARIANTS if "Point" not in env_id else ((4, 0),)):
        env = VecEnv(env_id, N, seed=1, max_episode_steps=25, **kw)
        if lanes != 4:
            _cabi.check(env.L.hrl_set_lanes_per_env(env.h, lanes))
        _cabi.check(env.L.hrl_set_compact_rows(env.h, compact))
        assert env.L.hrl_get_compact_rows(env.h) == (compact if "Point" not in env_id else 0)
        env.reset()
        for t in range(60):
            a = torch.rand(N, env.A, generator=g, device="cuda") * 2 - 1
            if t % 3 == 0:
                a = torch.sign(a)
            env.step(a, want_terminal_obs=True)
            if t == 20 and "Point" not in env_id:
                # throw the ants: random orientation (upside down: torso + many leg spheres touch), low height, fast, towards walls / the box
                f, i = env.get_state()
                q = torch.randn(N, 4, generator=g, device="cuda"); q = q / q.norm(dim=1, keepdim=True)
                f[:, K.SF_QUAT:K.SF_QUAT + 4] = q
                f[:, K.SF_POS + 2] = 0.3
                half = 4.0 if "Maze" in env_id else 5.0
                f[:, K.SF_POS] = (torch.rand(N, generator=g, device="cuda") * 2 - 1) * half
                f[:, K.SF_LINVEL:K.SF_LINVEL + 3] = torch.randn(N, 3, generator=g, device="cuda") * 6
                f[:, K.SF_ANGVEL:K.SF_ANGVEL + 3] = torch.randn(N, 3, generator=g, device="cuda") * 4
                if "Gather" in env_id:   # cubes right under the ants: cube colliders + contact pickup
                    f[:, K.SF_ITEMS:K.SF_ITEMS + 32] = (f[:, K.SF_POS:K.SF_POS + 2].repeat(1, 16) + torch.randn(N, 32, generator=g, device="cuda") * 0.4)
                env.set_state(f, i)
        env.step(np.random.uniform(-1, 1, (N, env.A)).astype(np.float32))   # host path
        env.observe()
        torch.cuda.synchronize()
        print("ok", env_id, kw, "lanes", lanes, "compact", compact)
        env.close()
print("bounds run complete")
