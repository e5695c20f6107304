"""GAE workload for the bounds-checked build (-DHRL_BOUNDS=1 -> libhrl_b200_chk.so; run with HRL_B200_LIB pointing at it):
ragged env counts (a last CTA with 1 or 8 of its 32 envs), T not divisible by the chunk count, every split of T from one
warp per env to 16, with and without terminal values.  A device-side assert aborts the process; the results are also
checked against the float64 reference.  Used by tests/test_gpu_gae.py."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
from hrl_pybullet_envs_b200 import _cabi
from test_gpu_gae import _buffer, check, synthetic

assert b"HRL_BOUNDS" in _cabi.lib().hrl_version(), "not the bounds-checked build: set HRL_B200_LIB=.../libhrl_b200_chk.so"
# (T, N): 1 warp per env for T = 1 and 7; chunks of T for 20 (2 warps), 37 (4), 100 (8), 1000 (16) at these env counts
CASES = [(1, 33), (7, 5000), (20, 1), (37, 33), (100, 5000), (1000, 33)]
G32, L32 = float(np.float32(0.99)), float(np.float32(0.95))
for T, N in CASES:
    d = synthetic(T, N, seed=T + N)
    buf = _buffer(d)
    values, tv = torch.from_numpy(d["values"]).cuda(), torch.from_numpy(d["tv"]).cuda()
    for with_tv in (True, False):
        adv, ret = buf.gae(values, 0.99, 0.95, terminal_values=tv if with_tv else None)
        torch.cuda.synchronize()
        flags = (d["info"][..., 2], d["tv"]) if with_tv else ()
        check(adv, ret, d["rew"], d["done"], d["values"], G32, L32, *flags)
        print("ok", T, N, "terminal values" if with_tv else "no terminal values", flush=True)
print("bounds gae run complete")
