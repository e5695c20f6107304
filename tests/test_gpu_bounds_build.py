"""compute-sanitizer is closed on the GPU pool, so memory safety of the kernels is checked with asserts of our own:
`libhrl_b200_chk.so` is the same source built with -DHRL_BOUNDS=1 (device-side asserts on every computed index into the
shared-memory row / impulse / candidate / staging buffers, csrc/hrl_math.cuh HRL_CHECK) and tools/bounds_run.py drives
it through every env family and Ant kernel variant (the compact solver rows included) with contact-rich states.  A failed
assert aborts that process."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHK = os.path.join(ROOT, "hrl_pybullet_envs_b200", "libhrl_b200_chk.so")


@pytest.mark.gpu
def test_bounds_checked_build_runs_clean():
    if not os.path.exists(CHK):
        pytest.skip("libhrl_b200_chk.so not built (__graft_entry__.build() makes it)")
    env = dict(os.environ, HRL_B200_LIB=CHK)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bounds_run.py")], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert "bounds run complete" in r.stdout
    assert r.stdout.count("\nok ") + r.stdout.startswith("ok ") >= 38   # 9 ant cases x 4 kernel variants + 2 point cases
