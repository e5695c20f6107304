"""GAE(lambda) kernel (include/hrl_b200.h `hrl_gae`, RolloutBuffer.gae) against the float64 reference of tests/test_gae.py:
synthetic buffers over ragged sizes and both ways of splitting T, real rollouts with TimeLimit truncations, NaN in every
value that must not be selected, determinism, CUDA-graph capture and the bounds-checked build."""
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_gae import gae_ref, gae_scale  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHK = os.path.join(ROOT, "hrl_pybullet_envs_b200", "libhrl_b200_chk.so")
TOL = 1e-5


def synthetic(T, N, seed=0):
    """A filled [T, N] buffer as numpy float32: done with p = 0.05, the truncation bit on about half of the dones, the Flagrun
    goal-switch bit at random, rewards with 5000-sized spikes (the Flagrun bonus); NaN in every terminal value that is not
    selected and in V(obs[T]) of envs that finished in step T - 1 (the value of a reset observation)."""
    rng = np.random.default_rng(seed)
    done = rng.random((T, N)) < 0.05
    trunc = done & (rng.random((T, N)) < 0.5)
    info = rng.normal(0, 1, (T, N, 4)).astype(np.float32)
    info[..., 2] = trunc + 2.0 * (rng.random((T, N)) < 0.3)
    rew = (rng.normal(0, 1, (T, N)) + 5000.0 * (rng.random((T, N)) < 0.01)).astype(np.float32)
    values = rng.normal(0, 10, (T + 1, N)).astype(np.float32)
    values[T][done[T - 1]] = np.nan
    tv = rng.normal(0, 10, (T, N)).astype(np.float32)
    tv[~trunc] = np.nan
    return dict(rew=rew, done=done, info=info, values=values, tv=tv)


def _buffer(d):
    """A RolloutBuffer on cuda:0 holding the synthetic data (the kernel reads only rew, done and info of it)."""
    from hrl_pybullet_envs_b200.vec_env import RolloutBuffer
    from hrl_pybullet_envs_b200 import config as K
    T, N = d["rew"].shape
    b = RolloutBuffer(SimpleNamespace(device=torch.device("cuda", 0), N=N, D=1, A=1, kind=K.HRL_ANT_FLAGRUN), T, info=True)
    b.rew.copy_(torch.from_numpy(d["rew"]))
    b.done.copy_(torch.from_numpy(d["done"]))
    b.info.copy_(torch.from_numpy(d["info"]))
    return b


def check(adv, ret, rew, done, values, gamma, lam, flags=None, tv=None, nan_at=None):
    """|A - A_ref| <= 1e-5 S_t and |ret - ret_ref| <= 1e-5 (S_t + |V_t|) with S_t = sum_{k >= t} (gamma lam)^(k - t) m_k,
    m_k = |r_k| + gamma |next_k| + |V_k| (>= |delta_k|; it also bounds the float32 rounding of delta_k, which the size of
    delta_k alone does not: r + gamma next - V can cancel).  NaN in the outputs exactly where `nan_at` says (default: none)."""
    adv, ret = adv.cpu().numpy().astype(np.float64), ret.cpu().numpy().astype(np.float64)
    a_ref, r_ref, delta = gae_ref(rew, done, values, gamma, lam, flags, tv)
    T = adv.shape[0]
    nan_at = np.zeros(adv.shape, bool) if nan_at is None else nan_at
    assert np.array_equal(np.isnan(adv), nan_at) and np.array_equal(np.isnan(ret), nan_at)
    assert np.array_equal(np.isnan(a_ref), nan_at)
    v = np.asarray(values, np.float64)[:T]
    r = np.asarray(rew, np.float64)
    S = gae_scale(np.nan_to_num(np.abs(r) + np.abs(delta - r + v) + np.abs(v)), gamma, lam)
    ok = ~nan_at
    ea, er = np.abs(adv - a_ref)[ok], np.abs(ret - r_ref)[ok]
    assert (ea <= TOL * S[ok]).all(), ea.max()
    assert (er <= TOL * (S + np.abs(v))[ok]).all(), er.max()


_CACHE = {}


def _data(T, N):
    if (T, N) not in _CACHE:
        d = synthetic(T, N, seed=T * 7919 + N)
        _CACHE[(T, N)] = (d, _buffer(d), torch.from_numpy(d["values"]).cuda(), torch.from_numpy(d["tv"]).cuda())
    return _CACHE[(T, N)]


# T = 1 and 7 split nothing (one warp per env); T = 128 and 1000 are split in chunks; N = 33 and 5000 leave a ragged last CTA
@pytest.mark.parametrize("N", [1, 33, 4096, 5000])
@pytest.mark.parametrize("T", [1, 7, 128, 1000])
@pytest.mark.parametrize("lam", [0.0, 0.95, 1.0])
@pytest.mark.parametrize("gamma", [0.0, 0.95, 1.0])
def test_gae_matches_reference_on_synthetic_buffers(T, N, gamma, lam):
    d, buf, values, tv = _data(T, N)
    g32, l32 = float(np.float32(gamma)), float(np.float32(lam))   # the reference uses the float32 parameters the kernel gets
    adv, ret = buf.gae(values, gamma, lam, terminal_values=tv)
    check(adv, ret, d["rew"], d["done"], d["values"], g32, l32, d["info"][..., 2], d["tv"])
    adv, ret = buf.gae(values, gamma, lam)                        # every done terminates
    check(adv, ret, d["rew"], d["done"], d["values"], g32, l32)


@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.9, 0.0)])
def test_nan_does_not_cross_an_episode_boundary(gamma, lam):
    """V(obs[t + 1]) of an env that finished in step t (a reset observation) set to NaN inside the buffer: it enters delta of
    step t + 1 and nothing else, so exactly A and ret of step t + 1 are NaN, also where the boundary falls between two chunks
    of T.  Everything else matches the reference."""
    T, N = 128, 4096
    d = synthetic(T, N, seed=3)
    hit = np.zeros((T + 1, N), bool)
    hit[1:T][d["done"][:T - 1]] = True
    d["values"][hit] = np.nan
    buf = _buffer(d)
    adv, ret = buf.gae(torch.from_numpy(d["values"]).cuda(), gamma, lam, terminal_values=torch.from_numpy(d["tv"]).cuda())
    check(adv, ret, d["rew"], d["done"], d["values"], float(np.float32(gamma)), float(np.float32(lam)), d["info"][..., 2], d["tv"],
          nan_at=hit[:T])


def _critic(D, seed=0):
    g = torch.Generator().manual_seed(seed)
    W1, b1 = (torch.rand(64, D, generator=g) - 0.5).cuda(), (torch.rand(64, generator=g) - 0.5).cuda()
    W2 = (torch.rand(1, 64, generator=g) * 20 - 10).cuda()
    return lambda x: (torch.tanh(x @ W1.t() + b1) @ W2.t())[..., 0].contiguous()


def _policy(D, A, seed=0):
    g = torch.Generator().manual_seed(seed)

    def lin(o, i, s):
        return ((torch.rand(o, i, generator=g) * 2 - 1) * s).cuda(), ((torch.rand(o, generator=g) * 2 - 1) * 0.1).cuda()
    return (lin(64, D, 0.3), lin(64, 64, 0.2), lin(A, 64, 0.3))


def _np(t):
    return t.cpu().numpy()


def _check_buffer(buf, values, tv, gamma=0.99, lam=0.95):
    flags = _np(buf.info[..., 2])
    adv, ret = buf.gae(values, gamma, lam, terminal_values=tv)
    check(adv, ret, _np(buf.rew), _np(buf.done), _np(values), float(np.float32(gamma)), float(np.float32(lam)), flags, _np(tv))
    adv, ret = buf.gae(values, gamma, lam)                        # truncations treated as terminations
    check(adv, ret, _np(buf.rew), _np(buf.done), _np(values), float(np.float32(gamma)), float(np.float32(lam)))


ROLLOUT_CASES = [("AntGatherBulletEnv-v0", {}), ("AntFlagrunBulletEnv-v0", dict(timeout=5)), ("PointGatherBulletEnv-v0", {})]


@pytest.mark.parametrize("env_id,kw", ROLLOUT_CASES)
def test_gae_on_fused_rollout_buffers(env_id, kw):
    """rollout_mlp(want_info, want_terminal_obs) with 5-step episodes; values from a random critic over buf.obs and over the
    whole of buf.terminal_obs, whose stale rows hold NaN here."""
    from hrl_pybullet_envs_b200 import RolloutBuffer, VecEnv
    N, T = 500, 24
    env = VecEnv(env_id, N, seed=4, max_episode_steps=5, **kw)
    env.reset()
    buf = RolloutBuffer(env, T, info=True, terminal_obs=True)
    buf.terminal_obs.fill_(float("nan"))
    env.rollout_mlp(_policy(env.D, env.A), T, buf=buf, sigma=0.3, noise_seed=2, want_info=True, want_terminal_obs=True)
    critic = _critic(env.D)
    values, tv = critic(buf.obs), critic(buf.terminal_obs)
    torch.cuda.synchronize()
    assert bool(buf.truncated.any()) and bool(torch.isnan(tv).any())
    if kw:
        assert bool(((buf.info[..., 2] >= 2) & buf.done).any())   # Flagrun: goal switch (bit 1) in a truncating step
    _check_buffer(buf, values, tv)


def test_gae_on_capture_rollout_buffer():
    """capture_rollout records info but no terminal observations: terminal values here are random, NaN where not selected."""
    from hrl_pybullet_envs_b200 import RolloutBuffer, VecEnv
    N, T = 300, 16
    env = VecEnv("AntGatherBulletEnv-v0", N, seed=6, max_episode_steps=5)
    env.reset()
    acts = (torch.rand(T, N, env.A, device="cuda") * 2 - 1).contiguous()
    graph, buf = env.capture_rollout(acts, RolloutBuffer(env, T, info=True))
    graph.replay()
    values = _critic(env.D, 1)(buf.obs)
    tv = torch.randn(T, N, device="cuda") * 10
    tv[~(buf.done & buf.truncated)] = float("nan")
    torch.cuda.synchronize()
    assert bool(buf.truncated.any())
    _check_buffer(buf, values, tv, 0.95, 0.9)


def test_gae_is_deterministic_and_capturable():
    """Two calls give the same bytes; with out= the call allocates nothing and replays from a CUDA graph with the same bytes."""
    d, buf, values, tv = _data(128, 4096)
    a1, r1 = buf.gae(values, 0.99, 0.95, terminal_values=tv)
    a2, r2 = buf.gae(values, 0.99, 0.95, terminal_values=tv)
    assert torch.equal(a1, a2) and torch.equal(r1, r2)
    adv, ret = torch.full_like(a1, float("nan")), torch.full_like(r1, float("nan"))
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated()
    buf.gae(values, 0.99, 0.95, terminal_values=tv, out=(adv, ret))
    assert torch.cuda.memory_allocated() == m0
    adv.fill_(float("nan")); ret.fill_(float("nan"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
        buf.gae(values, 0.99, 0.95, terminal_values=tv, out=(adv, ret))
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(adv, a1) and torch.equal(ret, r1)


def test_bounds_checked_build_runs_gae_clean():
    """tools/bounds_run_gae.py under libhrl_b200_chk.so (device-side asserts on the chunk and shared-memory indices)."""
    if not os.path.exists(CHK):
        pytest.skip("libhrl_b200_chk.so not built (__graft_entry__.build() makes it)")
    env = dict(os.environ, HRL_B200_LIB=CHK)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bounds_run_gae.py")], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert "bounds gae run complete" in r.stdout
    assert r.stdout.count("ok ") >= 12
