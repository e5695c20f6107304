"""Observation and reward normalization on the GPU (hrl_rollout_mlp_norm, hrl_obs_moments, hrl_reward_scale; RunningNormalizer)
against the float64 references of tests/test_normalize.py: the normalized fused rollout (identity statistics reproduce the
plain rollout bit for bit; real statistics with a binding clip match the torch policy on norm.normalize(obs) and replay
through step()), the two statistics kernels over ragged sizes, determinism, CUDA-graph capture, a PPO loop at 4096 envs and
the bounds-checked build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_gae import gae_ref  # noqa: E402
from test_gpu_rollout_training import REPLAY_CASES, _mlp, _mlp_forward, _twins  # noqa: E402
from test_normalize import normalize_ref, obs_moments_ref, reward_scale_ref  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHK = os.path.join(ROOT, "hrl_pybullet_envs_b200", "libhrl_b200_chk.so")


def _norm(env, **kw):
    from hrl_pybullet_envs_b200 import RunningNormalizer
    return RunningNormalizer(env, **kw)


def _compare_buffers(x, y):
    for name in ("obs", "act", "rew", "done", "info", "terminal_obs"):
        assert torch.equal(getattr(x, name), getattr(y, name)), name


@pytest.mark.parametrize("env_id,H,kw", REPLAY_CASES)
def test_identity_normalization_reproduces_the_rollout(env_id, H, kw):
    """mean 0, rstd 1 and a clip above every observation: the normalized instantiation writes the same bytes as the plain
    one (N = 203: ragged last CTA), and both handles end in the same state."""
    N, T = 203, 12
    a, b = _twins(env_id, N, max_episode_steps=5, **kw)
    norm = _norm(a, clip_obs=3e38)
    norm.mean.zero_(); norm.rstd.fill_(1.0)
    layers = _mlp(a.D, H, a.A)
    x = a.rollout_mlp(layers, T, sigma=0.2, noise_seed=4, want_info=True, want_terminal_obs=True, obs_norm=norm)
    y = b.rollout_mlp(layers, T, sigma=0.2, noise_seed=4, want_info=True, want_terminal_obs=True)
    torch.cuda.synchronize()
    assert bool(x.done.any())
    _compare_buffers(x, y)
    fa, ia = a.get_state(); fb, ib = b.get_state()
    assert torch.equal(fa, fb) and torch.equal(ia, ib)


NORM_CASES = [("AntGatherBulletEnv-v0", 32, {}), ("AntGatherBulletEnv-v0", 64, {}), ("AntFlagrunBulletEnv-v0", 64, {}),
              ("PointGatherBulletEnv-v0", 32, {}), ("PointGatherBulletEnv-v0", 64, dict(use_sensor=False))]


@pytest.mark.parametrize("env_id,H,kw", NORM_CASES)
def test_normalized_policy_matches_torch_and_replays(env_id, H, kw):
    """Statistics of a previous rollout, one dimension's rstd inflated so that the clip binds.  At sigma = 0 the in-kernel
    actions equal the torch MLP on norm.normalize(buf.obs[t]) at every step; replaying buf.act through step() on a twin
    reproduces every output bit for bit, and the buffer holds the raw observations."""
    N, T = 203, 10
    a, b = _twins(env_id, N, max_episode_steps=6, **kw)
    layers = _mlp(a.D, H, a.A, seed=H)
    norm = _norm(a, clip_obs=5.0)
    pre = a.rollout_mlp(layers, T, sigma=0.3, noise_seed=1)
    b.rollout_mlp(layers, T, sigma=0.3, noise_seed=1)
    norm.update_obs(pre.obs[1:].contiguous())
    norm.rstd[1] *= 1e3
    buf = a.rollout_mlp(layers, T, noise_seed=2, want_info=True, want_terminal_obs=True, obs_norm=norm)
    torch.cuda.synchronize()
    assert bool(buf.done.any())
    clipped = 0
    for t in range(T):
        x = norm.normalize(buf.obs[t])
        ref = normalize_ref(buf.obs[t].cpu().numpy(), norm.mean.cpu().numpy(), norm.rstd.cpu().numpy(), 5.0)
        assert np.array_equal(x.cpu().numpy(), ref), t
        clipped += int((x.abs() == 5.0).sum())
        err = float((buf.act[t] - _mlp_forward(layers, x)).abs().max())
        assert err < 1e-5, (t, err)
    assert clipped > 0
    assert torch.equal(b.observe(), buf.obs[0])       # raw observations in the buffer
    for t in range(T):
        o, r, d, info = b.step(buf.act[t], want_terminal_obs=True)
        assert torch.equal(o, buf.obs[t + 1]) and torch.equal(r, buf.rew[t]) and torch.equal(d, buf.done[t]), t
        assert torch.equal(info.raw, buf.info[t]), t
        assert torch.equal(info["terminal_obs"][d], buf.terminal_obs[t][d]), t
    fa, ia = a.get_state(); fb, ib = b.get_state()
    assert torch.equal(fa, fb) and torch.equal(ia, ib)


def test_rollout_mlp_norm_rejects_bad_statistics():
    from hrl_pybullet_envs_b200 import RolloutBuffer, VecEnv
    e = VecEnv("AntGatherBulletEnv-v0", 16, seed=0)
    e.reset()
    w = e.pack_mlp(_mlp(e.D, 32, 8))
    buf = RolloutBuffer(e, 2)
    m, r = torch.zeros(e.D, device="cuda"), torch.ones(e.D, device="cuda")
    p = [C.c_void_p(t.data_ptr()) for t in (buf.obs, buf.act, buf.rew, buf.done)]
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    pm, pr = C.c_void_p(m.data_ptr()), C.c_void_p(r.data_ptr())
    for mm, rr, clip in ((pm, None, 10.0), (None, pr, 10.0), (pm, pr, 0.0), (pm, pr, -1.0), (pm, pr, float("inf")), (pm, pr, float("nan"))):
        before = e.L.hrl_launch_count()
        assert e.L.hrl_rollout_mlp_norm(e.h, 2, C.c_void_p(w.data_ptr()), 32, 0.0, None, 0, mm, rr, clip, *p, None, None, s) == -1
        assert e.L.hrl_launch_count() == before and b"hrl_rollout_mlp_norm" in e.L.hrl_last_error()
    assert e.L.hrl_rollout_mlp_norm(e.h, 2, C.c_void_p(w.data_ptr()), 32, 0.0, None, 0, None, None, 0.0, *p, None, None, s) == 0
    with pytest.raises(ValueError):
        e.rollout_mlp(_mlp(e.D, 32, 8), 2, obs_norm=_norm((16, e.D - 1)))


# ---- hrl_obs_moments ---------------------------------------------------------------------------------------------------
def _obs_data(M, D, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(0, 1, (M, D)).astype(np.float32) * rng.uniform(0.1, 10, D).astype(np.float32)
    x[:, D // 2] = (1e3 + rng.normal(0, 1e-2, M)).astype(np.float32)     # the offset dimension: mean 1e3, std 1e-2
    if D > 3:
        x[:, 0] = 0.0                                                     # a dimension that is zero for long stretches
    return x


@pytest.mark.parametrize("D", [2, 18, 28, 46, 60])
@pytest.mark.parametrize("M", [1, 7, 203, 128 * 4096])
def test_obs_moments_match_reference(M, D):
    """Three chained updates against three sequential reference updates; rstd_f is the reference rounded to float32;
    the same call from the same state gives the same bytes."""
    n = _norm((1, D))
    ref = (1e-4, np.zeros(D), np.ones(D))
    for k in range(3):
        x = _obs_data(M, D, seed=M + D + k)
        before = n.obs_moments.clone()
        xt = torch.from_numpy(x).cuda()
        n.update_obs(xt)
        c, m, v, mf, rf = obs_moments_ref(ref, x, 1e-8)
        ref = (c, m, v)
        got = n.obs_moments.cpu().numpy()
        assert got[0] == c
        std = np.sqrt(v)
        assert (np.abs(got[1:1 + D] - m) <= 1e-9 * std + 1e-15 * np.abs(m)).all(), np.abs(got[1:1 + D] - m).max()
        assert (np.abs(got[1 + D:] - v) <= 1e-9 * v).all(), (np.abs(got[1 + D:] - v) / v).max()
        assert np.array_equal(n.mean.cpu().numpy(), mf) and np.array_equal(n.rstd.cpu().numpy(), rf)
        after = n.obs_moments.clone()
        n.obs_moments.copy_(before)
        n.update_obs(xt)
        assert torch.equal(n.obs_moments, after)


# ---- hrl_reward_scale --------------------------------------------------------------------------------------------------
def _rew_data(T, N, seed):
    rng = np.random.default_rng(seed)
    rew = (rng.normal(0.5, 1, (T, N)) + 5000.0 * (rng.random((T, N)) < 0.002)).astype(np.float32)
    rew[T // 2, N // 2] = 5000.0                                          # at least one spike, so the clip binds for T > 1
    done = rng.random((T, N)) < 0.02
    return rew, done


def _check_scaled(out, n, ref_out, ref_R, ref_mom):
    o = out.cpu().numpy()
    assert (np.abs(o - ref_out) <= 1e-6 * np.abs(ref_out)).all(), np.abs(o - ref_out).max()
    assert np.array_equal(n.returns.cpu().numpy(), ref_R)
    got = n.ret_moments.cpu().numpy()
    assert got[0] == ref_mom[0] and abs(got[1] - ref_mom[1]) <= 1e-6 * (abs(ref_mom[1]) + np.sqrt(ref_mom[2]))
    assert abs(got[2] - ref_mom[2]) <= 1e-6 * ref_mom[2]


@pytest.mark.parametrize("N", [1, 33, 4096, 16384])
@pytest.mark.parametrize("T", [1, 7, 128, 1000])
def test_reward_scale_matches_reference(T, N):
    """Against the step-by-step reference, with dones, 5000-sized spikes and a binding clip; two consecutive calls equal
    one call over the concatenated buffers, bit for bit; a repeat from the same state gives the same bytes."""
    rew, done = _rew_data(T, N, seed=T * 31 + N)
    n = _norm((N, 1), clip_reward=5.0)
    r, d = torch.from_numpy(rew).cuda(), torch.from_numpy(done).cuda()
    out = n.scale_rewards(r, d)
    ref_out, ref_R, ref_mom, _ = reward_scale_ref(rew, done, np.zeros(N), (1e-4, 0.0, 1.0), 0.99, 5.0, 1e-8)
    _check_scaled(out, n, ref_out, ref_R, ref_mom)
    if T > 1:
        assert (np.abs(ref_out) == np.float32(5.0)).any()
    sd = n.state_dict()
    n.reset_statistics()
    h = T // 2 if T > 1 else 1
    parts = [n.scale_rewards(r[:h].contiguous(), d[:h].contiguous())]
    if h < T:
        parts.append(n.scale_rewards(r[h:].contiguous(), d[h:].contiguous()))
    assert torch.equal(torch.cat(parts), out)
    assert torch.equal(n.returns, sd["returns"]) and torch.equal(n.ret_moments, sd["ret_moments"])
    n.reset_statistics()
    again = n.scale_rewards(r, d)
    assert torch.equal(again, out) and torch.equal(n.ret_moments, sd["ret_moments"])


def test_one_graph_holds_update_scale_and_gae():
    """update_obs, scale_rewards and gae(rew=...) captured in one CUDA graph: a replay equals the eager calls bit for bit."""
    from test_gpu_gae import _buffer, synthetic
    T, N, D = 128, 4096, 28
    d = synthetic(T, N, seed=9)
    buf = _buffer(d)
    values = torch.from_numpy(d["values"]).cuda()
    x = torch.from_numpy(_obs_data(T * N, D, 3)).cuda()
    n = _norm((N, D))
    scaled = torch.empty(T, N, device="cuda")
    adv, ret = torch.empty(T, N, device="cuda"), torch.empty(T, N, device="cuda")

    def work():
        n.update_obs(x)
        n.scale_rewards(buf.rew, buf.done, out=scaled)
        buf.gae(values, 0.99, 0.95, out=(adv, ret), rew=scaled)

    work()                                        # eager (allocates the work buffer once)
    torch.cuda.synchronize()
    want = [t.clone() for t in (n.obs_moments, n.mean, n.rstd, n.ret_moments, n.returns, scaled, adv, ret)]
    n.reset_statistics()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
        work()
    torch.cuda.current_stream().wait_stream(s)
    n.reset_statistics()
    scaled.fill_(float("nan")); adv.fill_(float("nan"))
    g.replay()
    torch.cuda.synchronize()
    got = (n.obs_moments, n.mean, n.rstd, n.ret_moments, n.returns, scaled, adv, ret)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    a_ref, _, _ = gae_ref(scaled.cpu().numpy(), d["done"], d["values"], float(np.float32(0.99)), float(np.float32(0.95)))
    assert np.allclose(adv.cpu().numpy(), a_ref, rtol=1e-4, atol=1e-4)


def test_ppo_loop_against_float64_pipeline():
    """The documented loop on AntGather at 4096 envs for 3 iterations, against a float64 reference pipeline run on the same
    buffers: observation statistics, the policy input, scaled rewards and GAE."""
    from hrl_pybullet_envs_b200 import VecEnv
    N, T = 4096, 32
    vec = VecEnv("AntGatherBulletEnv-v0", N, seed=21, max_episode_steps=40)
    layers = _mlp(vec.D, 64, vec.A, seed=5)
    g = torch.Generator().manual_seed(0)
    W1, W2 = (torch.rand(64, vec.D, generator=g) - 0.5).cuda(), (torch.rand(1, 64, generator=g) - 0.5).cuda()
    critic = lambda x: (torch.tanh(x @ W1.t()) @ W2.t())[..., 0].contiguous()  # noqa: E731
    norm = _norm(vec)
    obs0 = vec.reset()
    norm.update_obs(obs0)
    ref_obs = obs_moments_ref((1e-4, np.zeros(vec.D), np.ones(vec.D)), obs0.cpu().numpy(), 1e-8)[:3]
    ref_R, ref_rm = np.zeros(N), (1e-4, 0.0, 1.0)
    log_std = torch.full((vec.A,), -0.5, device="cuda")
    for it in range(3):
        buf = vec.rollout_mlp(layers, T, sigma=log_std.exp(), noise_seed=it, want_info=True, want_terminal_obs=True, obs_norm=norm)
        x, xt = norm.normalize(buf.obs), norm.normalize(buf.terminal_obs)
        mean_f = ref_obs[1].astype(np.float32)
        rstd_f = (1.0 / np.sqrt(ref_obs[2] + float(np.float32(1e-8)))).astype(np.float32)
        assert np.array_equal(norm.mean.cpu().numpy(), mean_f) and np.array_equal(norm.rstd.cpu().numpy(), rstd_f)
        assert np.array_equal(x.cpu().numpy(), normalize_ref(buf.obs.cpu().numpy(), mean_f, rstd_f, 10.0))
        for t in (0, T // 2, T - 1):                           # the in-kernel policy saw x (noise removed)
            mu = _mlp_forward(layers, x[t])
            eps = (buf.act[t] - mu) / log_std.exp()
            assert float(eps.abs().max()) < 8 and abs(float(eps.std()) - 1) < 0.05
        norm.update_obs(buf.obs[1:])
        ref_obs = obs_moments_ref(ref_obs, buf.obs[1:].cpu().numpy(), 1e-8)[:3]
        r = norm.scale_rewards(buf.rew, buf.done)
        ref_out, ref_R, ref_rm, _ = reward_scale_ref(buf.rew.cpu().numpy(), buf.done.cpu().numpy(), ref_R, ref_rm, 0.99, 10.0, 1e-8)
        _check_scaled(r, norm, ref_out, ref_R, ref_rm)
        v, vt = critic(x), critic(xt)
        adv, ret = buf.gae(v, 0.99, 0.95, vt, rew=r)
        a_ref, _, _ = gae_ref(ref_out, buf.done.cpu().numpy(), v.cpu().numpy(), float(np.float32(0.99)), float(np.float32(0.95)),
                              buf.info[..., 2].cpu().numpy(), vt.cpu().numpy())
        assert np.allclose(adv.cpu().numpy(), a_ref, rtol=1e-4, atol=1e-4)
    assert bool(buf.done.any())


def test_bounds_checked_build_runs_normalization_clean():
    """tools/bounds_run_normalize.py under libhrl_b200_chk.so (device-side index asserts, -DHRL_BOUNDS=1)."""
    if not os.path.exists(CHK):
        pytest.skip("libhrl_b200_chk.so not built (__graft_entry__.build() makes it)")
    env = dict(os.environ, HRL_B200_LIB=CHK)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bounds_run_normalize.py")], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert "bounds normalize run complete" in r.stdout
    assert r.stdout.count("ok ") >= 14
