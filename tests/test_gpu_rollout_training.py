"""Fused rollout for training (hrl_rollout_mlp_ex / VecEnv.rollout_mlp): per-step info and terminal observations,
per-action noise scales, PointGather, and RolloutBuffer.info filled by capture_rollout."""
import ctypes as C
import os
import subprocess
import sys

import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHK = os.path.join(ROOT, "hrl_pybullet_envs_b200", "libhrl_b200_chk.so")


def _mlp(D, H, A, seed=0):
    g = torch.Generator().manual_seed(seed)

    def lin(o, i, s):
        return ((torch.rand(o, i, generator=g) * 2 - 1) * s).cuda(), ((torch.rand(o, generator=g) * 2 - 1) * 0.1).cuda()
    return (lin(H, D, 0.3), lin(H, H, 0.2), lin(A, H, 0.3))


def _mlp_forward(layers, obs):
    x = obs
    for W, b in layers:
        x = torch.tanh(x @ W.t() + b)
    return x


def _twins(env_id, N, pre_steps=3, **kw):
    """Two envs in the same state, a few random steps away from the reset pose."""
    from hrl_pybullet_envs_b200 import VecEnv
    a = VecEnv(env_id, N, seed=13, **kw)
    b = VecEnv(env_id, N, seed=13, **kw)
    a.reset(); b.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(pre_steps):
        act = torch.rand(N, a.A, generator=g, device="cuda") * 2 - 1
        a.step(act); b.step(act)
    return a, b


# the Flagrun case with timeout=5 switches the goal in the steps that also hit the 5-step TimeLimit: the terminal
# observation is then the one composed with the new goal, before the reset (the reference's ordering)
REPLAY_CASES = [("AntGatherBulletEnv-v0", 64, {}), ("AntMazeBulletEnv-v0", 32, {}), ("AntFlagrunBulletEnv-v0", 64, {}),
                ("AntFlagrunBulletEnv-v0", 32, dict(timeout=5)), ("AntMjBulletEnv-v0", 64, {}), ("PointGatherBulletEnv-v0", 64, {}),
                ("PointGatherBulletEnv-v0", 32, dict(use_sensor=False)),
                # cube colliders and contact pickup inside the rollout; the widest observations (AntMazeMj n_bins = 11: D = 63)
                ("AntGatherBulletEnv-v0", 64, dict(robot_coll_dist=0)), ("AntGatherBulletEnv-v0", 32, dict(n_bins=16)),
                ("AntMazeBulletEnv-v0", 64, dict(sense_target=True)), ("AntMazeBulletEnv-v0", 32, dict(max_steps=20, done_at_target=False)),
                ("AntMazeMjEnv-v0", 32, {}), ("AntMazeMjEnv-v0", 64, dict(n_bins=11)), ("AntFlagrunBulletEnv-v0", 64, dict(use_sensor=True)),
                ("AntFlagrunBulletEnv-v0", 32, dict(max_targets=0, max_target_dist=4)), ("AntFlagrunBulletEnv-v0", 64, dict(enclosed=False))]


@pytest.mark.parametrize("env_id,H,kw", REPLAY_CASES)
def test_rollout_info_and_terminal_obs_match_stepping(env_id, H, kw):
    """Replaying buf.act through step(want_terminal_obs=True) on a twin reproduces obs / rew / done, all four info columns
    and the terminal observations of the finished envs, bit for bit; the final states are identical.  N = 203 leaves a
    ragged last CTA for both the Ant (16 envs) and the PointGather (8 envs) kernels."""
    N, T = 203, 12
    a, b = _twins(env_id, N, max_episode_steps=5, **kw)
    layers = _mlp(a.D, H, a.A)
    buf = a.rollout_mlp(layers, T, sigma=0.2, noise_seed=4, want_info=True, want_terminal_obs=True)
    torch.cuda.synchronize()
    assert buf.info.shape == (T, N, 4) and buf.terminal_obs.shape == (T, N, a.D)
    assert buf.truncated.any() and (~buf.done.any(dim=1)).any()      # truncations, and steps in which no env finished
    assert torch.equal(b.observe(), buf.obs[0])
    for t in range(T):
        o, r, d, info = b.step(buf.act[t], want_terminal_obs=True)
        assert torch.equal(o, buf.obs[t + 1]) and torch.equal(r, buf.rew[t]) and torch.equal(d, buf.done[t]), t
        assert torch.equal(info.raw, buf.info[t]), t
        assert torch.equal(info["terminal_obs"][d], buf.terminal_obs[t][d]), t
        assert torch.equal(info["TimeLimit.truncated"], buf.truncated[t]), t
        assert torch.equal(buf.infos(t)["terminal_obs"][d], info["terminal_obs"][d]), t
    if kw.get("timeout"):
        switched = buf.info[..., 2] >= 2
        assert (switched & buf.done).any()                             # goal switch and reset in the same step
    fa, ia = a.get_state(); fb, ib = b.get_state()
    assert torch.equal(fa, fb) and torch.equal(ia, ib)


@pytest.mark.parametrize("H", [32, 64])
@pytest.mark.parametrize("use_sensor", [True, False])
def test_point_gather_policy_matches_torch(H, use_sensor):
    """The 16-lane in-kernel MLP of the PointGather rollout equals the torch MLP on the observation it saw, every step."""
    from hrl_pybullet_envs_b200 import VecEnv
    N, T = 1000, 10
    e = VecEnv("PointGatherBulletEnv-v0", N, seed=2, max_episode_steps=4, use_sensor=use_sensor)
    e.reset()
    layers = _mlp(e.D, H, 2, seed=H)
    buf = e.rollout_mlp(layers, T)
    torch.cuda.synchronize()
    assert torch.isfinite(buf.obs).all() and buf.done.any()
    for t in range(T):
        err = float((buf.act[t] - _mlp_forward(layers, buf.obs[t])).abs().max())
        assert err < 1e-5, (t, err)


@pytest.mark.parametrize("env_id", ["AntGatherBulletEnv-v0", "PointGatherBulletEnv-v0"])
def test_per_action_sigma(env_id):
    from hrl_pybullet_envs_b200 import VecEnv
    N = 4096
    e = VecEnv(env_id, N, seed=3)
    e.reset()
    layers = _mlp(e.D, 64, e.A, seed=1)
    f0, i0 = e.get_state()
    # a noise-scale vector filled with s draws exactly the actions of the scalar s
    scalar = e.rollout_mlp(layers, 4, sigma=0.5, noise_seed=7)
    e.set_state(f0, i0)
    vec = e.rollout_mlp(layers, 4, sigma=torch.full((e.A,), 0.5, device="cuda"), noise_seed=7)
    torch.cuda.synchronize()
    for name in ("obs", "act", "rew", "done"):
        assert torch.equal(getattr(scalar, name), getattr(vec, name)), name
    # component c gets sigma[c] * N(0, 1): the noise is measured against the torch MLP on the observation of each step
    e.set_state(f0, i0)
    sig = torch.arange(1, e.A + 1, device="cuda", dtype=torch.float32) * (0.1 if e.A == 8 else 0.3)
    T = 8
    buf = e.rollout_mlp(layers, T, sigma=sig, noise_seed=11)
    torch.cuda.synchronize()
    eps = torch.stack([(buf.act[t] - _mlp_forward(layers, buf.obs[t])) / sig for t in range(T)]).reshape(-1, e.A)
    assert (eps.mean(0).abs() < 0.02).all(), eps.mean(0)
    assert ((eps.std(0) - 1).abs() < 0.02).all(), eps.std(0)


def test_rollout_defaults_unchanged():
    """rollout_mlp without the new arguments, hrl_rollout_mlp and hrl_rollout_mlp_ex with NULLs: identical buffers."""
    from hrl_pybullet_envs_b200 import RolloutBuffer, VecEnv
    N, T = 300, 6
    e = VecEnv("AntGatherBulletEnv-v0", N, seed=5, max_episode_steps=4)
    e.reset()
    layers = _mlp(e.D, 64, 8, seed=2)
    w = e.pack_mlp(layers)
    f0, i0 = e.get_state()
    ref = e.rollout_mlp(layers, T, sigma=0.1, noise_seed=1)
    assert ref.info is None and ref.terminal_obs is None
    for call in ("old", "ex"):
        e.set_state(f0, i0)
        buf = RolloutBuffer(e, T)
        p = [C.c_void_p(t.data_ptr()) for t in (buf.obs, buf.act, buf.rew, buf.done)]
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        if call == "old":
            rc = e.L.hrl_rollout_mlp(e.h, T, C.c_void_p(w.data_ptr()), 64, 0.1, 1, *p, s)
        else:
            rc = e.L.hrl_rollout_mlp_ex(e.h, T, C.c_void_p(w.data_ptr()), 64, 0.1, None, 1, *p, None, None, s)
        assert rc == 0
        torch.cuda.synchronize()
        for name in ("obs", "act", "rew", "done"):
            assert torch.equal(getattr(ref, name), getattr(buf, name)), (call, name)


def test_capture_rollout_fills_info():
    """capture_rollout into a buffer with info: info[t] equals what step() reports, bit for bit."""
    from hrl_pybullet_envs_b200 import RolloutBuffer, VecEnv
    N, T = 128, 8
    a = VecEnv("AntGatherBulletEnv-v0", N, seed=3, max_episode_steps=3)
    b = VecEnv("AntGatherBulletEnv-v0", N, seed=3, max_episode_steps=3)
    a.reset(); b.reset()
    acts = (torch.rand(T, N, 8, device="cuda") * 2 - 1).contiguous()
    fa, ia = a.get_state()
    graph, buf = b.capture_rollout(acts, RolloutBuffer(b, T, info=True))
    b.set_state(fa, ia)
    graph.replay(); torch.cuda.synchronize()
    for t in range(T):
        o, r, d, info = a.step(acts[t])
        assert torch.equal(o, buf.obs[t + 1]) and torch.equal(r, buf.rew[t]) and torch.equal(d, buf.done[t])
        assert torch.equal(info.raw, buf.info[t]), t
    assert buf.truncated.any()


def test_rollout_argument_checks():
    from hrl_pybullet_envs_b200 import RolloutBuffer, VecEnv
    e = VecEnv("PointGatherBulletEnv-v0", 16, seed=0)
    e.reset()
    layers = _mlp(e.D, 32, 2)
    for bad in (torch.ones(3, device="cuda"), torch.tensor([0.1, -0.1], device="cuda"), torch.tensor([0.1, float("nan")], device="cuda")):
        with pytest.raises(ValueError):
            e.rollout_mlp(layers, 2, sigma=bad)
    with pytest.raises(ValueError):                        # the buffer has no room for the info the caller asked for
        e.rollout_mlp(layers, 2, buf=RolloutBuffer(e, 2), want_info=True)
    with pytest.raises(ValueError):
        RolloutBuffer(e, 2).truncated
    with pytest.raises(ValueError):                        # W3 must have A = 2 rows for PointGather
        e.rollout_mlp(_mlp(e.D, 32, 8), 2)
    with pytest.raises(ValueError):
        e.step(torch.zeros(16, 2, device="cuda"), out=RolloutBuffer(e, 1).slot(0) + (torch.zeros(16, 3, device="cuda"),))


def test_bounds_checked_build_runs_rollouts_clean():
    """tools/bounds_run_rollout.py under libhrl_b200_chk.so (device-side index asserts, -DHRL_BOUNDS=1)."""
    if not os.path.exists(CHK):
        pytest.skip("libhrl_b200_chk.so not built (__graft_entry__.build() makes it)")
    env = dict(os.environ, HRL_B200_LIB=CHK)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bounds_run_rollout.py")], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert "bounds rollout run complete" in r.stdout
    assert r.stdout.count("ok ") >= 20
