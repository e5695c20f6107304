"""The fused rollout's policy contract (include/hrl_b200.h `hrl_rollout_mlp_ex` / `hrl_rollout_mlp_norm`, VecEnv.rollout_mlp)

    act[t] = mlp(policy_input(obs[t])) + sigma * eps[t]

held at every env, step and component to the float64 MLP and the Philox noise references of tests/test_rollout_reference.py,
at every observation width (up to AntMazeMjEnv n_bins = 11, D = 63), both hidden widths, the plain and the normalized
policy input; and the properties a trainer relies on: two launches of T/2 steps equal one of T, two index-offset shards
equal the full batch, a launch across the 2000-step TimeLimit replays through step() bit for bit."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_gpu_rollout_training import _twins  # noqa: E402
from test_normalize import normalize_ref  # noqa: E402
from test_rollout_reference import action_tolerance, eps_actions, mlp64, torch_like_layers  # noqa: E402

from hrl_pybullet_envs_b200.config import SF_FEET, SI_STEPS, SI_T  # noqa: E402

pytestmark = pytest.mark.gpu


def _layers(D, H, A, seed):
    """nn.Linear-initialised weights: (float32 numpy layers for the references, the same values as CUDA tensors)."""
    np_layers = torch_like_layers(D, H, A, seed)
    return np_layers, tuple((torch.from_numpy(W).cuda(), torch.from_numpy(b).cuda()) for W, b in np_layers)


def _sigma(A):
    """A noise scale per component with a 0 entry (component 1) and scales from 0.1 to 0.6."""
    s = np.array([0.3, 0.0, 0.5, 0.2, 0.4, 0.25, 0.1, 0.6][:A], np.float32)
    return s, torch.from_numpy(s).cuda()


def check_policy_and_noise(buf, np_layers, draws0, genv, sigma, seed, norm=None):
    """|act - mlp64(input) - sigma eps_ref| <= tolerance at every env, step and component.  draws0: int [N], SI_STEPS of
    every env before the launch (it advances by one per step, across auto-resets); genv: global env indices [N].
    Returns the fraction of layer-3 pre-activations with |z| < 1 (the check is vacuous where tanh saturates)."""
    T, N, A = buf.act.shape
    obs, act = buf.obs[:T].cpu().numpy(), buf.act.cpu().numpy()
    if norm is not None:
        stats = (norm.mean.cpu().numpy(), norm.rstd.cpu().numpy(), norm.clip_obs)
    chunk = max(1, 16384 // N)
    small = 0
    for t0 in range(0, T, chunk):
        t1 = min(T, t0 + chunk)
        x = obs[t0:t1] if norm is None else normalize_ref(obs[t0:t1], *stats)
        y, bound, z3 = mlp64(np_layers, x)
        draws = (np.asarray(draws0, np.int64)[None, :] + np.arange(t0, t1)[:, None]).astype(np.uint64)
        eps = eps_actions(seed, np.asarray(genv, np.uint64)[None, :], draws, A)
        a = act[t0:t1]
        dev = np.abs(a - y - sigma * eps)
        bad = dev > action_tolerance(bound, a, np.broadcast_to(sigma, a.shape))
        if bad.any():
            t, e, c = np.argwhere(bad)[0]
            raise AssertionError("step %d env %d component %d: act %.9g, mlp64 %.9g, sigma eps %.9g, |dev| %.3g > bound %.3g "
                                 "(%d violations)" % (t0 + t, e, c, a[t, e, c], y[t, e, c], sigma[c] * eps[t, e, c], dev[t, e, c],
                                                      bound[t, e, c], int(bad.sum())))
        small += int((np.abs(z3) < 1).sum())
    return small / (T * N * A)


def _state_draws(env):
    f, i = env.get_state()
    return f, i, i[:, SI_STEPS].cpu().numpy()


# every family at its default width, and the widths that stress the layer-1 loop and the shared-memory sizing
POLICY_CASES = [("AntGatherBulletEnv-v0", {}, 46), ("AntMazeBulletEnv-v0", {}, None), ("AntFlagrunBulletEnv-v0", {}, 28),
                ("AntMjBulletEnv-v0", {}, 29), ("AntMazeMjEnv-v0", {}, 60), ("PointGatherBulletEnv-v0", {}, None),
                ("AntMazeMjEnv-v0", dict(n_bins=11), 63), ("AntGatherBulletEnv-v0", dict(n_bins=16), 58),
                ("AntGatherBulletEnv-v0", dict(use_sensor=False), None), ("AntMazeBulletEnv-v0", dict(sense_target=True), None),
                ("AntFlagrunBulletEnv-v0", dict(use_sensor=True), None), ("PointGatherBulletEnv-v0", dict(use_sensor=False), None)]


@pytest.mark.parametrize("normalized", [False, True])
@pytest.mark.parametrize("H", [32, 64])
@pytest.mark.parametrize("env_id,kw,D", POLICY_CASES)
def test_policy_and_noise_match_references(env_id, kw, D, H, normalized):
    """N = 203 (ragged last CTA), T = 24 across auto-resets (7-step TimeLimit).  Every action equals the float64 MLP on the
    policy input plus sigma times the Philox noise of (seed, env, SI_STEPS + t, leg), within the bound.  The component
    whose sigma is 0 equals the sigma = 0 rollout bit for bit."""
    from hrl_pybullet_envs_b200 import RunningNormalizer, VecEnv
    N, T = 203, 24
    env = VecEnv(env_id, N, seed=13, max_episode_steps=7, **kw)
    if D is not None:
        assert env.D == D
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(3):
        env.step(torch.rand(N, env.A, generator=g, device="cuda") * 2 - 1)
    norm = None
    if normalized:
        norm = RunningNormalizer(env, clip_obs=5.0)
        norm.update_obs(env.observe().clone())
        norm.rstd[1] *= 1e3                                   # the clip binds in one dimension
    np_layers, layers = _layers(env.D, H, env.A, seed=env.D + H)
    s_np, s_t = _sigma(env.A)
    seed = (0x5A5A << 32) | (17 + H)                        # both key words non-zero
    f0, i0, draws0 = _state_draws(env)
    buf = env.rollout_mlp(layers, T, sigma=s_t, noise_seed=seed, want_info=True, obs_norm=norm)
    torch.cuda.synchronize()
    assert bool(buf.done.any())
    live = check_policy_and_noise(buf, np_layers, draws0, np.arange(N), s_np, seed, norm)
    assert live >= 0.5, live
    if normalized:
        assert bool((norm.normalize(buf.obs).abs() == 5.0).any())
    env.set_state(f0, i0)
    zero = env.rollout_mlp(layers, 1, sigma=0.0, noise_seed=seed, obs_norm=norm)
    torch.cuda.synchronize()
    assert torch.equal(zero.obs[0], buf.obs[0])
    assert torch.equal(zero.act[0, :, 1], buf.act[0, :, 1])
    assert not torch.equal(zero.act[0, :, 0], buf.act[0, :, 0])


CHAIN_CASES = [("AntGatherBulletEnv-v0", {}), ("AntMazeBulletEnv-v0", {}), ("AntFlagrunBulletEnv-v0", {}),
               ("AntFlagrunBulletEnv-v0", dict(timeout=5)), ("AntMjBulletEnv-v0", {}), ("AntMazeMjEnv-v0", {}),
               ("PointGatherBulletEnv-v0", {})]


def _state_observation_columns(env_id, D):
    """The observation columns in which slot 0 of a rollout, composed from the state like hrl_observe, differs from the
    observation the step that reached that state returned, and how to read their values from the state (f, i).  Both
    follow the reference's step: the Bullet walkers' feet-contact flags measured in a step appear in the next step's
    observation (quirk Q2), and AntMazeMjEnv's time feature is self.t * 0.001 from before the step's increment."""
    if env_id in ("AntMazeBulletEnv-v0", "AntFlagrunBulletEnv-v0"):
        off = 2 if env_id == "AntFlagrunBulletEnv-v0" else 0
        return list(range(22 + off, 26 + off)), lambda f, i: f[:, SF_FEET:SF_FEET + 4]
    if env_id == "AntMazeMjEnv-v0":
        return [D - 1], lambda f, i: (i[:, SI_T].float() * 0.001)[:, None]
    return [], None


@pytest.mark.parametrize("env_id,kw", CHAIN_CASES)
def test_two_half_launches_equal_one(env_id, kw):
    """Two launches of T/2 steps give the bytes of one launch of T: act, rew, done, info, terminal observations, the
    observations and the final state.  The one exception is slot 0 of the second launch in the columns of
    _state_observation_columns: there it holds the values of the state (checked exactly), where slot T/2 of the long launch
    holds what the step returned.  The policy's weights on those columns are zero, so the actions stay comparable."""
    N, T = 203, 16
    a, b = _twins(env_id, N, max_episode_steps=5, **kw)
    _, layers = _layers(a.D, 64, a.A, seed=3)
    cols, from_state = _state_observation_columns(env_id, a.D)
    layers[0][0][:, cols] = 0.0
    _, s_t = _sigma(a.A)
    kw_r = dict(sigma=s_t, noise_seed=99, want_info=True, want_terminal_obs=True)
    full = a.rollout_mlp(layers, T, **kw_r)
    torch.cuda.synchronize()
    h = T // 2
    first = b.rollout_mlp(layers, h, **kw_r)
    f, i = b.get_state()
    second = b.rollout_mlp(layers, h, **kw_r)
    torch.cuda.synchronize()
    assert bool(full.done[:h].any()) and bool(full.done[h:].any())
    assert torch.equal(first.obs, full.obs[:h + 1]) and torch.equal(second.obs[1:], full.obs[h + 1:])
    keep = [c for c in range(a.D) if c not in cols]
    assert torch.equal(second.obs[0][:, keep], full.obs[h][:, keep])
    if cols:
        assert torch.equal(second.obs[0][:, cols], from_state(f, i))
        assert not torch.equal(second.obs[0][:, cols], full.obs[h][:, cols])
    for name in ("act", "rew", "done", "info"):
        assert torch.equal(torch.cat([getattr(first, name), getattr(second, name)]), getattr(full, name)), name
    d = full.done
    tcat = torch.cat([first.terminal_obs, second.terminal_obs])
    assert torch.equal(tcat[d], full.terminal_obs[d])
    fa, ia = a.get_state(); fb, ib = b.get_state()
    assert torch.equal(fa, fb) and torch.equal(ia, ib)


@pytest.mark.parametrize("env_id", ["AntGatherBulletEnv-v0", "PointGatherBulletEnv-v0"])
def test_index_offset_shards_equal_the_full_batch(env_id):
    """Two handles of N/2 envs with env_index_offset 0 and N/2 (the multi-GPU rule of sharding.py) write the bytes of the
    full-N rollout, noise included, and end in its state."""
    from hrl_pybullet_envs_b200 import VecEnv
    N, T = 406, 12
    full = VecEnv(env_id, N, seed=9, max_episode_steps=6)
    shards = [VecEnv(env_id, N // 2, seed=9, env_index_offset=o, max_episode_steps=6) for o in (0, N // 2)]
    o_full = full.reset().clone()
    o_sh = torch.cat([s.reset().clone() for s in shards])
    assert torch.equal(o_full, o_sh)
    np_layers, layers = _layers(full.D, 64, full.A, seed=4)
    s_np, s_t = _sigma(full.A)
    kw = dict(sigma=s_t, noise_seed=1234, want_info=True, want_terminal_obs=True)
    _, _, draws0 = _state_draws(full)
    bf = full.rollout_mlp(layers, T, **kw)
    bs = [s.rollout_mlp(layers, T, **kw) for s in shards]
    torch.cuda.synchronize()
    assert bool(bf.done.any())
    for name in ("obs", "act", "rew", "done", "info", "terminal_obs"):
        assert torch.equal(torch.cat([getattr(x, name) for x in bs], dim=1), getattr(bf, name)), name
    f, i = full.get_state()
    st = [s.get_state() for s in shards]
    assert torch.equal(torch.cat([x[0] for x in st]), f) and torch.equal(torch.cat([x[1] for x in st]), i)
    # the second shard's noise is that of global envs N/2 .. N - 1
    check_policy_and_noise(bs[1], np_layers, draws0[N // 2:], np.arange(N // 2, N), s_np, 1234)


def test_launch_across_the_time_limit():
    """AntGather at the default 2000-step TimeLimit, T = 2050 from reset, N = 203: every env still running at step 2000
    is truncated there (info), the noise reference holds at every step, and step() replays the launch bit for bit."""
    N, T = 203, 2050
    a, b = _twins("AntGatherBulletEnv-v0", N, pre_steps=0)
    np_layers, layers = _layers(a.D, 64, a.A, seed=8)
    s_np, s_t = _sigma(a.A)
    _, _, draws0 = _state_draws(a)
    buf = a.rollout_mlp(layers, T, sigma=s_t, noise_seed=77, want_info=True, want_terminal_obs=True)
    torch.cuda.synchronize()
    tr, done, length = buf.truncated, buf.done, buf.info[..., 3]
    alive = ~done[:1999].any(dim=0)
    assert bool(alive.any())
    assert torch.equal(tr[1999], alive) and not bool(tr[:1999].any())
    assert bool((length[tr] == 2000).all())
    check_policy_and_noise(buf, np_layers, draws0, np.arange(N), s_np, 77)
    assert torch.equal(b.observe(), buf.obs[0])
    for t in range(T):
        o, r, d, info = b.step(buf.act[t], want_terminal_obs=True)
        assert torch.equal(o, buf.obs[t + 1]) and torch.equal(r, buf.rew[t]) and torch.equal(d, buf.done[t]), t
        assert torch.equal(info.raw, buf.info[t]), t
        assert torch.equal(info["terminal_obs"][d], buf.terminal_obs[t][d]), t
    fa, ia = a.get_state(); fb, ib = b.get_state()
    assert torch.equal(fa, fb) and torch.equal(ia, ib)


@pytest.mark.parametrize("env_id,N", [("AntFlagrunBulletEnv-v0", 16384), ("AntGatherBulletEnv-v0", 4096)])
def test_policy_and_noise_at_production_size(env_id, N):
    """The normalized rollout at training size (T = 128, H = 64), every step against the references."""
    from hrl_pybullet_envs_b200 import RunningNormalizer, VecEnv
    T = 128
    env = VecEnv(env_id, N, seed=31, max_episode_steps=100)
    norm = RunningNormalizer(env)
    norm.update_obs(env.reset().clone())
    np_layers, layers = _layers(env.D, 64, env.A, seed=11)
    s_np, s_t = _sigma(env.A)
    _, _, draws0 = _state_draws(env)
    buf = env.rollout_mlp(layers, T, sigma=s_t, noise_seed=2026, obs_norm=norm)
    torch.cuda.synchronize()
    assert bool(buf.done.any())
    assert check_policy_and_noise(buf, np_layers, draws0, np.arange(N), s_np, 2026, norm) >= 0.5
