"""Observation and reward normalization (include/hrl_b200.h `hrl_rollout_mlp_norm`, `hrl_obs_moments`, `hrl_reward_scale`;
RunningNormalizer) without a GPU: float64 references of the three contracts against a hand-worked case, every rejection of
the C entry points, and the Python-side checks.  tests/test_gpu_normalize.py compares the kernels with these references."""
import ctypes as C
from fractions import Fraction as F

import numpy as np
import pytest


def sb3_merge(count, mean, var, bmean, bvar, bcount):
    """SB3 RunningMeanStd.update_from_moments, in its order of operations (float64 numpy or Fractions)."""
    delta = bmean - mean
    tot = count + bcount
    new_mean = mean + delta * bcount / tot
    m2 = var * count + bvar * bcount + delta * delta * count * bcount / tot
    return tot, new_mean, m2 / tot


def obs_moments_ref(moments, x, eps):
    """hrl_obs_moments: moments = (count, mean[D], var[D]) float64, x [..., D].  Returns (count, mean, var, mean_f, rstd_f)."""
    count, mean, var = moments
    x = np.asarray(x, np.float64)
    x = x.reshape(-1, x.shape[-1])
    count, mean, var = sb3_merge(count, np.asarray(mean, np.float64), np.asarray(var, np.float64), x.mean(0), x.var(0),
                                 float(x.shape[0]))
    rstd = (1.0 / np.sqrt(var + float(np.float32(eps)))).astype(np.float32)
    return count, mean, var, mean.astype(np.float32), rstd


def reward_scale_ref(rew, done, returns, moments, gamma, clip, eps):
    """hrl_reward_scale step by step (SB3 VecNormalize step_wait -> _update_reward -> normalize_reward), float64 returns.
    gamma, clip and eps are used as the float32 values the kernel receives.  Returns (out f32[T, N], returns, moments, s)."""
    g, c, e = (float(np.float32(v)) for v in (gamma, clip, eps))
    rew = np.asarray(rew, np.float32)
    done = np.asarray(done).astype(bool)
    R = np.array(returns, np.float64)
    count, mean, var = moments
    out = np.zeros(rew.shape, np.float32)
    s_all = np.zeros(rew.shape[0], np.float32)
    for t in range(rew.shape[0]):
        R = R * g + rew[t].astype(np.float64)
        count, mean, var = sb3_merge(count, mean, var, R.mean(), R.var(), float(R.shape[0]))
        s = np.float32(1.0 / np.sqrt(var + e))
        out[t] = np.clip(rew[t] * s, np.float32(-c), np.float32(c))
        s_all[t] = s
        R = np.where(done[t], 0.0, R)
    return out, R, (count, mean, var), s_all


def normalize_ref(obs, mean_f, rstd_f, clip):
    """The policy input of hrl_rollout_mlp_norm: subtract, multiply, clamp, each in float32."""
    c = np.float32(clip)
    return np.minimum(np.maximum((np.float32(obs) - mean_f) * rstd_f, -c), c).astype(np.float32)


# ---- hand-worked cases -------------------------------------------------------------------------------------------------
def test_obs_moments_reference_matches_the_hand_worked_case():
    """D = 2 from (count 1, mean 0, var 1).  Batch 1 [[1, 2], [3, 2]]: bmean (2, 2), bvar (1, 0), delta 2, tot 3,
    mean 4/3, M2 = var + 2 bvar + 4 * 2/3 = (17/3, 11/3), var (17/9, 11/9).  Batch 2 [[0, 4]]: delta (-4/3, 8/3), tot 4,
    mean (1, 2), M2 = 3 var + delta^2 * 3/4 = (7, 9), var (7/4, 9/4)."""
    st = (1.0, np.zeros(2), np.ones(2))
    c, m, v, _, _ = obs_moments_ref(st, [[1, 2], [3, 2]], 1e-8)
    assert c == 3 and np.allclose(m, [4 / 3, 4 / 3], rtol=1e-15) and np.allclose(v, [17 / 9, 11 / 9], rtol=1e-15)
    c, m, v, mf, rf = obs_moments_ref((c, m, v), [[0, 4]], 0.25)
    assert c == 4 and np.allclose(m, [1, 2], rtol=1e-15) and np.allclose(v, [7 / 4, 9 / 4], rtol=1e-15)
    assert mf.dtype == np.float32 and np.array_equal(rf, np.float32([1 / np.sqrt(2.0), 1 / np.sqrt(2.5)]))   # 1 / sqrt(var + 0.25)


def test_reward_scale_reference_matches_the_hand_worked_case():
    """2 envs, 3 steps, gamma 0.5, from moments (count 2, mean 0, var 1), env 1 done in step 0, clip 2.2 binding once.
    t0: R (1, 2), bmean 1.5, bvar 0.25 -> count 4, mean 0.75, var (2 + 0.5 + 2.25 * 2 * 2/4) / 4 = 1.1875; env 1 restarts.
    t1: R (3.5, 0), bmean 1.75, bvar 3.0625 -> count 6, mean 13/12, var 293/144; 3 s_1 = 2.103 stays below 2.2.
    t2: R (1.75, 4), bmean 23/8, bvar 81/64 -> count 8, mean 49/32, var 7509/3072; 4 s_2 = 2.558 is clipped to 2.2."""
    rew = [[1, 2], [3, 0], [0, 4]]
    done = [[0, 1], [0, 0], [0, 0]]
    out, R, (c, m, v), s = reward_scale_ref(rew, done, [0.0, 0.0], (2.0, 0.0, 1.0), 0.5, 2.2, 1e-8)
    # the same chain in exact arithmetic
    fc, fm, fv = F(2), F(0), F(1)
    for bm, bv in ((F(3, 2), F(1, 4)), (F(7, 4), F(49, 16)), (F(23, 8), F(81, 64))):
        fc, fm, fv = sb3_merge(fc, fm, fv, bm, bv, F(2))
    assert (fc, fm, fv) == (8, F(49, 32), F(7509, 3072))
    assert c == 8 and m == 49 / 32 and abs(v - 7509 / 3072) < 1e-15
    assert R.tolist() == [1.75, 4.0]
    e = float(np.float32(1e-8))
    s_exact = [1 / np.sqrt(1.1875 + e), 1 / np.sqrt(293 / 144 + e), 1 / np.sqrt(7509 / 3072 + e)]
    assert np.array_equal(s, np.float32(s_exact))
    c32 = np.float32(2.2)
    assert out[2, 1] == c32 and (np.abs(out) < c32).sum() == 5                       # exactly one clipped reward
    assert out[0, 0] == np.float32(1) * s[0] and out[1, 0] == np.float32(3) * s[1] and out[1, 1] == 0.0


def test_reward_scale_reference_splits_over_calls():
    """Two calls over consecutive halves (returns and moments carried) equal one call over the whole buffer."""
    rng = np.random.default_rng(0)
    rew = rng.normal(0, 1, (20, 5)).astype(np.float32)
    done = rng.random((20, 5)) < 0.2
    st = (1e-4, 0.0, 1.0)
    out, R, mom, _ = reward_scale_ref(rew, done, np.zeros(5), st, 0.99, 10, 1e-8)
    o1, R1, m1, _ = reward_scale_ref(rew[:7], done[:7], np.zeros(5), st, 0.99, 10, 1e-8)
    o2, R2, m2, _ = reward_scale_ref(rew[7:], done[7:], R1, m1, 0.99, 10, 1e-8)
    assert np.array_equal(np.concatenate([o1, o2]), out) and np.array_equal(R2, R) and m2 == mom


def test_normalize_reference_clamps_after_scaling():
    x = normalize_ref([[1.0, -3.0, 1e30]], np.float32([0.5, 0, 0]), np.float32([2, 1e4, 1]), 10.0)
    assert x.tolist() == [[1.0, -10.0, 10.0]]


# ---- C entry points: every rejection returns HRL_E_INVALID before any launch --------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G
    from hrl_pybullet_envs_b200 import _cabi
    G.build()
    return _cabi.lib()


def _mem(**shapes):
    """Buffers of the right sizes: device memory where a GPU exists, host memory otherwise (no launch can happen there)."""
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    keep = {k: torch.zeros(*s, dtype=dt, device=dev) for k, (s, dt) in shapes.items()}
    return keep, {k: C.c_void_p(v.data_ptr()) for k, v in keep.items()}


def _rejects(lib, fn, name, good, bad, call):
    for change in bad:
        a = dict(good, **change)
        before = lib.hrl_launch_count()
        assert call(fn, a) == -1, change
        assert lib.hrl_launch_count() == before, change
        assert name.encode() in lib.hrl_last_error(), change


def test_hrl_obs_moments_rejects_bad_arguments(lib):
    import torch
    keep, p = _mem(x=((7, 5), torch.float32), mom=((11,), torch.float64), mf=((5,), torch.float32), rf=((5,), torch.float32))
    good = dict(M=7, D=5, x=p["x"], mom=p["mom"], eps=1e-8, mf=p["mf"], rf=p["rf"])
    bad = [dict(M=0), dict(M=-1), dict(D=0), dict(D=-2), dict(D=65), dict(x=None), dict(mom=None), dict(mf=None), dict(rf=None),
           dict(eps=0.0), dict(eps=-1e-8), dict(eps=float("nan"))]
    _rejects(lib, lib.hrl_obs_moments, "hrl_obs_moments", good, bad,
             lambda f, a: f(a["M"], a["D"], a["x"], a["mom"], a["eps"], a["mf"], a["rf"], None))
    del keep


def test_hrl_reward_scale_rejects_bad_arguments(lib):
    import torch
    T, N = 4, 6
    keep, p = _mem(rew=((T, N), torch.float32), done=((T, N), torch.uint8), ret=((N,), torch.float64), mom=((3,), torch.float64),
                   work=((2 * T,), torch.float64), out=((T, N), torch.float32))
    good = dict(T=T, N=N, gamma=0.99, clip=10.0, eps=1e-8, **p)
    nan = float("nan")
    bad = [dict(T=0), dict(T=-1), dict(N=0), dict(N=-5), dict(gamma=-0.1), dict(gamma=1.01), dict(gamma=nan), dict(clip=0.0),
           dict(clip=-1.0), dict(clip=nan), dict(eps=0.0), dict(eps=-1.0), dict(eps=nan), dict(rew=None), dict(done=None),
           dict(ret=None), dict(mom=None), dict(work=None), dict(out=None)]
    _rejects(lib, lib.hrl_reward_scale, "hrl_reward_scale", good, bad,
             lambda f, a: f(a["T"], a["N"], a["gamma"], a["clip"], a["eps"], a["rew"], a["done"], a["ret"], a["mom"], a["work"],
                            a["out"], None))
    del keep


def test_hrl_rollout_mlp_norm_rejects_a_null_handle(lib):
    """Without a GPU no handle exists: a NULL handle is rejected with and without statistics, and nothing launches.
    The checks of the statistics themselves need a handle: tests/test_gpu_normalize.py makes them."""
    import torch
    keep, p = _mem(w=((64 * 64 * 3,), torch.float32), m=((30,), torch.float32), r=((30,), torch.float32),
                   obs=((3, 4, 30), torch.float32), act=((2, 4, 8), torch.float32), rew=((2, 4), torch.float32),
                   done=((2, 4), torch.uint8))
    good = dict(m=p["m"], r=p["r"], clip=10.0)
    bad = [dict(), dict(m=None, r=None, clip=0.0), dict(m=None), dict(clip=float("nan"))]
    _rejects(lib, lib.hrl_rollout_mlp_norm, "hrl_rollout_mlp", good, bad,
             lambda f, a: f(None, 2, p["w"], 64, 0.0, None, 0, a["m"], a["r"], a["clip"], p["obs"], p["act"], p["rew"], p["done"],
                            None, None, None))
    del keep


# ---- RunningNormalizer argument checks (CPU tensors: they raise before anything reaches the library) ---------------------
def _norm(N=3, D=4):
    import torch
    from hrl_pybullet_envs_b200.normalize import RunningNormalizer
    return RunningNormalizer((N, D, torch.device("cpu")))


def test_running_normalizer_initial_state_and_settings():
    import torch
    from hrl_pybullet_envs_b200.normalize import RunningNormalizer
    n = _norm()
    assert n.obs_moments.dtype == torch.float64 and n.obs_moments.tolist() == [1e-4] + [0.0] * 4 + [1.0] * 4
    assert n.ret_moments.tolist() == [1e-4, 0.0, 1.0] and n.returns.tolist() == [0.0] * 3
    assert torch.equal(n.rstd, torch.full((4,), float(np.float32(1 / np.sqrt(1 + float(np.float32(1e-8))))))) and n.mean.abs().sum() == 0
    for kw in (dict(gamma=1.5), dict(gamma=-0.1), dict(clip_obs=0.0), dict(clip_obs=float("inf")), dict(clip_reward=-1.0),
               dict(epsilon=0.0)):
        with pytest.raises(ValueError):
            RunningNormalizer((3, 4, torch.device("cpu")), **kw)
    for dims in ((0, 4, "cpu"), (3, 0, "cpu"), (3, 65, "cpu")):
        with pytest.raises(ValueError):
            RunningNormalizer(dims)


def test_running_normalizer_validates_its_arguments():
    import torch
    n = _norm()
    for x in (torch.zeros(5, 3), torch.zeros(5, 4, dtype=torch.float64), torch.zeros(4, 5).t(), np.zeros((5, 4), np.float32),
              torch.zeros(0, 4), torch.zeros(5, 4, device="meta")):
        with pytest.raises(ValueError):
            n.update_obs(x)
    rew, done = torch.zeros(2, 3), torch.zeros(2, 3, dtype=torch.bool)
    for r in (torch.zeros(2, 4), torch.zeros(2, 3, dtype=torch.float64), torch.zeros(3, 2).t(), torch.zeros(6)):
        with pytest.raises(ValueError, match="rew"):
            n.scale_rewards(r, done)
    for d in (torch.zeros(2, 4, dtype=torch.bool), torch.zeros(2, 3), torch.zeros(3, 2, dtype=torch.bool).t()):
        with pytest.raises(ValueError, match="done"):
            n.scale_rewards(rew, d)
    for o in (torch.zeros(2, 4), torch.zeros(2, 3, dtype=torch.float16), rew):
        with pytest.raises(ValueError, match="out"):
            n.scale_rewards(rew, done, out=o)
    with pytest.raises(ValueError, match="mask"):
        n.reset_returns(torch.ones(4, dtype=torch.bool))


def test_running_normalizer_state_dict_round_trip_and_reset_returns():
    import torch
    a, b = _norm(), _norm()
    a.obs_moments.copy_(torch.tensor([10.0, 1, 2, 3, 4, 0.25, 1, 4, 9], dtype=torch.float64))
    a.ret_moments.copy_(torch.tensor([5.0, 2.0, 3.0], dtype=torch.float64))
    a.returns.copy_(torch.tensor([1.0, -2.0, 3.0], dtype=torch.float64))
    b.load_state_dict(a.state_dict())
    assert torch.equal(a.obs_moments, b.obs_moments) and torch.equal(a.ret_moments, b.ret_moments) and torch.equal(a.returns, b.returns)
    e = float(np.float32(1e-8))
    assert b.mean.tolist() == [1.0, 2.0, 3.0, 4.0]
    assert np.array_equal(b.rstd.numpy(), (1 / np.sqrt(np.array([0.25, 1, 4, 9]) + e)).astype(np.float32))
    with pytest.raises(ValueError):
        _norm(D=5).load_state_dict(a.state_dict())
    from hrl_pybullet_envs_b200.normalize import RunningNormalizer
    with pytest.raises(ValueError):
        RunningNormalizer((3, 4, torch.device("cpu")), gamma=0.9).load_state_dict(a.state_dict())
    b.reset_returns(torch.tensor([True, False, True]))
    assert b.returns.tolist() == [0.0, -2.0, 0.0]
    b.reset_returns()
    assert b.returns.tolist() == [0.0, 0.0, 0.0]


def test_normalize_matches_the_reference_bit_for_bit():
    import torch
    n = _norm(D=4)
    n.mean.copy_(torch.tensor([0.1, -3.0, 1e3, 0.0]))
    n.rstd.copy_(torch.tensor([3.0, 0.5, 1e4, 7.0]))
    x = torch.tensor(np.random.default_rng(1).normal(0, 5, (50, 4)).astype(np.float32)) + torch.tensor([0, 0, 1e3, 0])
    ref = normalize_ref(x.numpy(), n.mean.numpy(), n.rstd.numpy(), 10.0)
    assert np.array_equal(n.normalize(x).numpy(), ref) and (np.abs(ref) == 10).any()
