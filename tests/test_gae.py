"""GAE(lambda) over a rollout buffer (include/hrl_b200.h `hrl_gae`, RolloutBuffer.gae) without a GPU: the float64 reference of
the contract against a hand-worked case, argument validation of the C entry point, and the Python-side checks.
tests/test_gpu_gae.py compares the kernel with `gae_ref`."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest


def gae_ref(rew, done, values, gamma, lam, flags=None, terminal_values=None):
    """float64 reference of hrl_gae: rew, done [T, N], values [T + 1, N], flags = info[..., 2] and terminal_values [T, N]
    (both or neither).  Every choice is an np.where, so a value that is not selected cannot reach the result.
    Returns (adv, ret, delta)."""
    rew = np.asarray(rew, np.float64)
    done = np.asarray(done).astype(bool)
    values = np.asarray(values, np.float64)
    T = rew.shape[0]
    if flags is not None:
        trunc = done & ((np.asarray(flags).astype(np.int64) & 1) == 1)   # bit 1 (Flagrun goal switch) is ignored
        boot = np.where(trunc, np.asarray(terminal_values, np.float64), 0.0)
    else:
        boot = np.zeros_like(rew)
    nxt = np.where(done, boot, values[1:])
    delta = rew + gamma * nxt - values[:T]
    adv = np.zeros_like(rew)
    a = np.zeros(rew.shape[1:])
    for t in range(T - 1, -1, -1):
        a = np.where(done[t], delta[t], delta[t] + gamma * lam * a)
        adv[t] = a
    return adv, adv + values[:T], delta


def gae_scale(terms, gamma, lam):
    """S_t = sum_{k >= t} (gamma lam)^(k - t) terms_k (float64): the magnitude the error bound of A_t is measured against."""
    S = np.zeros_like(terms, dtype=np.float64)
    s = np.zeros(terms.shape[1:])
    for t in range(terms.shape[0] - 1, -1, -1):
        s = terms[t] + gamma * lam * s
        S[t] = s
    return S


# 2 envs, T = 4, gamma = lam = 0.5 (gamma lam = 0.25); rows are steps, columns envs
HAND = dict(
    rew=[[1, 0], [2, 0], [3, 5000], [4, 1]],
    done=[[0, 0], [1, 0], [0, 1], [1, 0]],
    # env 0: truncation at t = 1, flag 2.0 (goal switched, not truncated) = termination at t = 3;
    # env 1: a stale truncation bit at t = 0 without done (ignored), flag 3.0 (truncated and switched) at t = 2
    flags=[[0, 1], [1, 0], [0, 3], [2, 0]],
    values=[[10, 1], [20, 2], [30, 3], [40, 4], [np.nan, 5]],        # V(obs[T]) of env 0, which terminated in step T - 1: unused
    terminal_values=[[np.nan, np.nan], [8, np.nan], [np.nan, 100], [np.nan, np.nan]],   # only [1, 0] and [2, 1] are selected
)
# worked by hand: env 0  delta = [1 + 0.5*20 - 10, 2 + 0.5*8 - 20, 3 + 0.5*40 - 30, 4 - 40] = [1, -14, -7, -36]
#                        A = [1 + 0.25*(-14), -14, -7 + 0.25*(-36), -36]
#                 env 1  delta = [0 + 0.5*2 - 1, 0 + 0.5*3 - 2, 5000 + 0.5*100 - 3, 1 + 0.5*5 - 4] = [0, -0.5, 5047, -0.5]
#                        A = [0.25*1261.25, -0.5 + 0.25*5047, 5047, -0.5]
HAND_ADV = [[-2.5, 315.3125], [-14, 1261.25], [-16, 5047], [-36, -0.5]]
HAND_RET = [[7.5, 316.3125], [6, 1263.25], [14, 5050], [4, 3.5]]
# without info every done terminates: env 0 step 1 delta = 2 - 20 = -18, env 1 step 2 delta = 5000 - 3 = 4997
HAND_ADV_NOINFO = [[-3.5, 312.1875], [-18, 1248.75], [-16, 4997], [-36, -0.5]]


def test_reference_matches_the_hand_worked_case():
    h = HAND
    adv, ret, _ = gae_ref(h["rew"], h["done"], h["values"], 0.5, 0.5, h["flags"], h["terminal_values"])
    assert np.array_equal(adv, np.array(HAND_ADV, np.float64))
    assert np.array_equal(ret, np.array(HAND_RET, np.float64))
    adv, ret, _ = gae_ref(h["rew"], h["done"], h["values"], 0.5, 0.5)
    assert np.array_equal(adv, np.array(HAND_ADV_NOINFO, np.float64))
    assert np.array_equal(ret, adv + np.array(h["values"], np.float64)[:4])


def test_reference_limits():
    """lam = 0 is TD(0); gamma = lam = 1 gives Monte-Carlo returns to the end of each episode (or of the buffer)."""
    h = HAND
    _, _, delta = gae_ref(h["rew"], h["done"], h["values"], 0.5, 0.0, h["flags"], h["terminal_values"])
    adv, _, _ = gae_ref(h["rew"], h["done"], h["values"], 0.5, 0.0, h["flags"], h["terminal_values"])
    assert np.array_equal(adv, delta)
    rew = np.array([[1.0], [2.0], [3.0], [4.0]])
    done = np.array([[0], [1], [0], [0]])
    values = np.array([[0.5], [7.0], [0.25], [9.0], [100.0]])
    _, ret, _ = gae_ref(rew, done, values, 1.0, 1.0)
    assert ret[:, 0].tolist() == [3.0, 2.0, 107.0, 104.0]


# ---- C entry point: every rejection returns HRL_E_INVALID before any launch ---------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G
    from hrl_pybullet_envs_b200 import _cabi
    G.build()
    return _cabi.lib()


def _buffers(T, N):
    """Pointers to buffers of the right sizes: device memory where a GPU exists (so that an argument check that failed to
    reject could not make a kernel touch a bad address), host memory otherwise (no launch can happen there)."""
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    keep = dict(rew=torch.zeros(T, N, device=dev), done=torch.zeros(T, N, dtype=torch.uint8, device=dev),
                info=torch.zeros(T, N, 4, device=dev), values=torch.zeros(T + 1, N, device=dev),
                tv=torch.zeros(T, N, device=dev), adv=torch.zeros(T, N, device=dev), ret=torch.zeros(T, N, device=dev))
    return keep, {k: C.c_void_p(v.data_ptr()) for k, v in keep.items()}


def test_hrl_gae_rejects_bad_arguments(lib):
    T, N = 4, 8
    keep, p = _buffers(T, N)
    good = dict(T=T, N=N, gamma=0.99, lam=0.95, rew=p["rew"], done=p["done"], info=p["info"], values=p["values"], tv=p["tv"],
                adv=p["adv"], ret=p["ret"])
    bad = [dict(T=0), dict(T=-3), dict(N=0), dict(N=-1), dict(gamma=-0.01), dict(gamma=1.01), dict(gamma=float("nan")),
           dict(lam=-1e-6), dict(lam=1.5), dict(lam=float("nan")), dict(gamma=float("inf")),
           dict(rew=None), dict(done=None), dict(values=None), dict(adv=None),
           dict(info=None), dict(tv=None)]                  # info without terminal values, and the reverse
    for change in bad:
        a = dict(good, **change)
        before = lib.hrl_launch_count()
        rc = lib.hrl_gae(a["T"], a["N"], a["gamma"], a["lam"], a["rew"], a["done"], a["info"], a["values"], a["tv"], a["adv"],
                         a["ret"], None)
        assert rc == -1, change
        assert lib.hrl_launch_count() == before, change
        assert b"hrl_gae" in lib.hrl_last_error(), change
    del keep


# ---- RolloutBuffer.gae argument checks (on the CPU: they raise before anything reaches the library) ----------------
def _buf(info=True):
    import torch
    from hrl_pybullet_envs_b200 import config as K
    from hrl_pybullet_envs_b200.vec_env import RolloutBuffer
    env = SimpleNamespace(device=torch.device("cpu"), N=3, D=5, A=8, kind=K.HRL_ANT_GATHER)
    return RolloutBuffer(env, 4, info=info, terminal_obs=info)


def test_rollout_buffer_gae_validates_its_arguments():
    import torch
    b = _buf()
    v, tv = torch.zeros(5, 3), torch.zeros(4, 3)
    bad_values = [torch.zeros(4, 3), torch.zeros(5, 3, dtype=torch.float64), torch.zeros(3, 5).t(), torch.zeros(5, 3, device="meta"),
                  np.zeros((5, 3), np.float32)]
    for x in bad_values:
        with pytest.raises(ValueError, match="values"):
            b.gae(x)
    for x in (torch.zeros(5, 3), torch.zeros(4, 3, dtype=torch.float16), torch.zeros(4, 6)[:, ::2]):
        with pytest.raises(ValueError, match="terminal_values"):
            b.gae(v, terminal_values=x)
    with pytest.raises(ValueError, match="info=True"):
        _buf(info=False).gae(v, terminal_values=tv)
    for g, l in ((1.5, 0.9), (0.9, -0.1), (float("nan"), 0.9), (0.9, float("nan"))):
        with pytest.raises(ValueError, match="gamma and lam"):
            b.gae(v, g, l)
    for out in ((torch.zeros(4, 3),), (torch.zeros(4, 3), torch.zeros(5, 3)), (torch.zeros(4, 3, dtype=torch.int32), torch.zeros(4, 3))):
        with pytest.raises(ValueError, match="out"):
            b.gae(v, out=out)
