"""Population evaluation (hrl_evaluate_mlp / VecEnv.evaluate_mlp): P MLP policies in one launch, per-env return, length and
finished flag of the first episode, no per-step buffers.  Every result is pinned bit for bit to the fused rollout: member m's
envs of one launch must equal a `rollout_mlp` of member m alone on a handle of its M envs (same seed, env_index_offset = m M),
with the rewards summed in float32 in step order up to the first done, and end in the same state."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHK = os.path.join(ROOT, "hrl_pybullet_envs_b200", "libhrl_b200_chk.so")
SEED, NOISE_SEED, SIGMA = 11, 5, 0.3


def _members(D, H, A, P, seed=0):
    """P distinct policies as batched layers ((W1[P,H,D], b1[P,H]), (W2[P,H,H], b2[P,H]), (W3[P,A,H], b3[P,A]))."""
    g = torch.Generator().manual_seed(seed)

    def lin(o, i, s):
        return ((torch.rand(P, o, i, generator=g) * 2 - 1) * s).cuda(), ((torch.rand(P, o, generator=g) * 2 - 1) * 0.1).cuda()
    return (lin(H, D, 0.3), lin(H, H, 0.2), lin(A, H, 0.3))


def _member(layers, m):
    return tuple((W[m], b[m]) for W, b in layers)


def _first_episode(buf):
    """float32 return (sequential sum), length and finished flag of each env's first episode in a RolloutBuffer."""
    rew, done = buf.rew.cpu().numpy(), buf.done.cpu().numpy()
    T, N = rew.shape
    ret, length, fin = np.zeros(N, np.float32), np.zeros(N, np.int32), np.zeros(N, bool)
    for t in range(T):
        o = ~fin
        ret[o] = ret[o] + rew[t, o]
        length[o] += 1
        fin |= o & done[t]
    return ret, length, fin


def _assert_equal_results(got, want, what):
    ret, length, fin = (x.reshape(-1).cpu().numpy() for x in got)
    assert np.array_equal(ret.view(np.int32), want[0].view(np.int32)), (what, ret, want[0])
    assert np.array_equal(length, want[1]), (what, length, want[1])
    assert np.array_equal(fin, want[2]), (what, fin, want[2])


def _staggered(vec, mes):
    """Reset, then spread the envs over the episode clock (step count e % mes) so that one launch shorter than
    max_episode_steps leaves some envs finished and others not.  Returns the state."""
    vec.reset()
    f, i = vec.get_state()
    i[:, 0] = torch.arange(vec.N, device=i.device, dtype=torch.int32) % mes
    vec.set_state(f, i)
    return f, i


def _shard(env_id, M, m, state, mes, kw):
    from hrl_pybullet_envs_b200 import VecEnv
    s = VecEnv(env_id, M, seed=SEED, env_index_offset=m * M, max_episode_steps=mes, **kw)
    s.reset()
    f, i = state
    s.set_state(f[m * M:(m + 1) * M], i[m * M:(m + 1) * M])
    return s


SHARD_CASES = [("AntGatherBulletEnv-v0", {}), ("AntGatherBulletEnv-v0", dict(robot_coll_dist=0)),
               ("AntMazeBulletEnv-v0", dict(sense_target=True)), ("AntFlagrunBulletEnv-v0", dict(timeout=5)),
               ("AntMjBulletEnv-v0", {}), ("AntMazeMjEnv-v0", dict(n_bins=11)),
               ("PointGatherBulletEnv-v0", {}), ("PointGatherBulletEnv-v0", dict(use_sensor=False))]


@pytest.mark.parametrize("H", [32, 64])
@pytest.mark.parametrize("env_id,kw", SHARD_CASES)
def test_members_equal_their_shards(env_id, kw, H):
    """P = 4 members, M = 16 envs each (8 for PointGather, one CTA per member there): ret / length / finished equal the
    member's own rollout bit for bit, and the member's rows of the final state equal the shard's final state."""
    from hrl_pybullet_envs_b200 import VecEnv
    P, mes, T = 4, 7, 6
    M = 8 if env_id.startswith("Point") else 16
    vec = VecEnv(env_id, P * M, seed=SEED, max_episode_steps=mes, **kw)
    state = _staggered(vec, mes)
    layers = _members(vec.D, H, vec.A, P, seed=H)
    ret, length, fin = vec.evaluate_mlp(layers, T, sigma=SIGMA, noise_seed=NOISE_SEED)
    assert ret.shape == length.shape == fin.shape == (P, M)
    assert ret.dtype == torch.float32 and length.dtype == torch.int32 and fin.dtype == torch.bool
    f_end, i_end = vec.get_state()
    torch.cuda.synchronize()
    assert fin.any() and (~fin).any()
    for m in range(P):
        s = _shard(env_id, M, m, state, mes, kw)
        buf = s.rollout_mlp(_member(layers, m), T, sigma=SIGMA, noise_seed=NOISE_SEED)
        want = _first_episode(buf)
        _assert_equal_results((ret[m], length[m], fin[m]), want, (env_id, kw, H, m))
        fs, is_ = s.get_state()
        assert torch.equal(f_end[m * M:(m + 1) * M], fs) and torch.equal(i_end[m * M:(m + 1) * M], is_), (env_id, kw, H, m)
        s.close()
    # each CTA read its own member: the same envs under member 0's weights everywhere end in other states
    vec.set_state(*state)
    vec.evaluate_mlp(tuple((W[:1].expand_as(W).contiguous(), b[:1].expand_as(b).contiguous()) for W, b in layers), T,
                     sigma=SIGMA, noise_seed=NOISE_SEED)
    f_one = vec.get_state()[0]
    assert torch.equal(f_one[:M], f_end[:M])
    for m in range(1, P):
        assert not torch.equal(f_one[m * M:(m + 1) * M], f_end[m * M:(m + 1) * M]), m


def _sigma_cases(A):
    return [("scalar", SIGMA), ("per-component", torch.linspace(0.05, 0.6, A, device="cuda")), ("zero", 0.0)]


@pytest.mark.parametrize("env_id", ["AntGatherBulletEnv-v0", "AntFlagrunBulletEnv-v0", "PointGatherBulletEnv-v0"])
def test_one_policy_ragged_batch_equals_rollout(env_id):
    """P = 1 at N = 203 (a ragged last CTA for both kernels): scalar, per-component and zero sigma, and a normalized
    input whose clip binds, each equal to a rollout_mlp twin from the same state."""
    from hrl_pybullet_envs_b200 import RunningNormalizer, VecEnv
    N, mes, T = 203, 7, 6
    vec = VecEnv(env_id, N, seed=SEED, max_episode_steps=mes)
    twin = VecEnv(env_id, N, seed=SEED, max_episode_steps=mes)
    state = _staggered(vec, mes)
    twin.reset()
    norm = RunningNormalizer(vec, clip_obs=0.5)
    norm.update_obs(vec.observe())
    layers = _member(_members(vec.D, 64, vec.A, 1, seed=3), 0)
    cases = [(name, s, None) for name, s in _sigma_cases(vec.A)] + [("obs_norm", SIGMA, norm)]
    for name, sigma, on in cases:
        vec.set_state(*state); twin.set_state(*state)
        got = vec.evaluate_mlp(layers, T, sigma=sigma, noise_seed=NOISE_SEED, obs_norm=on)
        assert got[0].shape == (1, N)
        buf = twin.rollout_mlp(layers, T, sigma=sigma, noise_seed=NOISE_SEED, obs_norm=on)
        if on is not None:
            assert bool((norm.normalize(buf.obs[:-1]).abs() == 0.5).any())    # the clip binds
        _assert_equal_results(got, _first_episode(buf), (env_id, name))
        assert all(torch.equal(a, b) for a, b in zip(vec.get_state(), twin.get_state())), (env_id, name)


def test_full_size_population():
    """AntGather, 4096 envs, P = 256 members of 16 envs, T = max_episode_steps = 1000 from reset(): every env finishes;
    three sampled members equal their shards; two twins evaluated from identical states give identical bytes."""
    from hrl_pybullet_envs_b200 import VecEnv
    env_id, N, P, T = "AntGatherBulletEnv-v0", 4096, 256, 1000
    M = N // P
    a = VecEnv(env_id, N, seed=SEED, max_episode_steps=T)
    b = VecEnv(env_id, N, seed=SEED, max_episode_steps=T)
    a.reset(); b.reset()
    state = a.get_state()
    layers = _members(a.D, 64, a.A, P, seed=9)
    ra = a.evaluate_mlp(layers, T, sigma=SIGMA, noise_seed=NOISE_SEED)
    rb = b.evaluate_mlp(layers, T, sigma=SIGMA, noise_seed=NOISE_SEED)
    torch.cuda.synchronize()
    assert bool(ra[2].all())
    assert torch.equal(ra[0].view(torch.int32), rb[0].view(torch.int32)) and torch.equal(ra[1], rb[1]) and torch.equal(ra[2], rb[2])
    f_end = a.get_state()
    for m in (0, 101, 255):
        s = _shard(env_id, M, m, state, T, {})
        buf = s.rollout_mlp(_member(layers, m), T, sigma=SIGMA, noise_seed=NOISE_SEED)
        _assert_equal_results((ra[0][m], ra[1][m], ra[2][m]), _first_episode(buf), m)
        assert all(torch.equal(x[m * M:(m + 1) * M], y) for x, y in zip(f_end, s.get_state())), m
        s.close()


def test_argument_checks():
    from hrl_pybullet_envs_b200 import RunningNormalizer, VecEnv, _cabi
    ant = VecEnv("AntGatherBulletEnv-v0", 64, seed=1)
    pt = VecEnv("PointGatherBulletEnv-v0", 48, seed=1)
    ant.reset(); pt.reset()
    lay = _members(ant.D, 32, ant.A, 4)
    with pytest.raises(ValueError, match="multiple of the member count"):
        ant.evaluate_mlp(_members(ant.D, 32, ant.A, 3), 4)                  # 64 % 3
    with pytest.raises(ValueError, match="multiple of 16"):
        ant.evaluate_mlp(_members(ant.D, 32, ant.A, 8), 4)                  # M = 8
    with pytest.raises(ValueError, match="multiple of 8"):
        pt.evaluate_mlp(_members(pt.D, 32, pt.A, 12), 4)                    # M = 4
    pt.evaluate_mlp(_members(pt.D, 32, pt.A, 6), 2)                         # M = 8 is fine for PointGather
    bad = [((lay[0][0][..., :-1], lay[0][1]), lay[1], lay[2]),               # W1 one input short
           (lay[0], (lay[1][0], lay[1][1][:, :-1]), lay[2]),                 # b2 one unit short
           (lay[0], lay[1], (lay[2][0][:, :4], lay[2][1])),                  # W3 with 4 actions
           tuple((W[:, :16], b[:, :16]) for W, b in lay),                     # H = 16
           (lay[0], _member(lay, 0)[1], lay[2])]                             # one layer unbatched
    for layers in bad:
        with pytest.raises(ValueError, match="layers must be"):
            ant.evaluate_mlp(layers, 4)
    with pytest.raises(ValueError, match="sigma"):
        ant.evaluate_mlp(lay, 4, sigma=-0.1)
    with pytest.raises(ValueError, match="sigma"):
        ant.evaluate_mlp(lay, 4, sigma=torch.full((ant.A,), -0.1, device="cuda"))
    with pytest.raises(ValueError, match="sigma"):
        ant.evaluate_mlp(lay, 4, sigma=torch.full((3,), 0.1, device="cuda"))
    with pytest.raises(ValueError, match="obs_norm"):
        ant.evaluate_mlp(lay, 4, obs_norm=RunningNormalizer(pt))
    with pytest.raises(ValueError, match="horizon"):
        ant.evaluate_mlp(lay, 0)
    good = (torch.zeros(64, device="cuda"), torch.zeros(64, dtype=torch.int32, device="cuda"), torch.zeros(64, dtype=torch.bool, device="cuda"))
    ant.evaluate_mlp(lay, 2, out=good)
    ant.evaluate_mlp(lay, 2, out=tuple(t.view(4, 16) for t in good))
    for wrong in [(good[0].double(), good[1], good[2]), (good[0], good[1].long(), good[2]), (good[0], good[1], good[2].to(torch.uint8)),
                  (good[0][:32], good[1], good[2]), (good[0].view(8, 8), good[1], good[2]), (good[0].cpu(), good[1], good[2]),
                  (torch.zeros(128, device="cuda")[::2], good[1], good[2]), good[:2]]:
        with pytest.raises(ValueError, match="out must be"):
            ant.evaluate_mlp(lay, 2, out=wrong)
    # the raw C-ABI
    L = _cabi.lib()
    w = VecEnv.pack_mlp(lay).cuda()
    p = [C.c_void_p(t.data_ptr()) for t in good]
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    call = lambda T, P, ret, ln, fin: L.hrl_evaluate_mlp(ant.h, T, P, C.c_void_p(w.data_ptr()), 32, 0.0, None, 0, None, None,  # noqa: E731
                                                         0.0, ret, ln, fin, s)
    assert call(2, 4, *p) == 0
    assert call(2, 0, *p) == -1 and b"P must be >= 1" in L.hrl_last_error()
    assert call(2, -3, *p) == -1
    assert call(0, 4, *p) == -1 and b"T must be >= 1" in L.hrl_last_error()
    for k in range(3):
        q = list(p)
        q[k] = None
        assert call(2, 4, *q) == -1 and b"must all be given" in L.hrl_last_error()
    assert call(2, 3, *p) == -1 and b"multiple of the member count" in L.hrl_last_error()
    assert call(2, 8, *p) == -1 and b"multiple of 16" in L.hrl_last_error()
    torch.cuda.synchronize()


def test_cuda_graph_replay_equals_direct_call():
    """evaluate_mlp(out=...) captured in a CUDA graph and replayed writes the bytes a direct call writes from the same state."""
    from hrl_pybullet_envs_b200 import VecEnv
    N, P, T = 128, 8, 9
    a = VecEnv("AntFlagrunBulletEnv-v0", N, seed=SEED, max_episode_steps=7)
    b = VecEnv("AntFlagrunBulletEnv-v0", N, seed=SEED, max_episode_steps=7)
    a.reset(); b.reset()
    layers = _members(a.D, 64, a.A, P, seed=2)
    out = (torch.zeros(N, device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda"), torch.zeros(N, dtype=torch.bool, device="cuda"))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                      # warm-up outside the capture (advances a; b follows below)
        a.evaluate_mlp(layers, T, sigma=SIGMA, noise_seed=NOISE_SEED, out=out)
    torch.cuda.current_stream().wait_stream(side)
    b.evaluate_mlp(layers, T, sigma=SIGMA, noise_seed=NOISE_SEED)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        a.evaluate_mlp(layers, T, sigma=SIGMA, noise_seed=NOISE_SEED, out=out)
    for _ in range(2):
        out[0].fill_(-1.0)
        g.replay()
        want = b.evaluate_mlp(layers, T, sigma=SIGMA, noise_seed=NOISE_SEED)
        torch.cuda.synchronize()
        assert torch.equal(out[0].view(torch.int32), want[0].reshape(-1).view(torch.int32))
        assert torch.equal(out[1], want[1].reshape(-1)) and torch.equal(out[2], want[2].reshape(-1))
        assert all(torch.equal(x, y) for x, y in zip(a.get_state(), b.get_state()))


def test_bounds_checked_build_evaluates_clean():
    """tools/bounds_run_evaluate.py against libhrl_b200_chk.so: every family, both widths, P = 1 (ragged) and P = 4."""
    if not os.path.exists(CHK):
        pytest.skip("libhrl_b200_chk.so not built (__graft_entry__.build() makes it)")
    env = dict(os.environ, HRL_B200_LIB=CHK)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bounds_run_evaluate.py")], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert "bounds evaluate run complete" in r.stdout
    assert r.stdout.count("ok ") == 10 * 2 * 2     # 10 env cases x 2 widths x P in {1, 4}
