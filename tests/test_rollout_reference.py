"""References of the fused rollout's policy contract (include/hrl_b200.h `hrl_rollout_mlp_ex` / `hrl_rollout_mlp_norm`)
without a GPU:

    act[t] = mlp(policy_input(obs[t])) + sigma * eps[t],   eps ~ N(0, 1), independent per env, step and component

- `philox4x32_10` / `eps_ref`: the counter RNG and the Box-Muller transform of the exploration noise, step by step as the
  kernels do them (hrl_math.cuh `rng_u4`, the noise blocks of `ant_env_kernel` and `point_env_kernel`).
- `mlp64`: the 3-layer tanh MLP in float64 on the float32 weights and the float32 policy input, with a per-component
  bound on how far a float32 evaluation can lie from it.

tests/test_gpu_rollout_reference.py holds every step of the kernels' actions to these references."""
import math

import numpy as np
import pytest

M32 = (1 << 32) - 1
U32 = 2.0 ** -24            # unit roundoff of float32
TANH_ULP = 2                # CUDA tanhf: at most 2 ulp from tanh of its argument (CUDA Math API, single precision)
STREAM_POLICY = 6           # hrl_b200.cu: the exploration-noise stream of the counter RNG


# ---- Philox4x32-10 and the noise ----------------------------------------------------------------------------------------
def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11) on uint32 arrays that broadcast: the round function of hrl_math.cuh."""
    c = [np.asarray(v, np.uint64) & M32 for v in (c0, c1, c2, c3)]
    k0, k1 = np.asarray(k0, np.uint64) & M32, np.asarray(k1, np.uint64) & M32
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & np.uint64(M32), p1 >> np.uint64(32), p1 & np.uint64(M32)
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & np.uint64(M32), (k1 + np.uint64(0xBB67AE85)) & np.uint64(M32)
    return [v.astype(np.uint32) for v in c]


def rng_u4(seed, env, stream, draw, sub):
    """hrl_math.cuh rng_u4: counter (draw, env, stream, sub), key (seed lo, seed hi); u_i = (o_i >> 8) * 2^-24 in float32."""
    o = philox4x32_10(draw, env, stream, sub, seed & M32, (seed >> 32) & M32)
    return [((v >> np.uint32(8)).astype(np.float32) * np.float32(U32)) for v in o]


def box_muller(u0, u1):
    """The kernels' transform of one draw: r = sqrtf(-2 logf(u0 + 2.98e-8f)), theta = 6.2831853f * u1 (both float32
    operations rounded as the kernel rounds them), then (r cos theta, r sin theta) in float64."""
    a = (np.float32(u0) + np.float32(2.98e-8)).astype(np.float32)
    theta = (np.float32(6.2831853) * np.float32(u1)).astype(np.float32).astype(np.float64)
    r = np.sqrt(-2.0 * np.log(a.astype(np.float64)))
    return r * np.cos(theta), r * np.sin(theta)


def eps_ref(seed, genv, draw, k):
    """Noise of global env `genv` at draw index `draw` (its SI_STEPS count before the step) for the pair k: the leg for
    an Ant (components 2k, 2k + 1), 0 for PointGather (x, y).  Arrays broadcast; returns (eps_2k, eps_2k+1) float64."""
    u = rng_u4(int(seed), genv, STREAM_POLICY, draw, k)
    return box_muller(u[0], u[1])


def eps_actions(seed, genv, draw, A):
    """eps [..., A] for envs `genv` [...] at draw indices `draw` [...]: the noise of every action component."""
    genv, draw = np.broadcast_arrays(np.asarray(genv, np.uint64), np.asarray(draw, np.uint64))
    out = np.empty(genv.shape + (A,))
    for k in range(A // 2):
        out[..., 2 * k], out[..., 2 * k + 1] = eps_ref(seed, genv, draw, k)
    return out


# ---- float64 MLP and its bound -------------------------------------------------------------------------------------------
def gamma(n):
    return n * U32 / (1 - n * U32)


def mlp64(layers, x):
    """layers ((W1[H, D], b1[H]), (W2[H, H], b2[H]), (W3[A, H], b3[A])) float32 (torch.nn.Linear layout), x float32
    [..., D].  Returns (y, bound, z3): the MLP in float64, the per-component bound on |y_f32 - y| of any float32
    evaluation that sums each pre-activation in some order with one rounding per addition (FMA or not) and takes tanhf
    of it, and the layer-3 pre-activations.

    Per layer, with x_hat the float32 input and e its bound: |z_hat - z| <= gamma(n + 1) (|b| + sum |W| (|x| + e)) +
    sum |W| e, n the fan-in; then |tanhf(z_hat) - tanh(z)| <= s dz + TANH_ULP 2^-23 (|y| + s dz), s = sech^2(max(|z| - dz, 0))
    the largest slope of tanh within dz of z (hrl_gae's S_t bound is built the same way)."""
    x = np.asarray(x, np.float32).astype(np.float64)
    e = np.zeros_like(x)
    for W, b in layers:
        W, b = np.asarray(W, np.float32).astype(np.float64), np.asarray(b, np.float32).astype(np.float64)
        aW = np.abs(W)
        z = x @ W.T + b
        ew = e @ aW.T
        dz = gamma(W.shape[1] + 1) * ((np.abs(x) + e) @ aW.T + np.abs(b)) + ew
        x = np.tanh(z)
        s = 1.0 / np.cosh(np.maximum(np.abs(z) - dz, 0.0)) ** 2
        e = s * dz + TANH_ULP * 2.0 ** -23 * (np.abs(x) + s * dz)
    return x, e, z


def action_tolerance(bound, act, sigma):
    """What |act - y - sigma eps_ref| may reach: the MLP bound, one rounding of the final addition (2^-24 |act|, doubled),
    and 1e-5 sigma for logf / sqrtf / sincosf / the products of the noise term (each a few ulp of |eps| <= 5.9)."""
    return bound + 2.0 ** -23 * np.abs(act) + 1e-5 * np.asarray(sigma, np.float64)


def fl32_mlp(layers, x, drop_b1=False):
    """A float32 evaluation in the kernel's order: fmaf chains from the bias (an exact float64 product plus one float64
    addition, rounded to float32), float32 tanh."""
    x = np.asarray(x, np.float32)
    for li, (W, b) in enumerate(layers):
        W, b = np.asarray(W, np.float32), np.asarray(b, np.float32)
        acc = np.broadcast_to(np.zeros_like(b) if (drop_b1 and li == 0) else b, x.shape[:-1] + b.shape).astype(np.float32)
        for j in range(W.shape[1]):
            acc = (x[..., j:j + 1].astype(np.float64) * W[:, j].astype(np.float64) + acc).astype(np.float32)
        x = np.tanh(acc).astype(np.float32)
    return x


def torch_like_layers(D, H, A, seed):
    """torch.nn.Linear's default initialisation, U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for weights and biases, float32."""
    rng = np.random.default_rng(seed)
    out = []
    for o, i in ((H, D), (H, H), (A, H)):
        s = 1.0 / math.sqrt(i)
        out.append((rng.uniform(-s, s, (o, i)).astype(np.float32), rng.uniform(-s, s, o).astype(np.float32)))
    return tuple(out)


# ---- known answers and hand-worked cases ---------------------------------------------------------------------------------
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((M32,) * 4, (M32, M32), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_matches_random123_known_answers(ctr, key, want):
    """The known-answer vectors of Random123 (kat_vectors, philox4x32_10)."""
    got = philox4x32_10(*ctr, *key)
    assert [int(v) for v in got] == list(want)


def test_philox_broadcasts_like_scalar_calls():
    draws = np.arange(5, dtype=np.uint32)
    vec = philox4x32_10(draws, 7, STREAM_POLICY, 3, 0x12345678, 0x9abcdef0)
    for i in range(5):
        one = philox4x32_10(int(draws[i]), 7, STREAM_POLICY, 3, 0x12345678, 0x9abcdef0)
        assert [int(v[i]) for v in vec] == [int(v) for v in one]


def test_rng_u4_addressing():
    """counter = (draw, env, stream, sub), key = (seed lo, seed hi), u = (o >> 8) 2^-24: exact multiples of 2^-24 in [0, 1)."""
    seed = (0xa4093822 << 32) | 0x299f31d0
    u = rng_u4(seed, 0x85a308d3, 0x13198a2e, 0x243f6a88, 0x03707344)
    o = philox4x32_10(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0x299f31d0, 0xa4093822)
    assert [float(v) for v in u] == [(int(w) >> 8) / 2.0 ** 24 for w in o]
    assert rng_u4(0, 0, 0, 0, 0)[0] == np.float32((0x6627e8d5 >> 8) / 2.0 ** 24)


def test_box_muller_hand_worked():
    """u0 = 1/2: 1/2 + 2.98e-8 rounds back to 1/2 in float32 (2.98e-8 is below half an ulp, 2^-25), r = sqrt(2 ln 2);
    u1 = 1/4: theta = fl32(6.2831853) / 4 = 1.5707963705062866, so cos theta = -4.371139e-8 and sin theta = 1 - 1e-15.
    u0 = 0: the guard keeps r finite, r = sqrt(-2 ln fl32(2.98e-8)) = sqrt(34.658) = 5.8871.  u0 = 1 - 2^-24 (the largest draw):
    u0 + 2.98e-8 rounds to u0, r = sqrt(-2 ln(1 - 2^-24)) = 3.4527e-4."""
    c, s = box_muller(np.float32(0.5), np.float32(0.25))
    r = math.sqrt(2 * math.log(2))
    assert abs(s - r * math.sin(1.5707963705062866)) < 1e-15 and abs(s - 1.1774100225154747) < 1e-14
    assert abs(c - r * -4.371139000186243e-08) < 1e-20
    c0, s0 = box_muller(np.float32(0.0), np.float32(0.0))
    assert abs(c0 - math.sqrt(-2 * math.log(float(np.float32(2.98e-8))))) < 1e-15 and abs(c0 - 5.88706) < 1e-5 and s0 == 0
    c1, _ = box_muller(np.float32(1 - 2.0 ** -24), np.float32(0.0))
    assert abs(c1 - math.sqrt(-2 * math.log1p(-2.0 ** -24))) < 1e-18 and abs(c1 - 3.4526698e-4) < 1e-10


def test_eps_ref_is_the_transform_of_the_addressed_draw():
    """eps_ref(seed, genv, draw, k) = box_muller of u0, u1 of the counter (draw, genv, 6, k); the pairs of an Ant go to
    components 2k, 2k + 1, and distinct envs, draws and legs read distinct counters."""
    seed = 0x0000000500000003
    u = rng_u4(seed, 11, STREAM_POLICY, 42, 3)
    assert eps_ref(seed, 11, 42, 3) == box_muller(u[0], u[1])
    e = eps_actions(seed, np.array([11, 12]), np.array([42, 42]), 8)
    assert e[0, 6] == eps_ref(seed, 11, 42, 3)[0] and e[0, 7] == eps_ref(seed, 11, 42, 3)[1]
    assert len(set(e.reshape(-1).tolist())) == 16
    assert eps_ref(seed, 11, 43, 3) != eps_ref(seed, 11, 42, 3)


def test_eps_ref_moments():
    """N(0, 1) per component, no correlation between the pair's two components or between neighbouring draws."""
    draws = np.arange(200000, dtype=np.uint64)
    c, s = eps_ref(17, 5, draws, 2)
    for v in (c, s):
        assert abs(v.mean()) < 0.01 and abs(v.std() - 1) < 0.01
    assert abs(np.corrcoef(c, s)[0, 1]) < 0.01 and abs(np.corrcoef(c[1:], c[:-1])[0, 1]) < 0.01


def test_mlp_bound_hand_worked():
    """One unit per layer, W = 1, b = 0, x = 1/2.  Layer 1: z = 1/2, dz = gamma(2) / 2, y = tanh(1/2),
    s = sech^2(1/2 - dz), e1 = s dz + 2^-22 (y + s dz).  Layer 2: z = y, dz = gamma(2) (y + e1) + e1, and so on."""
    one = (np.ones((1, 1), np.float32), np.zeros(1, np.float32))
    y, e, z = mlp64((one, one, one), np.array([0.5], np.float32))
    g2 = 2 * U32 / (1 - 2 * U32)
    xv, ev = 0.5, 0.0
    for _ in range(3):
        dz = g2 * (xv + ev) + ev
        zv = xv
        xv = math.tanh(zv)
        s = 1 / math.cosh(zv - dz) ** 2
        ev = s * dz + 2.0 ** -22 * (xv + s * dz)
    assert abs(z[0] - math.tanh(math.tanh(0.5))) < 1e-16
    assert abs(y[0] - math.tanh(math.tanh(math.tanh(0.5)))) < 1e-16
    assert abs(e[0] - ev) <= 1e-12 * ev
    # the numbers: about 1.7e-7 after layer 1 and 3.9e-7 after layer 3 (tanhf's 2 ulp dominate; each tanh shrinks the rest)
    assert 3.5e-7 < e[0] < 4.5e-7


def test_mlp_bound_holds_and_is_tight_enough():
    """A float32 evaluation in the kernel's order stays inside the bound at the widest observation (D = 64) and both hidden
    widths, with inputs up to 15 in magnitude, and the bound is small enough to catch a dropped first-layer bias in 95 % of
    the components.  The bound is the worst case of each summation (gamma(n) times the sum of magnitudes), so it lies
    two to three orders of magnitude above the error a real evaluation makes."""
    rng = np.random.default_rng(0)
    for D, H, A in ((64, 64, 8), (29, 32, 8), (28, 64, 2)):
        layers = torch_like_layers(D, H, A, seed=D + H)
        x = (rng.normal(0, 1, (512, D)) * rng.uniform(0.1, 5, D)).astype(np.float32)
        y, bound, z3 = mlp64(layers, x)
        err = np.abs(fl32_mlp(layers, x) - y)
        assert (err <= bound).all(), (err / bound).max()
        assert bound.max() < 1e-3 and (np.abs(z3) < 1).mean() > 0.5
        assert (np.abs(fl32_mlp(layers, x, drop_b1=True) - y) > bound).mean() > 0.95


def test_action_tolerance_terms():
    b = np.array([1e-6, 1e-6])
    t = action_tolerance(b, np.array([0.5, -3.0]), np.array([0.0, 0.5]))
    assert t[0] == 1e-6 + 2.0 ** -24 and t[1] == 1e-6 + 3 * 2.0 ** -23 + 5e-6
