"""Batched VecEnv.pack_mlp (the [P, nw] weights of hrl_evaluate_mlp) on CPU tensors: row m is member m's packed vector."""
import pytest

torch = pytest.importorskip("torch")

from hrl_pybullet_envs_b200.vec_env import VecEnv  # noqa: E402


@pytest.mark.parametrize("D,H,A,P", [(46, 64, 8, 5), (28, 32, 2, 3), (63, 32, 8, 1)])
def test_batched_pack_is_the_stack_of_member_packs(D, H, A, P):
    g = torch.Generator().manual_seed(D + H + P)
    layers = tuple((torch.randn(P, o, i, generator=g), torch.randn(P, o, generator=g)) for o, i in ((H, D), (H, H), (A, H)))
    packed = VecEnv.pack_mlp(layers)
    nw = D * H + H + H * H + H + H * A + A
    assert packed.shape == (P, nw) and packed.dtype == torch.float32 and packed.is_contiguous()
    for m in range(P):
        member = tuple((W[m], b[m]) for W, b in layers)
        assert torch.equal(packed[m], VecEnv.pack_mlp(member))


def test_unbatched_pack_keeps_its_layout():
    g = torch.Generator().manual_seed(0)
    (W1, b1), (W2, b2), (W3, b3) = layers = tuple((torch.randn(o, i, generator=g), torch.randn(o, generator=g))
                                                  for o, i in ((32, 10), (32, 32), (8, 32)))
    packed = VecEnv.pack_mlp(layers)
    assert packed.shape == (10 * 32 + 32 + 32 * 32 + 32 + 32 * 8 + 8,)
    assert torch.equal(packed, torch.cat([W1.t().reshape(-1), b1, W2.t().reshape(-1), b2, W3.t().reshape(-1), b3]))
