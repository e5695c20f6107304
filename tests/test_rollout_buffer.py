"""Host-side logic of RolloutBuffer's training fields (no GPU: the buffer is built on the CPU from a stand-in env)."""
from types import SimpleNamespace

import pytest

torch = pytest.importorskip("torch")

from hrl_pybullet_envs_b200 import config as K  # noqa: E402
from hrl_pybullet_envs_b200.vec_env import RolloutBuffer  # noqa: E402


def _env(kind=K.HRL_ANT_FLAGRUN):
    return SimpleNamespace(device=torch.device("cpu"), N=3, D=5, A=8, kind=kind)


def test_buffer_fields_follow_the_flags():
    b = RolloutBuffer(_env(), 4)
    assert b.info is None and b.terminal_obs is None
    with pytest.raises(ValueError):
        b.truncated
    with pytest.raises(ValueError):
        b.infos(0)
    b = RolloutBuffer(_env(), 4, info=True, terminal_obs=True)
    assert b.info.shape == (4, 3, 4) and b.info.dtype == torch.float32
    assert b.terminal_obs.shape == (4, 3, 5) and b.terminal_obs.dtype == torch.float32


def test_truncated_and_infos_read_the_step_info_columns():
    b = RolloutBuffer(_env(), 2, info=True, terminal_obs=True)
    b.info[1, :, 2] = torch.tensor([0.0, 1.0, 3.0])      # flag bits: 1 = TimeLimit.truncated, 2 = Flagrun goal switched
    b.info[1, :, 1] = torch.tensor([7.0, 6.0, 5.0])
    b.terminal_obs[1, 2] = 9.0
    assert b.truncated.tolist() == [[False] * 3, [False, True, True]]
    i = b.infos(1)
    assert i["TimeLimit.truncated"].tolist() == [False, True, True]
    assert i["target_switched"].tolist() == [False, False, True]
    assert i["goals_left"].tolist() == [7.0, 6.0, 5.0]
    assert torch.equal(i["terminal_obs"][2], torch.full((5,), 9.0))
    assert "target" not in i                              # the current goal is not step t's: not offered for a past step
    assert "terminal_obs" not in RolloutBuffer(_env(K.HRL_POINT_GATHER), 1, info=True).infos(0)
