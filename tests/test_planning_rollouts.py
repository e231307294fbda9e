"""best_sequence's choice rule and cem_plan's argument checks on the CPU, against a stand-in env: discounted float64 returns
over the valid rows, ties to the lowest k, NaN never over a number."""
import math

import pytest
import torch

from wfcrl_b200.planning import best_sequence, cem_plan

NAN = math.nan


class _Env:
    """Stands in for a VecWindFarmEnv: evaluate_rollouts returns fixed rewards and valid masks [B, K, H]."""

    device = torch.device("cpu")
    num_envs, num_turbines = 4, 2
    controls = {"yaw": (-40, 40, 5)}

    def __init__(self, reward=None, valid=None, per_agent=False, continuous_control=True):
        self.reward = None if reward is None else torch.tensor(reward, dtype=torch.float32)
        self.valid = None if valid is None else torch.tensor(valid, dtype=torch.bool)
        self.per_agent = per_agent
        self.continuous_control = continuous_control

    def evaluate_rollouts(self, actions, observations=True):
        assert actions.shape[:3] == self.reward.shape and not observations
        info = {"valid": self.valid, "power": None, "load": None}
        if self.per_agent:
            return None, {"turbine_1": self.reward, "turbine_2": self.reward}, None, None, \
                {"turbine_1": info, "turbine_2": info}
        return None, self.reward, None, None, info


T_, F_ = True, False
# [B = 4][K = 3][H = 3]
REWARD = [
    [[1.0, 1.0, 1.0], [0.0, 0.0, 4.0], [2.0, 0.5, 0.0]],  # discounting decides
    [[1.0, 2.0, 9.0], [1.0, 2.0, 3.0], [0.5, 0.5, 0.5]],  # the 9.0 lies after a truncation: not counted
    [[NAN, 1.0, 1.0], [1.0, 1.0, 0.0], [2.0, 0.0, 0.0]],  # NaN return loses; rows 1, 2 tie (2.0 at gamma 1)
    [[NAN, NAN, NAN], [NAN, 0.0, 0.0], [NAN, 1.0, 1.0]],  # every return NaN: index 0
]
VALID = [
    [[T_, T_, T_], [T_, T_, T_], [T_, T_, T_]],
    [[T_, T_, F_], [T_, T_, T_], [T_, T_, T_]],
    [[T_, T_, T_], [T_, T_, T_], [T_, T_, T_]],
    [[T_, T_, T_], [T_, T_, T_], [T_, T_, T_]],
]


def _expected(gamma):
    r = torch.tensor(REWARD, dtype=torch.float64)
    ret = torch.zeros(4, 3, dtype=torch.float64)
    for h in range(3):
        ret = ret + torch.where(torch.tensor(VALID)[:, :, h], (gamma ** h) * r[:, :, h], 0.0)
    return ret


@pytest.mark.parametrize("per_agent", [False, True])
@pytest.mark.parametrize("gamma, index", [(1.0, [1, 1, 1, 0]), (0.5, [2, 1, 2, 0])])
def test_best_sequence_choice_rule(per_agent, gamma, index):
    seq = torch.arange(4 * 3 * 3 * 2, dtype=torch.float32).reshape(4, 3, 3, 2)
    action, ret, idx = best_sequence(_Env(REWARD, VALID, per_agent), seq, gamma=gamma)
    assert idx.tolist() == index
    assert ret.dtype == torch.float64
    assert torch.equal(action, seq[torch.arange(4), idx, 0])
    expect = _expected(gamma)[torch.arange(4), idx]
    assert torch.allclose(ret, expect, rtol=0, atol=0, equal_nan=True)
    if gamma == 1.0:  # env 1: 1 + 2 + 3 beats 1 + 2 (+ 9 after the truncation); env 0: 4.0 beats 3.0
        assert ret[:2].tolist() == [4.0, 6.0]


def test_cem_plan_refusals():
    env = _Env()
    with pytest.raises(ValueError, match="discrete"):
        cem_plan(_Env(continuous_control=False), horizon=2, samples=8)
    for horizon in (0, -1):
        with pytest.raises(ValueError, match="horizon"):
            cem_plan(env, horizon=horizon, samples=8)
    for iterations in (0, -1):
        with pytest.raises(ValueError, match="iterations"):
            cem_plan(env, horizon=2, samples=8, iterations=iterations)
    for elites in (0, -2, 9):
        with pytest.raises(ValueError, match="elites"):
            cem_plan(env, horizon=2, samples=8, elites=elites)


def test_cem_plan_all_nan_returns_nan():
    """Where every sequence's return is NaN, the return reported is NaN (what an evaluation of the sequence gives)."""
    nan = [[[NAN, NAN]] * 4] * 4  # [B = 4][samples = 4][horizon = 2]
    valid = [[[True, True]] * 4] * 4
    gen = torch.Generator().manual_seed(0)
    action, ret, seq = cem_plan(_Env(nan, valid), horizon=2, samples=4, iterations=2, generator=gen)
    assert bool(ret.isnan().all()) and action.shape == (4, 2) and seq.shape == (4, 2, 2)
