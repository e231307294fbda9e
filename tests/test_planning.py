"""greedy_lookahead's choice rule on the CPU: highest predicted reward, ties to the lowest k, NaN never over a number."""
import math

import torch

from wfcrl_b200.planning import greedy_lookahead


class _Env:
    """Stands in for a VecWindFarmEnv: evaluate_actions returns fixed rewards [B, K]."""

    device = torch.device("cpu")

    def __init__(self, reward, per_agent=False):
        self.reward = torch.tensor(reward, dtype=torch.float32)
        self.per_agent = per_agent

    def evaluate_actions(self, action):
        assert action.shape[:2] == self.reward.shape
        r = {"turbine_1": self.reward, "turbine_2": self.reward} if self.per_agent else self.reward
        return None, r, None, None, None


NAN = math.nan
REWARD = [[0.1, 0.3, 0.2], [0.5, 0.5, 0.4], [NAN, -1.0, NAN], [NAN, NAN, NAN], [0.2, NAN, 0.7]]


def test_choice_rule():
    cand = torch.arange(5 * 3 * 2, dtype=torch.float32).reshape(5, 3, 2)
    for per_agent in (False, True):
        action, reward, index = greedy_lookahead(_Env(REWARD, per_agent), cand)
        assert index.tolist() == [1, 0, 1, 0, 2]
        assert torch.equal(action, cand[torch.arange(5), index])
        expect = torch.tensor(REWARD, dtype=torch.float32)[torch.arange(5), index]
        assert torch.allclose(reward, expect, rtol=0, atol=0, equal_nan=True)
