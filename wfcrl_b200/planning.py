"""Greedy one-step lookahead: a reference policy to read RL results against, built on ``evaluate_actions``."""
from __future__ import annotations

import torch


def greedy_lookahead(env, candidates: torch.Tensor):
    """Evaluate the candidate actions ``candidates`` [B, K, T] of every env of the ``VecWindFarmEnv`` ``env`` (the joint
    form on a multi-agent env) and return ``(action [B, T], reward [B], index [B])``: per env the candidate of highest
    predicted reward, that reward and its index k.  Ties go to the lowest k; a NaN reward is never chosen over a finite
    one.  No host synchronisation; ``env`` does not change."""
    candidates = torch.as_tensor(candidates, dtype=torch.float32, device=env.device)
    reward = env.evaluate_actions(candidates)[1]
    if isinstance(reward, dict):  # multi-agent env: every agent gets the farm's reward
        reward = next(iter(reward.values()))
    # argmax returns the first of equal maxima; NaN ranks below every number
    index = torch.where(reward.isnan(), -torch.inf, reward).argmax(dim=1)
    action = candidates.gather(1, index[:, None, None].expand(-1, 1, candidates.shape[2]))[:, 0]
    return action, reward.gather(1, index[:, None])[:, 0], index
