"""Reference planners to read RL results against: greedy one-step lookahead on ``evaluate_actions``, and open-loop H-step
planning on ``evaluate_rollouts`` (best of given sequences, and the cross-entropy method).  None synchronises with the host
and none changes the env."""
from __future__ import annotations

from typing import Optional

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


def _returns(env, sequences: torch.Tensor, gamma: float) -> torch.Tensor:
    """float64 [B, K]: per candidate sequence, the sum over its valid rows (up to and including its truncating step) of
    gamma**h * reward, accumulated in h order."""
    _obs, reward, _term, _trunc, info = env.evaluate_rollouts(sequences, observations=False)
    if isinstance(reward, dict):  # multi-agent env: every agent gets the farm's reward
        agent = next(iter(reward))
        reward, info = reward[agent], info[agent]
    reward, valid = reward.double(), info["valid"]
    ret = torch.zeros(reward.shape[:2], dtype=torch.float64, device=reward.device)
    for h in range(reward.shape[2]):
        ret = ret + torch.where(valid[:, :, h], (gamma ** h) * reward[:, :, h], 0.0)
    return ret


def _rank(ret: torch.Tensor) -> torch.Tensor:
    """``ret`` with NaN below every number, for argmax / topk."""
    return torch.where(ret.isnan(), -torch.inf, ret)


def best_sequence(env, sequences: torch.Tensor, gamma: float = 1.0):
    """The H-step analogue of ``greedy_lookahead``: evaluate the K candidate action sequences ``sequences`` [B, K, H, T]
    of every env of ``env`` (open loop, ``evaluate_rollouts``) and return ``(action [B, T], return [B], index [B])``: per
    env the first action of the sequence of highest discounted return (float64 sum of gamma**h * reward over the rows up
    to and including its truncating step), that return and its index k.  Ties go to the lowest k; a NaN return is never
    chosen over a number."""
    sequences = torch.as_tensor(sequences, dtype=torch.float32, device=env.device)
    ret = _returns(env, sequences, gamma)
    index = _rank(ret).argmax(dim=1)
    best = sequences[torch.arange(sequences.shape[0], device=sequences.device), index]
    return best[:, 0], ret.gather(1, index[:, None])[:, 0], index


def cem_plan(env, horizon: int, samples: int, iterations: int = 3, elites: Optional[int] = None, gamma: float = 1.0,
             generator: Optional[torch.Generator] = None):
    """Cross-entropy method over continuous action sequences of ``horizon`` steps for every env of ``env``.

    Iteration 0 draws ``samples`` sequences per env from N(0, yaw_step) clipped to +-yaw_step, the first of them the
    all-zero sequence; every iteration evaluates its sequences (``evaluate_rollouts``, discounted return as
    ``best_sequence``) and refits the per-(h, t) mean and standard deviation of the next draw to its ``elites`` best
    (default samples // 8, at least 1), ``iterations`` times.  The best sequence so far is replaced only by one of
    strictly greater return, so the result never falls below the all-zero sequence.  Returns ``(action [B, T], return
    [B], sequence [B, H, T])``; the return is NaN only where every sequence evaluated had a NaN return.  Draws from ``generator`` (a ``torch.Generator`` on the env's device) when given: a seeded call is reproducible."""
    if not env.continuous_control:
        raise ValueError("cem_plan samples continuous actions; this env has discrete control")
    if horizon < 1:
        raise ValueError(f"horizon must be >= 1, got {horizon}")
    if samples < 1:
        raise ValueError(f"samples must be >= 1, got {samples}")
    if iterations < 1:
        raise ValueError(f"iterations must be >= 1, got {iterations}")
    elites = max(1, samples // 8) if elites is None else int(elites)
    if not 1 <= elites <= samples:
        raise ValueError(f"elites must be in [1, samples = {samples}], got {elites}")
    B, T, step = env.num_envs, env.num_turbines, float(env.controls["yaw"][2])
    shape = (B, horizon, T)
    mean = torch.zeros(shape, dtype=torch.float32, device=env.device)
    std = torch.full(shape, step, dtype=torch.float32, device=env.device)
    best_score = torch.full((B,), -torch.inf, dtype=torch.float64, device=env.device)  # best return, NaN ranked lowest
    best_ret = torch.full((B,), torch.nan, dtype=torch.float64, device=env.device)  # ... and that return as evaluated
    best_seq = torch.zeros(shape, dtype=torch.float32, device=env.device)
    rows = torch.arange(B, device=env.device)
    for it in range(iterations):
        noise = torch.randn((B, samples) + shape[1:], generator=generator, device=env.device)
        seq = (mean[:, None] + std[:, None] * noise).clamp_(-step, step)
        if it == 0:
            seq[:, 0] = 0.0
        ret = _returns(env, seq.contiguous(), gamma)
        top = _rank(ret).topk(elites, dim=1)
        # iteration 0 always takes its best, the all-zero sequence or better (a NaN return only when every one is NaN)
        better = (top.values[:, 0] > best_score) | (it == 0)
        best_score = torch.where(better, top.values[:, 0], best_score)
        best_ret = torch.where(better, ret.gather(1, top.indices[:, :1])[:, 0], best_ret)
        best_seq = torch.where(better[:, None, None], seq[rows, top.indices[:, 0]], best_seq)
        elite = seq[rows[:, None], top.indices]  # [B, elites, H, T]
        mean, std = elite.mean(dim=1), elite.std(dim=1, unbiased=False)
    return best_seq[:, 0], best_ret, best_seq
