"""Batched static yaw optimisation: which yaw setting maximises farm power in each env's current wind?

``serial_refine`` optimises every env of a batch at once with the candidate evaluation of the library
(``FlorisBatch.evaluate_yaw``, one launch per stage, no state change).  It is the reference point RL results on these envs are
read against (and against zero yaw).  The schedule is this project's own serial-refine search, in the spirit of FLORIS'
``YawOptimizationSR``; it is not claimed to reproduce FLORIS' optimiser digit for digit:

1. start at yaw 0 clipped into the bounds, evaluated with K = 1 for the current farm power;
2. pass p runs T stages; stage r varies, in every env at once, the turbine at sorted position r of the env's geometry
   (state ``order``, upstream first) with the others held; in an env of n <= r turbines every candidate is its current yaw;
3. pass 0 tries ``linspace(lo, hi, N0)`` (spacing s0 = (hi - lo) / (N0 - 1)); pass p >= 1 tries
   ``y* + s_(p-1) * linspace(-1, 1, Np)`` clipped to the bounds, y* the current value, and has spacing s_p = 2 s_(p-1) / (Np - 1);
4. the candidate of highest farm power wins (ties: the lowest candidate index) and replaces the current yaw only if its
   power is strictly greater than the current farm power, so the result is monotone by construction.

Farm power is the float64 sum of the per-turbine powers over the env's turbines, left to right in the original turbine order
(``farm_power``).  The stage loop never synchronises with the host.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from .backend import FlorisBatch


def farm_power(power: torch.Tensor) -> torch.Tensor:
    """Float64 farm power of per-turbine powers [..., T]: their sum from column 0 to T-1, one column at a time, so that the
    result of an env does not depend on the batch around it.  Padding columns hold 0 and add nothing."""
    p = power.to(torch.float64)
    acc = p[..., 0].clone()
    for t in range(1, p.shape[-1]):
        acc = acc + p[..., t]
    return acc


def _check_passes(passes) -> tuple:
    try:
        passes = tuple(int(n) for n in passes)
    except TypeError:
        raise TypeError("passes must be a sequence of candidate counts, e.g. (5, 5, 5)") from None
    if not passes or any(n < 2 for n in passes):
        raise ValueError(f"passes must be a non-empty sequence of candidate counts >= 2, got {passes}")
    return passes


def _check_bounds(bounds) -> tuple:
    lo, hi = (float(v) for v in bounds)
    if not (math.isfinite(lo) and math.isfinite(hi) and lo < hi):
        raise ValueError(f"bounds must be finite with low < high, got {(lo, hi)}")
    return lo, hi


def serial_refine(env, passes: Sequence[int] = (5, 5, 5), bounds: Optional[Sequence[float]] = None) -> Dict:
    """Serial-refine yaw optimisation of every env of ``env`` (a ``VecWindFarmEnv``, through ``env.backend``, or a
    ``FlorisBatch``) in its current wind, TI and layout; ``passes`` = candidates per stage of each pass, ``bounds`` =
    (low, high) in degrees, default the env's yaw control bounds.  Nothing of the env's state changes.

    Returns ``{"yaw": float64 [B, T]`` (original turbine order, padding columns 0), ``"farm_power": [B]`` (W, float64, of
    that yaw), ``"start_power": [B]`` (of the start yaw), ``"evaluations": int`` (candidate solves per env,
    1 + T * sum(passes))}."""
    passes = _check_passes(passes)
    if bounds is not None:
        bounds = _check_bounds(bounds)
    fb = getattr(env, "backend", env)
    if not isinstance(fb, FlorisBatch):
        raise TypeError("env must be a VecWindFarmEnv or a FlorisBatch")
    lo, hi = bounds if bounds is not None else _check_bounds((fb.cfg.yaw_lo, fb.cfg.yaw_hi))
    B, T, dev = fb.B, fb.T, fb.device
    counts = torch.as_tensor(fb.get_state("turbine_count").astype(np.int64), device=dev)
    order = torch.as_tensor(fb.get_state("order").astype(np.int64), device=dev)  # sorted position -> original index
    rows = torch.arange(B, device=dev)
    valid = torch.arange(T, device=dev)[None, :] < counts[:, None]
    yaw = torch.full((B, T), min(max(0.0, lo), hi), dtype=torch.float64, device=dev).masked_fill_(~valid, 0.0)

    kmax = max(passes)
    if fb.eval_capacity < kmax:  # size the evaluation buffers now, so that no call of the stage loop allocates (and syncs)
        fb.evaluate_yaw(yaw[:, None, :].expand(B, kmax, T).contiguous())
    cur = farm_power(fb.evaluate_yaw(yaw[:, None, :].contiguous())["power"][:, 0])
    start = cur.clone()
    evaluations = 1

    spacing = 0.0
    for p, n_cand in enumerate(passes):
        # candidate grids on the host in float64 (numpy), so that they are the same numbers in any restatement
        if p == 0:
            grid = torch.as_tensor(np.linspace(lo, hi, n_cand), device=dev)[None, :].expand(B, n_cand)
            spacing = (hi - lo) / (n_cand - 1)
        else:
            offset = torch.as_tensor(spacing * np.linspace(-1.0, 1.0, n_cand), device=dev)[None, :]
            spacing = 2.0 * spacing / (n_cand - 1)
        for r in range(T):
            tid = order[:, r]
            ystar = yaw[rows, tid]
            vals = grid if p == 0 else (ystar[:, None] + offset).clamp(lo, hi)
            vals = torch.where((r < counts)[:, None], vals, ystar[:, None])
            cand = yaw[:, None, :].repeat(1, n_cand, 1)
            cand.scatter_(2, tid[:, None, None].expand(B, n_cand, 1), vals[:, :, None])
            fp = farm_power(fb.evaluate_yaw(cand)["power"])
            best = fp.argmax(dim=1)  # the first maximum: ties go to the lowest candidate index
            best_p = fp[rows, best]
            better = best_p > cur
            yaw[rows, tid] = torch.where(better, vals[rows, best], ystar)
            cur = torch.where(better, best_p, cur)
            evaluations += n_cand
    return {"yaw": yaw, "farm_power": cur, "start_power": start, "evaluations": evaluations}
