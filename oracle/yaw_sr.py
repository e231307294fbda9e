"""Restatement of ``wfcrl_b200.yaw_optimization.serial_refine`` on the C oracle (TEST INFRASTRUCTURE ONLY).

The same schedule, written independently in numpy over ``c_oracle.solve_batch``: start at yaw 0 clipped into the bounds;
pass p runs T stages, stage r varies the turbine at sorted position r (upstream first) over ``linspace(lo, hi, N0)`` in pass 0
and over ``clip(y* + s_(p-1) * linspace(-1, 1, Np), lo, hi)`` afterwards (s0 = (hi - lo) / (N0 - 1), s_p = 2 s_(p-1) / (Np - 1));
the candidate of highest farm power (the float64 sum of the per-turbine powers in original turbine order, left to right;
ties: the lowest index) replaces the current yaw only when its power is strictly greater.

Besides the result it records, per env, every choice made and the smallest relative gap of a decision: between the winner
and the best candidate of a different yaw value, and between the winner and the current power when the winner's yaw differs
from the current one.  Envs whose smallest gap is below the solver's precision can legitimately choose differently.
"""
from __future__ import annotations

import numpy as np

from oracle import c_oracle


def farm_power(power_w: np.ndarray) -> np.ndarray:
    return np.add.accumulate(power_w, axis=-1)[..., -1]  # left to right


def serial_refine(layout_x, layout_y, ws, wd, passes=(5, 5, 5), bounds=(-40.0, 40.0), ti_ambient=0.06):
    lx = np.asarray(layout_x, dtype=np.float64)
    ly = np.asarray(layout_y, dtype=np.float64)
    ws = np.atleast_1d(np.asarray(ws, dtype=np.float64))
    wd = np.atleast_1d(np.asarray(wd, dtype=np.float64))
    B, T = ws.shape[0], lx.shape[0]
    lo, hi = float(bounds[0]), float(bounds[1])
    dev = (((wd % 360.0) - 270.0) % 360.0 + 360.0) % 360.0
    cs = np.stack([np.cos(np.radians(dev)), np.sin(np.radians(dev))], 1)

    def solve(yaw):  # yaw [B, K, T] -> per-turbine power [B, K, T], sorted order of each env
        K = yaw.shape[1]
        out = c_oracle.solve_batch(lx, ly, np.repeat(ws, K), np.repeat(wd, K), yaw.reshape(B * K, T),
                                   cs=np.repeat(cs, K, axis=0), ti_ambient=ti_ambient)
        return out["power_W"].reshape(B, K, T), out["order"].reshape(B, K, T)[:, 0]

    yaw = np.full((B, T), min(max(0.0, lo), hi))
    p0, order = solve(yaw[:, None, :])
    cur = farm_power(p0[:, 0])
    start = cur.copy()
    min_gap = np.full(B, np.inf)
    choices = []
    spacing = 0.0
    for p, n in enumerate(passes):
        if p == 0:
            grid = np.linspace(lo, hi, n)
            spacing = (hi - lo) / (n - 1)
        else:
            offset = spacing * np.linspace(-1.0, 1.0, n)
            spacing = 2.0 * spacing / (n - 1)
        for r in range(T):
            tid = order[:, r]
            ystar = yaw[np.arange(B), tid]
            vals = np.broadcast_to(grid, (B, n)).copy() if p == 0 else np.clip(ystar[:, None] + offset[None, :], lo, hi)
            cand = np.repeat(yaw[:, None, :], n, axis=1)
            cand[np.arange(B), :, tid] = vals
            fp = farm_power(solve(cand)[0])
            best = np.argmax(fp, axis=1)
            bp = fp[np.arange(B), best]
            bv = vals[np.arange(B), best]
            for b in range(B):
                other = fp[b][vals[b] != bv[b]]
                scale = max(abs(bp[b]), 1.0)
                if other.size:
                    min_gap[b] = min(min_gap[b], (bp[b] - other.max()) / scale)
                if bv[b] != ystar[b]:
                    min_gap[b] = min(min_gap[b], abs(bp[b] - cur[b]) / scale)
            better = bp > cur
            yaw[np.arange(B), tid] = np.where(better, bv, ystar)
            cur = np.where(better, bp, cur)
            choices.append(np.where(better, best, -1))
    return {"yaw": yaw, "farm_power": cur, "start_power": start, "min_gap": min_gap, "choices": np.stack(choices, 1)}
