"""Candidate evaluation (wf_evaluate_yaw) against interface-mode solves, and the serial-refine optimiser, on HornsRev1 x 8192
envs in strict FP32, relaxed FP32 and FP64.  Writes profiles/evaluate_yaw_bench.json (or --out).

Per precision:
  - one evaluate_yaw call of K = 5 U(-40, 40) candidates per env, and the K interface-mode calls (update_command with
    candidate k) that solve the same B*K yaw settings, alternated, each timed with CUDA events after the L2 is overwritten;
  - candidate solves per second of the evaluation, env solves per second of interface mode, and their ratio;
  - wall time of serial_refine with passes (5, 5, 5) and its evaluation count;
and the relative gap of the strict FP32 optimum, evaluated in FP64, to the FP64 optimum.  Card name and power limit are read
in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from wfcrl_b200.backend import FlorisBatch  # noqa: E402
from wfcrl_b200.layouts import get_layout  # noqa: E402
from wfcrl_b200.yaw_optimization import farm_power, serial_refine  # noqa: E402

MODES = {"f32_strict": ("f32", True), "f32_relaxed": ("f32", False), "f64": ("f64", True)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--K", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "evaluate_yaw_bench.json"))
    args = ap.parse_args()
    case = get_layout("HornsRev1_")
    lx, ly = np.asarray(case["xcoords"]), np.asarray(case["ycoords"])
    B, K, T = args.envs, args.K, len(lx)
    rng = np.random.default_rng(0)
    ws = np.clip(8 * rng.weibull(8, B), 3, 28)
    wd = np.clip(rng.normal(270, 20, B) % 360, 0, 360)
    yaw = torch.as_tensor(rng.uniform(-40, 40, (B, K, T)), device="cuda")
    cols = [yaw[:, k].contiguous() for k in range(K)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # 256 MB > the 126 MB of L2
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    res = {"card": card(), "layout": "HornsRev1_", "envs": B, "turbines": T, "K": K, "reps": args.reps,
           "l2": "overwritten (256 MB) before every timed call", "modes": {}}
    handles, optima = {}, {}
    for mode, (precision, strict) in MODES.items():
        fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=10**9, strict=strict)
        fb.reset(ws, wd, host_trig=True)
        handles[mode] = fb

        def timed(fn):
            flush.zero_()
            ev[0].record()
            fn()
            ev[1].record()
            torch.cuda.synchronize()
            return ev[0].elapsed_time(ev[1])

        def interface():
            for c in cols:
                fb.update_command(c)

        for _ in range(2):  # warm-up of both shapes
            fb.evaluate_yaw(yaw)
            interface()
        t_eval, t_if = [], []
        for _ in range(args.reps):
            t_eval.append(timed(lambda: fb.evaluate_yaw(yaw)))
            t_if.append(timed(interface))
        me, mi = float(np.median(t_eval)), float(np.median(t_if))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt = serial_refine(fb, passes=(5, 5, 5))
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        optima[mode] = opt
        res["modes"][mode] = {
            "evaluate_ms": {"median": me, "min": float(np.min(t_eval)), "max": float(np.max(t_eval))},
            "interface_K_calls_ms": {"median": mi, "min": float(np.min(t_if)), "max": float(np.max(t_if))},
            "candidate_solves_per_s": B * K / (me * 1e-3),
            "interface_env_solves_per_s": B * K / (mi * 1e-3),
            "ratio": mi / me,
            "serial_refine_555": {"wall_s": wall, "evaluations_per_env": opt["evaluations"],
                                  "mean_gain_rel": float(((opt["farm_power"] - opt["start_power"]) /
                                                          opt["start_power"]).mean())},
        }
        print(mode, json.dumps(res["modes"][mode]), flush=True)
    # the strict FP32 optimum judged in FP64
    fb64 = handles["f64"]
    p32 = farm_power(fb64.evaluate_yaw(optima["f32_strict"]["yaw"][:, None, :].contiguous())["power"][:, 0])
    gap = ((optima["f64"]["farm_power"] - p32) / optima["f64"]["farm_power"]).cpu().numpy()
    below_zero = ((optima["f64"]["start_power"] - p32) / optima["f64"]["start_power"]).cpu().numpy()
    res["f32_strict_vs_f64_optimum"] = {
        "rel_gap_quantiles": {q: float(np.quantile(gap, float(q))) for q in ("0", "0.5", "0.9", "0.99", "1")},
        "share_equal_or_better": float((gap <= 0).mean()),
        "max_rel_shortfall_vs_f64_zero_yaw": float(below_zero.max()),
    }
    print(json.dumps(res["f32_strict_vs_f64_optimum"]))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fp:
        json.dump(res, fp, indent=1)
    for fb in handles.values():
        fb.close()


if __name__ == "__main__":
    main()
