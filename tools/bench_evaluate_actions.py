"""Action evaluation (wf_evaluate_actions) against stepping, on HornsRev1 x 8192 envs in strict FP32, relaxed FP32 and FP64.
Writes profiles/evaluate_actions_bench.json (or --out).

Per precision:
  - one evaluate_actions call of K = 5 U(-5, 5) candidate actions per env, and K step calls on the same handle (one per
    candidate), alternated, each timed with CUDA events after the L2 is overwritten; candidate evaluations per second, env
    steps per second, and their ratio;
  - at a small batch (--small-envs), the host wall time of one evaluate_actions call against the loop it replaces,
    state_dict -> step(candidate k) -> load_state_dict for every k, both ending in a device synchronise.
Card name, power limit and max SM clock are read in the same run.
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

MODES = {"f32_strict": ("f32", True), "f32_relaxed": ("f32", False), "f64": ("f64", True)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def stats(t):
    return {"median": float(np.median(t)), "min": float(np.min(t)), "max": float(np.max(t))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--small-envs", type=int, default=64)
    ap.add_argument("--K", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "evaluate_actions_bench.json"))
    args = ap.parse_args()
    case = get_layout("HornsRev1_")
    lx, ly = np.asarray(case["xcoords"]), np.asarray(case["ycoords"])
    K, T = args.K, len(lx)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # 256 MB > the 126 MB of L2
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    res = {"card": card(), "layout": "HornsRev1_", "envs": args.envs, "small_envs": args.small_envs, "turbines": T, "K": K,
           "reps": args.reps, "l2": "overwritten (256 MB) before every timed call (large batch)", "modes": {}}

    def handle(B, precision, strict):
        rng = np.random.default_rng(0)
        ws = np.clip(8 * rng.weibull(8, B), 3, 28)
        wd = np.clip(rng.normal(270, 20, B) % 360, 0, 360)
        fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=10**9, strict=strict)
        fb.reset(ws, wd, host_trig=True)
        act = torch.as_tensor(rng.uniform(-5, 5, (B, K, T)).astype(np.float32), device="cuda")
        return fb, act, [act[:, k].contiguous() for k in range(K)]

    for mode, (precision, strict) in MODES.items():
        fb, act, cols = handle(args.envs, precision, strict)

        def timed(fn):
            flush.zero_()
            ev[0].record()
            fn()
            ev[1].record()
            torch.cuda.synchronize()
            return ev[0].elapsed_time(ev[1])

        def steps():
            for c in cols:
                fb.step(c)

        for _ in range(2):  # warm-up of both arms
            fb.evaluate_actions(act)
            steps()
        t_eval, t_step = [], []
        for _ in range(args.reps):
            t_eval.append(timed(lambda: fb.evaluate_actions(act)))
            t_step.append(timed(steps))
        fb.close()
        me, ms = float(np.median(t_eval)), float(np.median(t_step))

        # the loop evaluate_actions replaces, at a small batch: host wall time, both arms ending in a synchronise
        sb, sact, scols = handle(args.small_envs, precision, strict)

        def restore_loop():
            for c in scols:
                sd = sb.state_dict()
                sb.step(c)
                sb.load_state_dict(sd)
            torch.cuda.synchronize()

        def evaluate_small():
            sb.evaluate_actions(sact)
            torch.cuda.synchronize()

        def wall(fn):
            t0 = time.perf_counter()
            fn()
            return (time.perf_counter() - t0) * 1e3

        for _ in range(2):
            evaluate_small()
            restore_loop()
        w_eval, w_loop = [], []
        for _ in range(args.reps):
            w_eval.append(wall(evaluate_small))
            w_loop.append(wall(restore_loop))
        sb.close()
        res["modes"][mode] = {
            "evaluate_ms": stats(t_eval),
            "step_K_calls_ms": stats(t_step),
            "candidate_evaluations_per_s": args.envs * K / (me * 1e-3),
            "env_steps_per_s": args.envs * K / (ms * 1e-3),
            "ratio": ms / me,
            "small_batch_wall_ms": {"evaluate_actions": stats(w_eval), "state_dict_step_load_loop": stats(w_loop),
                                    "ratio": float(np.median(w_loop) / np.median(w_eval))},
        }
        print(mode, json.dumps(res["modes"][mode]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fp:
        json.dump(res, fp, indent=1)


if __name__ == "__main__":
    main()
