"""Rollout evaluation (wf_evaluate_rollouts) against stepping a handle of B*K envs, on HornsRev1 x 1024 envs, K = 16
candidate sequences of H = 8 steps, in strict FP32, relaxed FP32 and FP64.  Writes profiles/evaluate_rollouts_bench.json
(or --out).

Per precision:
  - arm 1: one evaluate_rollouts call (reward and truncated only);
  - arm 2: H step calls on a second handle of B*K envs whose state was copied from the B envs (only the steps are timed:
    the best case for that alternative);
  the two arms alternated, each timed with CUDA events after the L2 is overwritten (256 MB); median and min-max of --reps;
  candidate-steps per second of both and their ratio;
  - strict FP32 and FP64: the host wall time of one cem_plan call (samples 64, iterations 3, H 8) on a VecWindFarmEnv of
    the same size, ending in a device synchronise (median and min-max of 3).
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
from wfcrl_b200.planning import cem_plan  # noqa: E402
from wfcrl_b200.vector_env import VecWindFarmEnv  # noqa: E402

MODES = {"f32_strict": ("f32", True), "f32_relaxed": ("f32", False), "f64": ("f64", True)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def stats(t):
    return {"median": float(np.median(t)), "min": float(np.min(t)), "max": float(np.max(t))}


def cem_wall(precision, B, H, samples):
    env = VecWindFarmEnv("HornsRev1_", B, precision=precision, max_num_steps=10**6)
    env.reset(seed=0)
    gen = torch.Generator(device="cuda")

    def plan():
        gen.manual_seed(0)
        cem_plan(env, H, samples=samples, iterations=3, generator=gen)
        torch.cuda.synchronize()

    plan()  # warm-up
    wall = []
    for _ in range(3):
        t0 = time.perf_counter()
        plan()
        wall.append((time.perf_counter() - t0) * 1e3)
    env.close()
    return {**stats(wall), "samples": samples, "iterations": 3, "H": H}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--K", type=int, default=16)
    ap.add_argument("--H", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cem-samples", type=int, default=64)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "evaluate_rollouts_bench.json"))
    args = ap.parse_args()
    case = get_layout("HornsRev1_")
    lx, ly = np.asarray(case["xcoords"]), np.asarray(case["ycoords"])
    B, K, H, T = args.envs, args.K, args.H, len(lx)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # 256 MB > the 126 MB of L2
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    res = {"card": card(), "layout": "HornsRev1_", "envs": B, "turbines": T, "K": K, "H": H, "reps": args.reps,
           "l2": "overwritten (256 MB) before every timed call", "modes": {}}

    def timed(fn):
        flush.zero_()
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1])

    for mode, (precision, strict) in MODES.items():
        rng = np.random.default_rng(0)
        ws = np.clip(8 * rng.weibull(8, B), 3, 28)
        wd = np.clip(rng.normal(270, 20, B) % 360, 0, 360)
        kw = dict(precision=precision, kernel="fast", max_iter=10**9, strict=strict)
        fb = FlorisBatch(lx, ly, B, **kw)
        fb.reset(ws, wd, host_trig=True)
        fb.step(torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda"))
        act = torch.as_tensor(rng.uniform(-5, 5, (B, K, H, T)).astype(np.float32), device="cuda")
        # arm 2: B*K envs, env b*K + k a copy of env b (state_dict arrays repeated K times along the env axis)
        twin = FlorisBatch(lx, ly, B * K, **kw)
        twin.reset(np.repeat(ws, K), np.repeat(wd, K), host_trig=True)
        twin.load_state_dict({name: np.repeat(v, K, axis=0) for name, v in fb.state_dict().items()})
        cols = [act[:, :, h].reshape(B * K, T).contiguous() for h in range(H)]

        def rollouts():
            fb.evaluate_rollouts(act, ("reward", "truncated"))

        def steps():
            for c in cols:
                twin.step(c)

        for _ in range(2):  # warm-up of both arms
            rollouts()
            steps()
        t_roll, t_step = [], []
        for _ in range(args.reps):
            t_roll.append(timed(rollouts))
            t_step.append(timed(steps))
        twin.close()
        fb.close()
        mr, ms = float(np.median(t_roll)), float(np.median(t_step))

        res["modes"][mode] = {
            "evaluate_rollouts_ms": stats(t_roll),
            "step_H_calls_BK_envs_ms": stats(t_step),
            "rollout_candidate_steps_per_s": B * K * H / (mr * 1e-3),
            "stepping_candidate_steps_per_s": B * K * H / (ms * 1e-3),
            "ratio": ms / mr,
        }
        if strict:  # the vector env runs strict FP32
            res["modes"][mode]["cem_plan_wall_ms"] = cem_wall(precision, B, H, args.cem_samples)
        print(mode, json.dumps(res["modes"][mode]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fp:
        json.dump(res, fp, indent=1)


if __name__ == "__main__":
    main()
