"""Layout pool of mixed turbine counts against one handle per farm: 8192 envs of {HornsRev1 (80), Turb32_Row5 (32),
Ablaincourt (7)} cycled, FP32 strict and FP64, in one run.

(a) one T = 80 handle whose envs run the three farms (wf_set_layouts_sized): one step launch for the batch.  The small farms'
    CTAs reserve the shared memory of 80 turbines, which can cost occupancy.
(b) three single-layout handles holding the same envs (2731 / 2731 / 2730), stepped back to back on one stream: three
    launches, three tails.
Each arm is timed per plain step and per auto-reset step (max_iter = 2, so every step truncates every env: step + geometry
+ warm-up solve; arm (a) also draws every env's layout).

Arms alternate, ten steps at a time; L2 is flushed (256 MiB memset) before every timed step, outside the CUDA-event
brackets, as bench.py does.  The median of 100 steps per arm is reported with the device name and power limit.

Usage: python tools/bench_mixed_pool.py [--steps 100] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from wfcrl_b200.backend import FlorisBatch
from wfcrl_b200.layouts import layout_xy

B = 8192
FARMS = ["HornsRev1_", "Turb32_Row5_", "Ablaincourt_"]
L2_FLUSH_BYTES = 256 << 20
CHUNK = 10


def make_mixed(precision, max_iter, sample):
    farms = [layout_xy(n) for n in FARMS]
    fb = FlorisBatch(*farms[0], B, precision=precision, kernel="fast", max_iter=max_iter)
    fb.set_mixed_layouts([f[0] for f in farms], [f[1] for f in farms])
    fb.assign_layouts(None, np.arange(B) % len(FARMS))
    fb.set_layout_sampling(sample)
    fb.reset_sampled(None, seed=1, env_id_offset=0)
    fb.set_autoreset(True, seed=1, env_id_offset=0)
    return [fb]


def make_singles(precision, max_iter):
    out = []
    for l, name in enumerate(FARMS):
        n_envs = len(range(l, B, len(FARMS)))
        fb = FlorisBatch(*layout_xy(name), n_envs, precision=precision, kernel="fast", max_iter=max_iter)
        fb.reset_sampled(None, seed=1, env_id_offset=0)
        fb.set_autoreset(True, seed=1, env_id_offset=0)
        out.append(fb)
    return out


def timed(handles, acts, steps, flush, autoreset):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.zero_()
        ev[k][0].record()
        for fb, act in zip(handles, acts[k % 2]):
            fb.step(act)
            if autoreset:
                fb.autoreset_finish()
        ev[k][1].record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def device_facts():
    idx = torch.cuda.current_device()
    q = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(idx),
            "nvidia_smi": q.stdout.strip() if q.returncode == 0 else f"unavailable ({q.stderr.strip()})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mixed_pool needs a CUDA device")
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    result = {"workload": f"{B} envs of {FARMS} cycled, fast kernel, FP32 strict and FP64, L2 flushed before each timed "
                          f"step, median of {args.steps} steps per arm", **device_facts(), "results": {}}
    for precision in ("f32", "f64"):
        # plain steps: episodes longer than the run; auto-reset steps: max_iter = 2, so every step truncates every env
        arms = {("mixed", "step"): make_mixed(precision, 10 ** 6, False),
                ("mixed", "autoreset_step"): make_mixed(precision, 2, True),
                ("singles", "step"): make_singles(precision, 10 ** 6),
                ("singles", "autoreset_step"): make_singles(precision, 2)}
        acts = {key: [[torch.rand(fb.B, fb.T, device="cuda", generator=g) * 10 - 5 for fb in hs] for _ in range(2)]
                for key, hs in arms.items()}
        ms = {key: [] for key in arms}
        for key, hs in arms.items():  # warm-up
            timed(hs, acts[key], 3, flush, key[1] == "autoreset_step")
        for _ in range(0, args.steps, CHUNK):
            for key, hs in arms.items():
                ms[key] += timed(hs, acts[key], CHUNK, flush, key[1] == "autoreset_step")
        res = {}
        for (arm, kind), v in ms.items():
            res[f"{arm}/{kind}"] = {"median_ms": float(np.median(v)), "p10_ms": float(np.percentile(v, 10)),
                                    "p90_ms": float(np.percentile(v, 90)), "n": len(v)}
        for kind in ("step", "autoreset_step"):
            res[f"mixed_over_singles/{kind}"] = res[f"mixed/{kind}"]["median_ms"] / res[f"singles/{kind}"]["median_ms"]
        a = arms[("mixed", "step")][0]
        info = a.device_info()
        res["mixed_step_kernel"] = {k: info[k] for k in ("ctas_per_sm", "regs_per_thread", "smem_per_cta")}
        result["results"][precision] = res
        for hs in arms.values():
            for fb in hs:
                fb.close()
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fp:
            fp.write(text + "\n")


if __name__ == "__main__":
    main()
