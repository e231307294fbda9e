"""Cost of the layout pool on HornsRev1 x 8192 envs, FP32 strict and FP64, in one run.

(a) a pool of one layout (how every handle ran before the pool existed) against a pool of 8 identical copies of HornsRev1
    with layout sampling on.  Both arms do the same work, so the difference is what the mechanism
    costs: per plain step, and per auto-reset step (every env truncates; step + geometry/layout draw + warm-up solve).
(b) a pool of 8 distinct 80-turbine farms (HornsRev1 rotated by 0/45/90/135 degrees and their mirror images) with layout
    sampling on: for information, since other farms are other work.

Arms alternate within each repetition; L2 is flushed (256 MiB memset) before every timed step, outside the CUDA-event
brackets, as bench.py does.  Prints one JSON document with the device name and power limit.

Usage: python tools/bench_layout_pool.py [--reps 5] [--steps 20] [--out FILE]
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
L2_FLUSH_BYTES = 256 << 20


def distinct_farms():
    x, y = (np.asarray(v, dtype=np.float64) for v in layout_xy("HornsRev1_"))
    farms = []
    for mirror in (1.0, -1.0):
        for deg in (0.0, 45.0, 90.0, 135.0):
            c, s = np.cos(np.radians(deg)), np.sin(np.radians(deg))
            farms.append((c * mirror * x - s * y, s * mirror * x + c * y))
    return farms


def make_arm(arm, precision, max_iter):
    lx, ly = layout_xy("HornsRev1_")
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=max_iter)
    if arm == "pool8_same":
        fb.set_layouts([lx] * 8, [ly] * 8)
    elif arm == "pool8_distinct":
        farms = distinct_farms()
        fb.set_layouts([f[0] for f in farms], [f[1] for f in farms])
    if arm != "pool1":
        fb.set_layout_sampling(True)
    fb.reset_sampled(None, seed=1, env_id_offset=0)
    fb.set_autoreset(True, seed=1, env_id_offset=0)
    return fb


def timed(fb, acts, steps, flush, autoreset):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.zero_()
        ev[k][0].record()
        fb.step(acts[k % len(acts)])
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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_layout_pool needs a CUDA device")
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    T = len(layout_xy("HornsRev1_")[0])
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = [torch.rand(B, T, device="cuda", generator=g) * 10 - 5 for _ in range(4)]
    arms = ["pool1", "pool8_same", "pool8_distinct"]
    result = {"workload": f"HornsRev1_ x {B} envs, fast kernel, L2 flushed before each timed step", **device_facts(),
              "results": {}}
    for precision in ("f32", "f64"):
        # plain steps: episodes longer than the run; auto-reset steps: max_iter = 2, so every step truncates every env
        handles = {(arm, kind): make_arm(arm, precision, 10 ** 6 if kind == "step" else 2)
                   for arm in arms for kind in ("step", "autoreset_step")}
        a, b = handles[("pool1", "step")], handles[("pool8_same", "step")]
        oa = {k: v.clone() for k, v in a.step(acts[0]).items()}
        ob = b.step(acts[0])
        torch.cuda.synchronize()
        same = all(torch.equal(oa[k], ob[k]) for k in oa)  # identical copies: the same results bit for bit
        ms = {key: [] for key in handles}
        for key, fb in handles.items():  # warm-up
            timed(fb, acts, 3, flush, key[1] == "autoreset_step")
        for _rep in range(args.reps):
            for key, fb in handles.items():
                ms[key] += timed(fb, acts, args.steps, flush, key[1] == "autoreset_step")
        res = {"pool1_equals_pool8_same": same}
        for (arm, kind), v in ms.items():
            res[f"{arm}/{kind}"] = {"median_ms": float(np.median(v)), "p10_ms": float(np.percentile(v, 10)),
                                    "p90_ms": float(np.percentile(v, 90)), "n": len(v)}
        for kind in ("step", "autoreset_step"):
            base = res[f"pool1/{kind}"]["median_ms"]
            res[f"pool8_same_over_pool1/{kind}"] = res[f"pool8_same/{kind}"]["median_ms"] / base
        result["results"][precision] = res
        for fb in handles.values():
            fb.close()
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fp:
            fp.write(text + "\n")


if __name__ == "__main__":
    main()
