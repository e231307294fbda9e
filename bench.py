#!/usr/bin/env python
"""Benchmark of the hot path BASELINE.json names: Floris env-steps/sec on HornsRev1 (80 turbines in the reference's
data_cases.py:269-291; README/BASELINE.json say 76), FP32 fast mode, env batch sharded over the GPUs of one box.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (CUDA kernels through the C-ABI)
    python bench.py --impl reference [--gpus N] ...                 # the reference's CPU path (oracle port, all cores)
    python bench.py ... --dump-outputs DIR                          # also write the last timed step's outputs as .npy

For N > 1 launch under torchrun (one rank per GPU).  Rank 0 prints ONE JSON line.
A "step" = one env step (constraint + yaw transition + full FLORIS GCH wake solve + measures + reward) for EVERY env of
the batch.  No collective in the step; NCCL only all-gathers the per-rank episode-return statistics at the end.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LAYOUT = "HornsRev1_"
ENVS_PER_GPU = 8192          # BASELINE.json configs[4]: 65536 envs over 8 GPUs
MAX_NUM_STEPS = 500          # simple_env.py:24 default episode length (truncation at step 499)
L2_FLUSH_BYTES = 256 << 20   # > 126 MB L2
DUMP_MAX_BYTES = 64 << 20    # --dump-outputs: above this, a fixed seeded sample of env rows is written


def dump_outputs(path: str, arrays: dict) -> None:
    """Writes the step outputs (numpy arrays, leading dim = env) as path/<name>.npy, float32 / float64 as computed (the
    uint8 `truncated` flag as float32).  Over DUMP_MAX_BYTES the same seeded sample of env rows is taken from every
    array, in env order, and its env indices are written as env_index.npy."""
    arrays = {k: a if a.dtype in (np.float32, np.float64) else a.astype(np.float32) for k, a in arrays.items()}
    B = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a.nbytes for a in arrays.values()) // B
    if row_bytes * B > DUMP_MAX_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(B, DUMP_MAX_BYTES // (row_bytes + 8), replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------------------------
# canonical algorithmic work per env-step (SURVEY.md section 8d / BASELINE.md section 4)
# ------------------------------------------------------------------------------------------------------------------
def canonical_work(T: int):
    n_pp = 9 * T * (T - 1) // 2
    w_fp32 = 121 * n_pp + 950 * T
    w_sp = 23.2 * n_pp + 190 * T
    return w_fp32, w_sp


def algorithmic_bytes(T: int) -> int:
    return 48 * T + 16


def _e2e_roofline(world: int, e2e_value: float, envs_per_gpu: int, bytes_per_step: int):
    """End-to-end bytes/s against the box's measured host<->device ceiling: the committed output of
    tools/pcie_probe_multi.py (plain cudaMemcpyAsync with the same byte counts, one GPU alone and all 8 GPUs at once)."""
    def probe(n):
        path = os.path.join(ROOT, "profiles", f"r2_pcie_probe_{n}gpu.json")
        if not os.path.exists(path):
            return None
        rec = json.load(open(path))
        return max(rec["one_copy_per_direction"]["aggregate_GBps"], rec["library_pattern_6x9_copies"]["aggregate_GBps"])

    alone, box = probe(1), probe(8)  # one GPU copying alone; all eight of the box at once (the host side's limit)
    if alone is None and box is None:
        return None
    peak = min(v for v in ((alone * world) if alone else None, box) if v is not None)
    n = "1 and 8" if alone and box else ("1" if alone else "8")
    achieved = e2e_value / envs_per_gpu * bytes_per_step / 1e9
    return {"bound": "host<->device copies (PCIe + host memory)", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "peak_source": f"min(n_gpus x one GPU copying alone, all 8 GPUs of the box copying at once) from "
                           f"profiles/r2_pcie_probe_*gpu.json (probes available: {n} GPU(s))"}


def _ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the step kernel, from the committed ncu --set full capture
    of this same command (profiles/ncu_traffic.json, written by hand from `ncu -i ... --page raw`); None if absent."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as fp:
            rec = json.load(fp)[kernel]
        return {"bytes_per_launch": rec["dram_bytes_read"] + rec["dram_bytes_write"], "source": rec["source"],
                "algorithmic_bytes_per_launch": rec.get("algorithmic_bytes"),
                "warp_instructions_per_env_step": rec.get("warp_instructions_per_env_step")}
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------------------------
# nvidia-smi clock sampler (B200_PROFILING.md "clocks DURING the timed region")
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ts, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                clk, mx = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            smax.append(mx)
            if t0 - 0.05 <= ts <= t1 + 0.05:
                sm.append(clk)
                try:
                    power.append(float(parts[3]))
                except ValueError:
                    pass
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                     parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # timed region shorter than the sampling period: fall back to every sample taken
            for ts, line in self.lines:
                parts = [p.strip() for p in line.split(",")]
                try:
                    sm.append(float(parts[1]))
                except Exception:
                    pass
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's Python+FLORIS step (numpy, same op structure), all host cores
# ------------------------------------------------------------------------------------------------------------------
def _cpu_worker(conn, layout, seed):
    sys.path.insert(0, ROOT)
    from oracle.env_oracle import EnvOracle
    from wfcrl_b200.layouts import get_layout

    case = get_layout(layout)
    env = EnvOracle(case["xcoords"], case["ycoords"], max_num_steps=MAX_NUM_STEPS)
    rng = np.random.default_rng(seed)
    env.reset(seed=seed)
    T = env.num_turbines
    done_steps = 0
    conn.send("ready")
    while True:
        n = conn.recv()
        if n <= 0:
            break
        t0 = time.perf_counter()
        for _ in range(n):
            env.step({"yaw": rng.uniform(-5, 5, T).astype(np.float32)})
            done_steps += 1
            if done_steps >= MAX_NUM_STEPS - 1:
                env.reset(seed=seed + done_steps)
                done_steps = 0
        conn.send(time.perf_counter() - t0)


class CpuFarm:
    """`workers` persistent single-env processes of the oracle port (the reference runs one env per process)."""

    def __init__(self, layout: str, workers: int):
        import multiprocessing as mp

        for var in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
            os.environ.setdefault(var, "1")
        ctx = mp.get_context("spawn")
        self.workers = workers
        self.conns, self.procs = [], []
        for w in range(workers):
            parent, child = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(child, layout, 1000 + w), daemon=True)
            p.start()
            self.conns.append(parent)
            self.procs.append(p)
        for c in self.conns:
            assert c.recv() == "ready"

    def run(self, steps_per_worker: int) -> float:
        """All workers step concurrently; returns aggregate env-steps/s (total steps / slowest worker)."""
        for c in self.conns:
            c.send(steps_per_worker)
        per = [c.recv() for c in self.conns]
        return self.workers * steps_per_worker / max(per)

    def close(self):
        for c in self.conns:
            try:
                c.send(0)
            except Exception:
                pass
        for p in self.procs:
            p.join(timeout=5)


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1



# ------------------------------------------------------------------------------------------------------------------
# device-timed legs shared by the headline workload and the other BASELINE configs
# ------------------------------------------------------------------------------------------------------------------
def _timed_steps(torch, step_fn, steps, flush):
    """`steps` calls of step_fn(k), each bracketed by CUDA events on the launching stream; L2 flushed outside the brackets.
    Returns the list of per-step milliseconds."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        if flush is not None:
            flush.zero_()
        ev[k][0].record()
        step_fn(k)
        ev[k][1].record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


OTHER_CONFIGS = [  # BASELINE.json configs[1..3] (configs[4] is the headline, configs[0] the CPU reference case)
    dict(key="configs[1] Dec_Ablaincourt_Floris", layout="Ablaincourt_", envs=4096, precision="f32", multi_agent=True,
         ti_range=None, note="PettingZoo 7 agents (one full agent cycle per launch, stale per-agent constraint), FP32 strict"),
    dict(key="configs[2] Turb16_TCRWP_Floris", layout="Turb16_TCRWP_", envs=16384, precision="f32", multi_agent=False,
         ti_range=(0.04, 0.12), note="wind speed / direction / TI sampled per env at every reset, FP32 strict"),
    dict(key="configs[3] Turb32_Row5_Floris FP64", layout="Turb32_Row5_", envs=8192, precision="f64", multi_agent=False,
         ti_range=None, note="FP64 bit-check mode (<= 1e-9 vs the oracle), weak scaling: 8192 envs per GPU"),
]


def run_other_configs(torch, dist, world, rank, local, steps, flush):
    """Device-timed throughput of BASELINE configs[1..3] on this rank's shard; max over ranks; same timing rules."""
    from wfcrl_b200.backend import FlorisBatch
    from wfcrl_b200.layouts import get_layout

    dev = torch.device("cuda", local)
    out = []
    for cfgd in OTHER_CONFIGS:
        case = get_layout(cfgd["layout"])
        T, B = case["num_turbines"], cfgd["envs"]
        fb = FlorisBatch(case["xcoords"], case["ycoords"], B, device=local, precision=cfgd["precision"], kernel="fast",
                         max_iter=MAX_NUM_STEPS, multi_agent=cfgd["multi_agent"])
        fb.reset_sampled(None, seed=7, env_id_offset=rank * B, turbulence_intensity_range=cfgd["ti_range"])
        gen = torch.Generator(device=dev)
        gen.manual_seed(4321 + rank)
        pool = [(torch.rand(B, T, device=dev, generator=gen) * 10 - 5).contiguous() for _ in range(4)]
        for k in range(3):
            fb.step(pool[k % 4])
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        l0 = fb.launch_count()
        ms = _timed_steps(torch, lambda k: fb.step(pool[k % 4]), steps, flush)
        launches = fb.launch_count() - l0
        n_fix = int(fb.get_state("ambiguous").sum()) if cfgd["precision"] == "f32" else 0
        tot = torch.tensor([float(sum(ms))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        total_ms = float(tot[0])
        info = fb.device_info()
        fb.close()
        if rank == 0:
            per_gpu = B * steps / (total_ms / 1e3)
            w_fp32, w_sp = canonical_work(T)
            lanes = 128 if cfgd["precision"] == "f32" else 64
            peak = info["sm_count"] * lanes * 1965.0e6
            out.append({
                "config": cfgd["key"], "turbines": T, "envs_per_gpu": B, "precision": cfgd["precision"], "note": cfgd["note"],
                "steps": steps, "ms_per_step": total_ms / steps, "value": world * per_gpu, "unit": "env-steps/s",
                "gpu_launches": int(launches), "envs_resolved_in_fp64_last_step": n_fix,
                "roofline": {"bound": "fp32_issue" if lanes == 128 else "fp64_issue",
                             "frac": per_gpu * (w_fp32 + w_sp) / peak,
                             "basis": f"canonical {w_fp32 + w_sp:.0f} lane-ops per env-step over {info['sm_count']} SMs x {lanes} lanes x 1965 MHz"},
            })
    return out


def run_sustained(torch, fb, pool, seconds, B, local, gid0):
    """Back-to-back steps for `seconds` (no L2 flush, one event pair around the whole run, an in-loop sampled reset of every
    env each 400 steps -- its cost is inside the figure) with the nvidia-smi sampler on: is the headline number a burst figure?"""
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    for k in range(20):
        fb.step(pool[k % len(pool)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    n = 0
    e0.record()
    while True:
        for k in range(200):
            fb.step(pool[k % len(pool)])
        n += 200
        if n % 400 == 0:
            fb.reset_sampled(None, seed=1, env_id_offset=gid0)  # (the handle never reaches max_iter here: explicit reset)
        torch.cuda.synchronize()
        if time.time() - t0 >= seconds:
            break
    e1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop(t0, t1)
    return {"seconds": ms / 1e3, "steps": n, "ms_per_step": ms / n, "value_per_gpu": B * n / (ms / 1e3), "unit": "env-steps/s",
            "l2": "not flushed (back-to-back launches)", "clocks": clocks}


def native_c_rate(layout, seconds=6.0):
    """The C restatement of the oracle (oracle/floris_oracle.c, all host threads) on a bounded sample of the headline workload:
    what a competent native CPU implementation of the reference's solve does on this box (checker code, never shipped)."""
    from oracle import c_oracle
    from wfcrl_b200.layouts import layout_xy

    lx, ly = layout_xy(layout)
    T = len(lx)
    rng = np.random.default_rng(3)
    n = 2048
    ws = np.clip(8 * rng.weibull(8, n), 3, 28)
    wd = np.clip(rng.normal(270, 20, n) % 360, 0, 360)
    yaw = rng.uniform(-40, 40, (n, T))
    c_oracle.solve_batch(lx, ly, ws[:64], wd[:64], yaw[:64])
    t0 = time.perf_counter()
    done = 0
    while time.perf_counter() - t0 < seconds:
        c_oracle.solve_batch(lx, ly, ws, wd, yaw)
        done += n
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "solves/s", "threads": os.cpu_count(), "kind": "port (C restatement, OpenMP/pthreads over envs)",
            "sample": f"{done} HornsRev1 solves in {dt:.1f} s"}

# ------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    workers = min(cores, 64)
    from wfcrl_b200.layouts import get_layout

    T = get_layout(LAYOUT)["num_turbines"]
    per_step = 2  # env steps per worker per bench "step" (bounded sample: ~0.1-0.2 s per env step at T=80)
    farm = CpuFarm(LAYOUT, workers)
    for _ in range(max(args.warmup, 0)):
        farm.run(1)
    rates, t0 = [], time.perf_counter()
    for _ in range(args.steps):
        rates.append(farm.run(per_step))
    wall = time.perf_counter() - t0
    farm.close()
    value = float(np.mean(rates))
    line = {
        "impl": "reference", "metric": "Floris env-steps/sec (HornsRev1)", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"HornsRev1_Floris T={T}, {workers} single-env host processes x {per_step} env steps per "
                               "bench step, U(-5,5) yaw actions, sampled wind"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": workers, "kind": "port",
                         "sample": f"{workers} procs x {per_step} steps x {args.steps} repeats of the numpy oracle port "
                                   "(FLORIS is not installable here; restated oracle, not the reference package)"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from wfcrl_b200.backend import FlorisBatch
    from wfcrl_b200.layouts import get_layout

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL announces its version on stdout when the first communicator comes up; stdout carries the JSON line only
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from wfcrl_b200.dist import bind_to_gpu_numa_node

    all_cpus = os.sched_getaffinity(0)  # restored before the CPU baseline, which wants every host core
    numa = bind_to_gpu_numa_node(local) if not os.environ.get("WFCRL_NO_NUMA_BIND") else {"bound": False}

    case = get_layout(LAYOUT)
    T, B = case["num_turbines"], args.envs_per_gpu
    precision = args.precision
    fb = FlorisBatch(case["xcoords"], case["ycoords"], B, device=local, precision=precision, kernel=args.kernel,
                     max_iter=MAX_NUM_STEPS)
    real = torch.float64 if precision == "f64" else torch.float32

    # synthetic wind-condition stream: the reference's reset distribution (mdp.py:242-258), keyed by the GLOBAL env id so
    # that 1/2/4/8-GPU runs see identical per-env streams (SURVEY 8e)
    gid0 = rank * B
    ws = np.empty(B)
    wd = np.empty(B)
    for b in range(B):
        rng = np.random.default_rng(gid0 + b)
        ws[b] = np.clip(8 * rng.weibull(8), 3, 28)
        wd[b] = np.clip(rng.normal(270, 20) % 360, 0, 360)

    # synthetic yaw-action stream U(-5, 5), a pool of distinct device buffers cycled through
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    pool = [(torch.rand(B, T, device=dev, generator=gen) * 10 - 5).contiguous() for _ in range(8)]
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    fb.reset(ws, wd, host_trig=False)
    # in-kernel auto-reset: the truncating step zeroes the envs' state itself; one geometry + warm-up launch pair draws the
    # fresh winds (keyed by (global env id, episode)) and restarts the episodes -- no host round trip
    fb.set_autoreset(True, seed=0, env_id_offset=gid0)
    steps_in_episode = 0
    returns = torch.zeros(B, dtype=torch.float64, device=dev)

    def env_step(k):
        nonlocal steps_in_episode
        out = fb.step(pool[k % len(pool)])
        steps_in_episode += 1
        if steps_in_episode >= MAX_NUM_STEPS - 1:  # every env truncates together (fixed episode length)
            fb.autoreset_finish()
            steps_in_episode = 0
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(max(args.warmup, 3)):
        env_step(k)
    barrier()

    # ---- timed region: K steps, L2 flushed before each, CUDA events on the launching stream -----------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = fb.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.time()
    for k in range(args.steps):
        flush.zero_()
        ev[k][0].record()
        out = env_step(k)
        ev[k][1].record()
        returns += out["reward"].double()
    barrier()
    t_wall1 = time.time()
    launches = fb.launch_count() - launches0
    if args.dump_outputs and rank == 0:  # before the legs below overwrite fb.out in place
        dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in out.items()})
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = float(sum(step_ms))
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    resolved = int(fb.get_state("ambiguous").sum()) if precision == "f32" and args.kernel == "fast" else 0

    # ---- per-kernel device time of the same steps (events between the launches inside the library; separate leg so that
    #      the headline region above is not perturbed): the roofline block is about the dominant kernel's own launches ------
    kernel_ms = None
    try:
        fb.set_kernel_timing(True)
        for k in range(args.steps):
            flush.zero_()
            env_step(k)
        kernel_ms = fb.kernel_timing()
        fb.set_kernel_timing(False)
        if not kernel_ms["calls"]:
            kernel_ms = None
    except Exception as exc:  # an older library without the hook
        log(f"kernel timing unavailable: {exc}")

    # ---- the same workload on a RELAXED handle (raw FP32, no FP64 re-solve launch): what strictness costs ------------
    relaxed_ms = None
    if precision == "f32" and args.kernel == "fast" and not args.quick:
        fr = FlorisBatch(case["xcoords"], case["ycoords"], B, device=local, precision=precision, kernel=args.kernel,
                         max_iter=10 ** 6, strict=False)
        fr.reset(ws, wd, host_trig=False)
        for k in range(3):
            fr.step(pool[k % len(pool)])
        barrier()
        relaxed_ms = float(sum(_timed_steps(torch, lambda k: fr.step(pool[k % len(pool)]), args.steps, flush)))
        fr.close()

    # ---- sustained leg: seconds of back-to-back steps with the clock sampler on ----------------------------------------
    sustained = None
    if not args.quick and rank == 0 and args.sustained_seconds > 0:
        sustained = run_sustained(torch, fb, pool, args.sustained_seconds, B, local, gid0)
    barrier()

    # ---- the other BASELINE configs (device-timed, this rank's shard, max over ranks) -------------------------------------
    other = run_other_configs(torch, dist, world, rank, local, max(5, min(args.steps, 20)), flush) if not args.quick else None

    # ---- end-to-end: host buffers, H2D + step + D2H inside the timed region -----------------------------------------
    host_pool = [p.cpu().pin_memory() for p in pool[:4]]
    e2e_steps = max(3, min(args.steps, 50))

    def e2e_run(**kw):
        fb.step_host(host_pool[0], **kw)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            res = fb.step_host(host_pool[k % len(host_pool)], **kw)
        barrier()
        dt = time.perf_counter() - t0
        assert bool(torch.isfinite(res["reward"]).all())
        return dt

    e2e_s = e2e_run()  # the library's own choice of host path (copy engines at this batch size)
    h2d, d2h = fb.last_h2d_bytes, fb.last_d2h_bytes
    os.environ["WFCRL_B200_HOST_PATH"] = "zero_copy"  # same call with the pinned buffers mapped into the step kernel
    e2e_zero_s = e2e_run()
    del os.environ["WFCRL_B200_HOST_PATH"]
    # what a policy consumes per step (observation + reward + flag), without the info arrays power / load
    e2e_obs_s = e2e_run(fields=("yaw", "wind_speed", "wind_direction", "freewind", "reward", "truncated"))
    d2h_obs = fb.last_d2h_bytes
    os.sched_setaffinity(0, all_cpus)

    # ---- max over ranks ---------------------------------------------------------------------------------------------
    stats = torch.tensor([total_ms, e2e_s, e2e_zero_s, e2e_obs_s, relaxed_ms or 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        # the only collective of the job: all-gather of per-rank episode-return statistics (north_star)
        mine = torch.stack([returns.mean(), returns.std()]).to(torch.float64)
        gathered = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        mean_return = float(torch.stack(gathered)[:, 0].mean())
    else:
        mean_return = float(returns.mean())
    total_ms, e2e_s, e2e_zero_s, e2e_obs_s, relaxed_ms = (float(v) for v in stats)

    if rank == 0:
        info = fb.device_info()
        value = world * B * args.steps / (total_ms / 1e3)
        per_gpu = value / world
        w_fp32, w_sp = canonical_work(T)
        sm_max_mhz = (clocks or {}).get("sm_max_mhz") or 1965.0
        sm_mhz = (clocks or {}).get("sm_mhz") or sm_max_mhz
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak, peak_src = 6650.0, "fallback"
        if os.path.exists(peaks_path):
            try:
                hbm_peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured"
            except Exception:
                pass
        lanes = 128 if precision == "f32" else 64  # FP32 / FP64 FMA lanes per SM per clock
        fp32_peak = info["sm_count"] * lanes * sm_max_mhz * 1e6
        mufu_peak = info["sm_count"] * 16 * sm_max_mhz * 1e6
        # rate of the DOMINANT kernel over its own launches (per GPU); the whole-step rate (incl. the FP64 re-solve launch of a
        # strict FP32 handle) is reported next to it as step_frac
        kern_rate = B / (kernel_ms["step_kernel_ms"] * 1e-3) if kernel_ms else per_gpu
        fp32_ach = kern_rate * (w_fp32 + w_sp)
        mufu_ach = kern_rate * w_sp
        hbm_ach = kern_rate * algorithmic_bytes(T) / 1e9
        roofline = {
            "bound": "fp32_issue" if precision == "f32" else "fp64_issue", "kernel": ("wf_step_fast64_kernel" if precision == "f64" else "wf_step_fast_kernel") if args.kernel == "fast" else "wf_step_basic_kernel",
            "achieved": fp32_ach / 1e9, "peak": fp32_peak / 1e9, "unit": "G lane-op/s", "frac": fp32_ach / fp32_peak,
            "frac_at_observed_clock": fp32_ach / (info["sm_count"] * lanes * sm_mhz * 1e6),
            "peak_basis": f"{info['sm_count']} SMs x {lanes} {'FP32' if lanes == 128 else 'FP64'} lanes x {sm_max_mhz:.0f} MHz "
                          f"(clocks.max.sm); canonical work {w_fp32 + w_sp:.0f} lane-ops per env-step (SURVEY 8d), not the "
                          "instructions actually issued" + ("" if lanes == 128 else "; every special function counted as ONE "
                          "op although FP64 evaluates it in software (10-40 instructions), so this fraction is a lower bound"),
            "mufu": {"achieved": mufu_ach / 1e9, "peak": mufu_peak / 1e9, "frac": mufu_ach / mufu_peak,
                     "unit": "G special/s",
                     "note": "CANONICAL special-function count of Appendix A per env-step; the kernel shares reciprocals and "
                             "exponentials and issues ~2.4x fewer MUFU instructions (ncu XU pipe ~51 % busy), so a value "
                             "above 1 is not a measurement error"} if precision == "f32" else None,  # FP64 specials run on the FP64 pipe
            "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "frac": hbm_ach / hbm_peak, "unit": "GB/s",
                    "peak_source": peak_src + " (MEASURED_PEAKS.json)" if peak_src == "measured" else "fallback"},
            "traffic": _ncu_traffic(("fast64" if precision == "f64" else "fast") if args.kernel == "fast" else
                                    ("basic" if precision == "f32" else "none")),
            "avg_launch_ms": kernel_ms["step_kernel_ms"] if kernel_ms else total_ms / max(launches, 1),
            "frac_basis": ("canonical work of one launch / the dominant kernel's own average launch duration, CUDA events "
                           "recorded between the launches inside the library (wf_set_kernel_timing) over a second pass of "
                           "the timed steps" if kernel_ms else "whole step (no per-kernel timing)"),
            "step_frac": per_gpu * (w_fp32 + w_sp) / fp32_peak,
            "step_frac_basis": "the same canonical work over the whole step = every launch of the step (value / n_gpus)",
            "resolve_kernel": ({"kernel": "wf_fixup64_kernel", "avg_launch_ms": kernel_ms["resolve_kernel_ms"],
                                "envs_resolved_last_step": resolved,
                                "what": "FP64 re-solve of the envs the FP32 launch flagged; latency-bound (one sequential "
                                        "sweep per env), not a throughput kernel"}
                               if kernel_ms and precision == "f32" and args.kernel == "fast" and kernel_ms["resolve_kernel_ms"] > 0.02 else None),
            "issue_slots": None,
            "occupancy": info,
        }
        tr = roofline["traffic"]
        if tr and tr.get("warp_instructions_per_env_step") and T == 80:
            # honest counterpart of the canonical fraction: instructions ACTUALLY issued (ncu count, committed) per second
            # over the issue-slot peak (4 warp-instructions / clk / SM)
            wi = tr["warp_instructions_per_env_step"]
            roofline["issue_slots"] = {"warp_instr_per_env_step": wi, "achieved_G_per_s": kern_rate * wi / 1e9,
                                       "peak_G_per_s": info["sm_count"] * 4 * sm_max_mhz * 1e6 / 1e9,
                                       "frac": kern_rate * wi / (info["sm_count"] * 4 * sm_max_mhz * 1e6)}
        line = {
            "metric": "Floris env-steps/sec (HornsRev1)", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if precision == "f32" else "f64", "data": "synthetic",
            "config": {"workload": f"HornsRev1_Floris, T={T} turbines (reference data_cases.py has 80; README says 76), "
                                   f"{B} envs per GPU x {world} GPU(s), U(-5,5) yaw actions, wind sampled per env from "
                                   f"the reference reset distribution, {MAX_NUM_STEPS}-step episodes",
                       "envs_per_gpu": B, "turbines": T, "precision": precision, "kernel": args.kernel,
                       "l2": "flushed between timed steps (256 MiB memset outside the event brackets)",
                       "parallelism": f"env-sharded x{world}, no collective in the step"},
            "e2e": {"value": world * B * e2e_steps / e2e_s, "unit": "env-steps/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "path": "FlorisBatch.step_host -> wf_step_host (pinned HOST action in, full step result out): "
                            "6 env chunks, one stream each, H2D + step kernel + D2H per chunk" +
                            (", then ONE FP64 re-solve launch whose envs come back as compact records scattered into the "
                             "caller's arrays" if precision == "f32" else ""),
                    "host_numa_binding": numa,
                    "observation_only_value": world * B * e2e_steps / e2e_obs_s,
                    "observation_only_d2h_bytes_per_step": int(d2h_obs),
                    "zero_copy_value": world * B * e2e_steps / e2e_zero_s,
                    "zero_copy_path": "same call with WFCRL_B200_HOST_PATH=zero_copy: host buffers mapped into the step "
                                      "kernel, one launch, no copy engine (the library's default up to 163840 env x "
                                      "turbine elements, where it is faster)"},
            "e2e_roofline": _e2e_roofline(world, world * B * e2e_steps / e2e_s, B, int(h2d) + int(d2h)),
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "mean_episode_return_so_far": mean_return,
            "parity_mode": {
                "mode": "strict" if precision == "f32" and args.kernel == "fast" else precision,
                "what": "every launch of the FP32 step kernel is followed by wf_fixup64_kernel, which re-solves in FP64 the envs "
                        "the FP32 kernel flagged (wake-overlap threshold inside its guard band, foot / cliff of the power "
                        "curve): every turbine within 1e-4 of the oracle (tests/test_fp32_strict_gpu.py)",
                "envs_resolved_in_fp64_last_step": resolved,
                "relaxed_value": (world * B * args.steps / (relaxed_ms / 1e3)) if relaxed_ms else None,
                "relaxed_ms_per_step": (relaxed_ms / args.steps) if relaxed_ms else None,
                "relaxed_what": "same workload, WfConfig.fp32_relaxed = 1: raw FP32 results, one launch per step; ~1e-4 of "
                                "the envs then carry a turbine off by up to ~1e-2 (profiles/r2_flag_sweep.json)",
            },
            "sustained": sustained,
            "other_configs": other,
        }
        if sustained:
            sm_obs = (sustained["clocks"] or {}).get("sm_mhz") or sm_max_mhz
            sustained["frac_at_observed_clock"] = sustained["value_per_gpu"] * (w_fp32 + w_sp) / (info["sm_count"] * lanes * sm_obs * 1e6)
            sustained["frac_at_max_clock"] = sustained["value_per_gpu"] * (w_fp32 + w_sp) / fp32_peak
        if world == 1 and not args.no_cpu_baseline:
            cores = host_cores()
            workers = min(cores, 64)
            t0 = time.perf_counter()
            farm = CpuFarm(LAYOUT, workers)
            farm.run(1)
            rate = farm.run(20)
            farm.close()
            wall = time.perf_counter() - t0
            line["cpu_baseline"] = {
                "value": rate, "unit": "env-steps/s", "cores": workers, "kind": "port",
                "sample": f"{workers} single-env processes x 20 HornsRev1 env steps of the numpy oracle port "
                          f"(wall {wall:.1f} s incl. process start)",
                "native_c": native_c_rate(LAYOUT)}
        print(json.dumps(line), flush=True)
    fb.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--kernel", default="fast", choices=["fast", "basic"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + e2e only (no relaxed / sustained / other-config legs)")
    ap.add_argument("--sustained-seconds", type=float, default=6.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                    "(rank 0's envs; at most 64 MB, a fixed seeded sample of envs beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours (the reference arm's steps run in worker processes)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
