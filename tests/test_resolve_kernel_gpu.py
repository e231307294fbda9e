"""The strict FP32 handle's FP64 re-solve (wf_fixup64_kernel<W> behind steps, updates and resets, wf_fixup64_eval_kernel<W>
behind evaluate_yaw / evaluate_actions / evaluate_rollouts, both running solve_env64 in wf_fast64.cu), held to an FP64 handle
and to the C oracle at every width W it runs with, in every mode, with most of the batch flagged.

A re-solved row is an FP64 result rounded to float32, so the bar is float32 rounding of the reference:
|x - ref| <= ulp32(ref) / 2 + 1e-9 max(|ref|, floor), with the floors of the FP64 parity tests.  Rewards, which have no
relative term, are held to one float32 ulp of the FP64 handle's; truncation, free wind and the committed state must match
it exactly.

Most of the batch is flagged with two existing levers: winds of 2.6-2.8 m/s put the front row on the foot of the power curve
(DESIGN.md section 3), and a wide guard band (WFCRL_B200_AMB_EPS, read at wf_create) flags envs at ordinary winds."""
import numpy as np
import pytest

from tests._util import host_trig, layout

pytestmark = pytest.mark.gpu

# Guard-band half-width for these tests: the band is 0.025-0.075 m/s around the 0.05 m/s overlap threshold.  Measured on a
# B200 with 2048 envs at ordinary winds (reset / step / update), the default 2e-5 flags 0.1-2 % of the envs; 0.5 flags
# 81-88 % on a 7-turbine row, 60-71 % on HornsRev1 and 62-87 % on the jittered 128-turbine grid, but only 15-35 % on
# Turb32_Row5 and a 12-turbine grid column, where the low winds do the rest.  Larger values add little (0.9: 21-35 % on
# those two).  It stays below 1, where the lower end of the band would reach 0 m/s.
AMB_EPS = "0.5"
SMS = 148  # launch_fixup_sized hard-codes the SM count of a B200
PER_TURBINE = ("yaw", "wind_speed", "wind_direction", "power", "load")
# floors of the FP64 parity tests (test_solve_parity_gpu.py): interface units (W, x1e7 loads) and env units (MW, loads)
FLOORS = {"interface": {"yaw": 1.0, "wind_speed": 1e-3, "wind_direction": 1.0, "power": 1.0, "load": 1e4},
          "env": {"yaw": 1.0, "wind_speed": 1e-3, "wind_direction": 1.0, "power": 1e-6, "load": 1e-3}}
ORACLE_ROWS = 256


def _resolve_warps(T, count):
    """Warps per env of the FP64 re-solve behind a launch of `count` CTAs (B, or B*K*H for an evaluation) on a handle of T
    turbines: a mirror of launch_fixup_sized in wfcrl_b200/csrc/wf_fast64.cu."""
    w = 8 if T > 40 else (4 if T > 20 else (2 if T > 10 else 1))
    expected = count // 64 + 1
    while w > 1 and expected > SMS * 8 // w:
        w >>= 1
    return w


def _resolve_grid(T, count):
    """CTAs of that launch: one per env up to the resident count, then a grid-stride loop."""
    return min(count, SMS * 8 // _resolve_warps(T, count))


@pytest.fixture
def wide_band(monkeypatch):
    monkeypatch.setenv("WFCRL_B200_AMB_EPS", AMB_EPS)
    monkeypatch.delenv("WFCRL_B200_NO_VTAB", raising=False)
    monkeypatch.delenv("WFCRL_B200_HOST_PATH", raising=False)
    return monkeypatch


# ---- layouts ------------------------------------------------------------------------------------------------------------
def _grid(n, jitter):
    """The 16 x 8 grid of test_edge_cases_gpu.py (700 m x 600 m), first n turbines; without jitter every column is x-tied
    at 270 deg."""
    rng = np.random.default_rng(128)
    gx, gy = np.meshgrid(np.arange(16) * 700.0, np.arange(8) * 600.0)
    lx, ly = gx.ravel().copy(), gy.ravel().copy()
    if jitter:
        lx += rng.uniform(-40, 40, lx.shape)
        ly += rng.uniform(-40, 40, ly.shape)
    return lx[:n], ly[:n]


def _farm(kind, n):
    if kind == "hornsrev":
        lx, ly = layout("HornsRev1_")
        return lx[:n].copy(), ly[:n].copy()
    return _grid(n, kind == "grid_jitter")


def _winds(rng, B, low_frac=0.5):
    """Ordinary winds (the reference's reset distribution) with a share of 2.6-2.8 m/s; every fifth env exactly at 270 deg."""
    ws = np.clip(8 * rng.weibull(8, B), 3, 28)
    low = rng.random(B) < low_frac
    ws[low] = rng.uniform(2.6, 2.8, int(low.sum()))
    wd = np.clip(rng.normal(270, 20, B) % 360, 0, 360)
    wd[::5] = 270.0
    return ws, wd


# ---- comparisons --------------------------------------------------------------------------------------------------------
def _np(t):
    return t.double().cpu().numpy() if hasattr(t, "cpu") else np.asarray(t, dtype=np.float64)


def _ulp32(ref):
    return np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)


def _assert_f32_of(got, ref, floor, where):
    """`got` (float32 results) is `ref` (FP64) rounded to nearest float32, up to 1e-9 of the reference (relative to
    `floor`): half an ulp for the rounding, the relative term for the difference of two FP64 solves."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (where, got.shape, ref.shape)
    err = np.abs(got - ref)
    bar = 0.5 * _ulp32(ref) + 1e-9 * np.maximum(np.abs(ref), floor)
    bad = ~(err <= bar)
    if bad.any():
        k = np.unravel_index(int(np.argmax(np.where(bad, err / bar, 0))), err.shape)
        pytest.fail(f"{where}: {int(bad.sum())} of {err.size} outside float32 rounding; worst at {k}: got {got[k]!r}, "
                    f"ref {ref[k]!r}, bar {bar[k]:.3e}")


def _assert_rows(got, ref, rows, mode, where, n=None):
    """Per-turbine outputs of `rows` (index arrays / masks over the leading axes) against the reference's rows."""
    for key in PER_TURBINE:
        if key not in got:
            continue
        g, r = _np(got[key])[rows], _np(ref[key])[rows]
        if n is not None:
            g, r = g[:, :n], r[:, :n]
        _assert_f32_of(g, r, FLOORS[mode][key], (where, key))


def _oracle(lx, ly, ws, wd, yaw, mode, warmup=False, cs=None):
    """The C oracle's outputs in the units of `mode` (warm-up: the clamps of WF_MODE_WARMUP), from the rotation cosines /
    sines `cs` (default: numpy's, as `host_trig=True` ships them)."""
    from oracle import c_oracle

    cs = np.stack(host_trig(wd), 1) if cs is None else cs
    ref = c_oracle.solve_batch(lx, ly, ws, wd, yaw, cs=cs)
    loads = np.stack([ref["ti"], ref["std_u"], ref["std_v"], ref["std_w"]], -1)
    out = {"yaw": np.asarray(yaw, dtype=np.float64), "wind_speed": ref["ws_local"], "wind_direction": ref["wd_local"]}
    if mode == "interface":
        out["power"], out["load"] = ref["power_W"], loads * 1e7
    else:
        out["power"], out["load"] = ref["power_W"] / 1e6, loads
    if warmup:
        out["wind_speed"] = np.clip(out["wind_speed"], 3.0, 28.0)
        out["wind_direction"] = np.clip(out["wind_direction"], 0.0, 360.0)
    return out, ref["order"]


def _oracle_check(got, lx, ly, ws, wd, yaw, mode, where, warmup=False, order=None, n=None, cs=None):
    """`got`: per-turbine outputs of some rows (first axis), from a solve at (ws, wd, yaw) per row."""
    ref, ref_order = _oracle(lx, ly, ws, wd, yaw, mode, warmup, cs)
    for key in PER_TURBINE:
        g = _np(got[key])
        if n is not None:
            g = g[:, :n]
        _assert_f32_of(g, ref[key], FLOORS[mode][key], (where, "oracle", key))
    if order is not None:
        assert np.array_equal(order, ref_order), (where, "turbine order")


def _pick(rng, idx, k=ORACLE_ROWS):
    idx = np.asarray(idx)
    return idx if len(idx) <= k else np.sort(rng.choice(idx, k, replace=False))


def _enough(n, floor, where):
    """At least `floor` rows were flagged, so the case tested the re-solve (each floor is at most about half of the count
    measured on a B200)."""
    assert n >= floor, (where, int(n))


def _outs(o):
    return {k: v.clone() for k, v in o.items()}


def test_width_mirror_matches_the_launch_table():
    """The mirror reproduces the table of launch_fixup_sized's comment: T > 40 at the four batch-size bands."""
    for count, w in ((1, 8), (9471, 8), (9472, 4), (18943, 4), (18944, 2), (37887, 2), (37888, 1)):
        assert _resolve_warps(80, count) == w, count
    for T, w in ((10, 1), (11, 2), (20, 2), (21, 4), (40, 4), (41, 8), (128, 8)):
        assert _resolve_warps(T, 512) == w, T
    assert _resolve_grid(80, 2048) == 148 and _resolve_grid(7, 512) == 512


# ---- 1. step, update_command and warm-up at every width -----------------------------------------------------------------
FARM_SIZES = [7, 11, 12, 13, 31, 32, 33, 71, 72, 73, 80, 128]
KINDS = ["hornsrev", "grid", "grid_jitter"]
TABLES = ["table", "direct", "stale"]
SHAPERS = ["none", "reference", "step"]
CASES = [(T, kind, TABLES[(i + k) % 3], SHAPERS[(i + 2 * k) % 3])
         for i, T in enumerate(FARM_SIZES) for k, kind in enumerate(KINDS) if not (kind == "hornsrev" and T > 80)]
B1 = 512
MAX_ITER = 4


@pytest.mark.parametrize("T,kind,table,shaper", CASES)
def test_step_update_and_warmup_match_fp64(cuda_device, wide_band, T, kind, table, shaper):
    """Reset (warm-up), three env steps (the third truncates) and one interface update on a strict FP32 handle and an FP64
    twin: every flagged row at float32 rounding of the twin and of the oracle, per-env outputs and state equal."""
    import torch

    from wfcrl_b200.backend import FlorisBatch

    if table == "direct":
        wide_band.setenv("WFCRL_B200_NO_VTAB", "1")
    W = {7: 1, 11: 2, 12: 2, 13: 2, 31: 4, 32: 4, 33: 4}.get(T, 8)
    assert _resolve_warps(T, B1) == W
    lx, ly = _farm(kind, T)
    rng = np.random.default_rng(1000 + T + 7 * KINDS.index(kind))
    ws, wd = _winds(rng, B1)
    kw = dict(kernel="fast", max_iter=MAX_ITER, reward_shaper=shaper, shaper_reference=0.5 if shaper == "reference" else 0.0)
    f32, f64 = FlorisBatch(lx, ly, B1, precision="f32", **kw), FlorisBatch(lx, ly, B1, precision="f64", **kw)
    hs = (f32, f64)
    sub = np.random.default_rng(T)

    # warm-up: reset at low winds clamps wind speed to [3, 28] in the outputs
    outs = [_outs(fb.reset(ws, wd, host_trig=True)) for fb in hs]
    torch.cuda.synchronize()
    flag = f32.get_state("ambiguous").astype(bool)
    _enough(flag.sum(), B1 // 4, ("warm-up", T, kind, table))
    _assert_rows(outs[0], outs[1], flag, "env", "warm-up")
    assert np.array_equal(_np(outs[0]["freewind"]), _np(outs[1]["freewind"]).astype(np.float32))
    rows = _pick(sub, np.flatnonzero(flag))
    _oracle_check({k: outs[0][k][torch.as_tensor(rows, device="cuda")] for k in PER_TURBINE}, lx, ly, ws[rows], wd[rows],
                  np.zeros((len(rows), T)), "env", "warm-up", warmup=True, order=f32.get_state("order")[rows])
    assert np.array_equal(f32.get_state("order"), f64.get_state("order"))

    if table == "stale":
        # wf_update_wind rebuilds the table when the wind has been steady (here the first call: geometry, table and wind
        # launches) and not when the wind moves again within 8 steps (geometry and wind only).  The table is then stale:
        # the steps and the update below ignore it and evaluate every pair directly, in the FP32 kernel, the re-solve and
        # the FP64 handle's scatter kernel.
        for launches in (3, 2):
            ws, wd = _winds(rng, B1)
            for fb in hs:
                n0 = fb.launch_count()
                fb.update_wind(torch.as_tensor(ws, device="cuda"), torch.as_tensor(wd, device="cuda"), host_trig=True)
                assert fb.launch_count() - n0 == launches, (fb.precision, launches)

    # the warm-up solve counts as the episode's first iteration: the steps left run to the truncating one
    it0 = f32.get_state("num_iter")
    assert np.all(it0 == 1) and np.array_equal(it0, f64.get_state("num_iter"))
    steps = MAX_ITER - 1
    ep = np.zeros(B1)
    prev_ref = f32.get_state("shaper_ref")
    for k in range(steps):
        a = torch.as_tensor(rng.uniform(-5, 5, (B1, T)).astype(np.float32), device="cuda")
        o32, o64 = _outs(f32.step(a)), _outs(f64.step(a))
        torch.cuda.synchronize()
        flag = f32.get_state("ambiguous").astype(bool)
        _enough(flag.sum(), B1 // 4, ("step", k, T, kind, table))
        where = ("step", k)
        _assert_rows(o32, o64, flag, "env", where)
        r32, r64 = _np(o32["reward"]), _np(o64["reward"])
        if shaper == "step":
            # StepPercentage: the relative change of the unshaped reward, which the handle keeps in shaper_ref (a re-solved
            # env its FP64 reward, an FP32-solved one its float32 reward); both routes shape it the same way, exactly
            ref32, ref64 = f32.get_state("shaper_ref"), f64.get_state("shaper_ref")
            with np.errstate(divide="ignore", invalid="ignore"):
                want = np.where(prev_ref == 0.0, 0.0, (ref32 - prev_ref) / prev_ref).astype(np.float32)
            assert np.array_equal(r32, want.astype(np.float64)), where
            prev_ref = ref32
            assert np.all(np.abs(ref32[flag] - ref64[flag]) <= 1e-9 * np.maximum(np.abs(ref64[flag]), 1e-3)), where
            # against the FP64 handle the shaped reward carries the relative error of the two unshaped rewards (1e-4 bar),
            # one of which either route may have solved, scaled by their ratio 1 + r (large after a change of wind)
            assert np.all(np.abs(r32 - r64) <= 1e-4 * np.maximum(1.0, np.abs(1.0 + r64))), where
        else:
            # one ulp: half for the rounding and room for an FP64 reward next to a rounding midpoint
            assert np.all(np.abs(r32[flag] - r64[flag]) <= _ulp32(r64[flag])), where
        for key in ("truncated", "freewind", "yaw"):
            assert np.array_equal(_np(o32[key]), _np(o64[key]).astype(np.float32)), (where, key)
        for name in ("num_iter", "num_moves", "acc", "acc_prev", "yaw", "ws_norm"):
            assert np.array_equal(f32.get_state(name), f64.get_state(name)), (where, name)
        trunc = _np(o32["truncated"]).astype(bool)
        assert trunc.all() == (k == steps - 1) and not (trunc.any() and k < steps - 1), where
        # the re-solve accounts the float32 reward the caller sees; the truncating step moves the return to fin_sum
        assert np.array_equal(f32.get_state("fin_sum"), np.where(trunc, ep + r32, 0.0)), where
        ep = np.where(trunc, 0.0, ep + r32)
        assert np.array_equal(f32.get_state("ep_return"), ep), where
        rows = _pick(sub, np.flatnonzero(flag))
        yaw = f64.get_state("yaw")[rows]
        _oracle_check({kk: o32[kk][torch.as_tensor(rows, device="cuda")] for kk in PER_TURBINE}, lx, ly, ws[rows],
                      wd[rows], yaw, "env", where, order=f32.get_state("order")[rows])

    cmd = torch.as_tensor(rng.uniform(-30, 30, (B1, T)).astype(np.float32).astype(np.float64), device="cuda")
    o32, o64 = _outs(f32.update_command(cmd)), _outs(f64.update_command(cmd))
    torch.cuda.synchronize()
    flag = f32.get_state("ambiguous").astype(bool)
    _enough(flag.sum(), B1 // 4, ("update", T, kind, table))
    _assert_rows(o32, o64, flag, "interface", "update")
    rows = _pick(sub, np.flatnonzero(flag))
    _oracle_check({kk: o32[kk][torch.as_tensor(rows, device="cuda")] for kk in PER_TURBINE}, lx, ly, ws[rows], wd[rows],
                  cmd.cpu().numpy()[rows], "interface", "update", order=f32.get_state("order")[rows])
    for fb in hs:
        fb.close()


# ---- 2. the same envs at every width: bit for bit ----------------------------------------------------------------------
ROWS2 = 64
# (farm, vortex table, {batch size: W}, flagged-row floor of the 64).  An 80-turbine table of 40000 envs (36 GB) would exceed
# the 24 GB default cap, so with a table HornsRev1 stops at 24000 and the 32-turbine farm (5.7 GB at 40000) reaches W = 1.
WIDTH_CASES = [("HornsRev1_", "direct", {64: 8, 12000: 4, 24000: 2, 40000: 1}, ROWS2 // 2),
               ("HornsRev1_", "table", {64: 8, 12000: 4, 24000: 2}, ROWS2 // 2),
               ("Turb32_Row5_", "table", {64: 4, 24000: 2, 40000: 1}, ROWS2 // 4)]


@pytest.mark.parametrize("name,table,sizes,floor", WIDTH_CASES, ids=["hornsrev-direct", "hornsrev-table", "turb32-table"])
def test_width_does_not_change_results(cuda_device, wide_band, name, table, sizes, floor):
    """The same 64 env rows in handles of 64 to 40000 envs: the re-solve runs them with every W the farm size allows and must
    give the same bits."""
    import torch

    from wfcrl_b200.backend import FlorisBatch

    if table == "direct":
        wide_band.setenv("WFCRL_B200_NO_VTAB", "1")
    lx, ly = layout(name)
    T = len(lx)
    rng = np.random.default_rng(21)
    ws0, wd0 = _winds(rng, ROWS2)
    acts = [rng.uniform(-5, 5, (ROWS2, T)).astype(np.float32) for _ in range(2)]
    cmd = rng.uniform(-30, 30, (ROWS2, T))
    results, flags = [], []
    for B, W in sizes.items():
        assert _resolve_warps(T, B) == W
        fill = np.random.default_rng(B)
        ws, wd = _winds(fill, B)
        ws[:ROWS2], wd[:ROWS2] = ws0, wd0
        fb = FlorisBatch(lx, ly, B, precision="f32", kernel="fast", max_iter=50, reward_shaper="step")
        res, flg = [fb.reset(ws, wd, host_trig=True)], [fb.get_state("ambiguous")[:ROWS2]]
        res[0] = {k: v[:ROWS2].cpu() for k, v in res[0].items()}
        for a0 in acts:
            a = fill.uniform(-5, 5, (B, T)).astype(np.float32)
            a[:ROWS2] = a0
            o = fb.step(torch.as_tensor(a, device="cuda"))
            res.append({k: v[:ROWS2].cpu() for k, v in o.items()})
            flg.append(fb.get_state("ambiguous")[:ROWS2])
        c = fill.uniform(-30, 30, (B, T))
        c[:ROWS2] = cmd
        o = fb.update_command(torch.as_tensor(c, device="cuda"))
        res.append({k: v[:ROWS2].cpu() for k, v in o.items() if k != "reward"})
        flg.append(fb.get_state("ambiguous")[:ROWS2])
        state = {name: fb.get_state(name)[:ROWS2] for name in ("yaw", "ep_return", "shaper_ref", "num_iter", "acc")}
        fb.close()
        results.append((res, state))
        flags.append(flg)
        torch.cuda.empty_cache()
    for flg in flags[1:]:
        assert all(np.array_equal(f, g) for f, g in zip(flg, flags[0]))
    for j, f in enumerate(flags[0]):
        _enough(f.sum(), floor, ("widths", name, table, j))
    (res0, st0) = results[0]
    for (res, st), B in zip(results[1:], list(sizes)[1:]):
        for j, (r, r0) in enumerate(zip(res, res0)):
            for k in r0:
                assert torch.equal(r[k], r0[k]), (B, j, k)
        for name in st0:
            assert np.array_equal(st[name], st0[name]), (B, name)


# ---- 3. grid-stride loop over a pool of mixed farm sizes ---------------------------------------------------------------
MIXED = [("Turb1_Row1_", 1), ("Turb2_Row1_", 2), ("Ablaincourt_", 7), ("Turb12_Row1_", 12), ("Turb32_Row5_", 32),
         ("HornsRev1_", 72), ("HornsRev1_", 80)]


def test_mixed_pool_grid_stride(cuda_device, wide_band):
    """2048 envs over farms of 1..80 turbines on an 80-column handle, most of them flagged: W = 8 with 148 CTAs, each
    re-solving about ten envs of different sizes back to back.  Every farm against the FP64 pool and the oracle; padding 0."""
    import torch

    from wfcrl_b200.backend import FlorisBatch

    farms = [tuple(a[:n].copy() for a in layout(name)) for name, n in MIXED]
    B, T = 2048, 80
    assert _resolve_warps(T, B) == 8 and _resolve_grid(T, B) == 148
    kw = dict(kernel="fast", max_iter=50)
    hs = [FlorisBatch(*farms[-1], B, precision=p, **kw) for p in ("f32", "f64")]
    ids = np.arange(B) % len(farms)
    for fb in hs:
        fb.set_mixed_layouts([f[0] for f in farms], [f[1] for f in farms])
        fb.assign_layouts(None, ids)
    counts = np.array([n for _, n in MIXED])[ids]
    rng = np.random.default_rng(33)
    ws, wd = _winds(rng, B, low_frac=0.85)
    sub = np.random.default_rng(34)

    def check(o32, o64, mode, where, yaw_of=None, warmup=False):
        torch.cuda.synchronize()
        flag = hs[0].get_state("ambiguous").astype(bool)
        assert flag.sum() > 148
        _enough(flag.sum(), B // 2, ("mixed", where))
        order = hs[0].get_state("order")
        assert np.array_equal(order, hs[1].get_state("order")), where
        for lay, (lx, ly) in enumerate(farms):
            n = len(lx)
            rows = np.flatnonzero(flag & (ids == lay))
            _enough(len(rows), 100, ("mixed", where, n))
            _assert_rows(o32, o64, rows, mode, (where, n), n=n)
            pick = _pick(sub, rows, ORACLE_ROWS // len(farms))
            yaw = np.zeros((len(pick), n)) if yaw_of is None else yaw_of[pick][:, :n]
            _oracle_check({k: o32[k][torch.as_tensor(pick, device="cuda")] for k in PER_TURBINE}, lx, ly, ws[pick],
                          wd[pick], yaw, mode, (where, n), warmup=warmup, order=order[pick][:, :n], n=n)
        for key in PER_TURBINE:
            v = _np(o32[key])
            for lay, (lx, _) in enumerate(farms):
                assert not v[ids == lay][:, len(lx):].any(), (where, key, "padding")

    outs = [_outs(fb.reset(ws, wd, host_trig=True)) for fb in hs]
    check(*outs, "env", "warm-up", warmup=True)
    for k in range(2):
        a = torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda")
        outs = [_outs(fb.step(a)) for fb in hs]
        check(*outs, "env", ("step", k), yaw_of=hs[1].get_state("yaw"))
        flag = hs[0].get_state("ambiguous").astype(bool)
        r32, r64 = _np(outs[0]["reward"]), _np(outs[1]["reward"])
        assert np.all(np.abs(r32[flag] - r64[flag]) <= _ulp32(r64[flag])), ("step", k)
    cmd = rng.uniform(-30, 30, (B, T)).astype(np.float32).astype(np.float64)
    outs = [_outs(fb.update_command(torch.as_tensor(cmd, device="cuda"))) for fb in hs]
    check(*outs, "interface", "update", yaw_of=cmd)
    for fb in hs:
        fb.close()


# ---- 4. warm-up of the in-kernel auto-reset ----------------------------------------------------------------------------
@pytest.mark.parametrize("T,W", [(7, 1), (12, 2), (32, 4), (80, 8)])
def test_autoreset_finish_matches_fp64(cuda_device, wide_band, T, W):
    """A truncating step with auto-reset armed, then autoreset_finish (a warm-up solve at the drawn winds): the strict FP32
    handle's state equals its FP64 twin's, its flagged rows are the twin's rounded to float32 and the clamped oracle's."""
    import torch

    from wfcrl_b200.backend import FlorisBatch

    B = 512
    assert _resolve_warps(T, B) == W
    lx, ly = _grid(T, True)  # rows along the wind: the sampler's ordinary winds leave wakes to flag
    hs = [FlorisBatch(lx, ly, B, precision=p, kernel="fast", max_iter=3) for p in ("f32", "f64")]
    rng = np.random.default_rng(40 + T)
    ws, wd = _winds(rng, B)
    for fb in hs:
        fb.reset(ws, wd, host_trig=True)
        fb.set_autoreset(True, seed=5)
    ep = np.zeros(B)
    for k in range(2):  # max_iter = 3 with the warm-up solve: the second step truncates
        a = torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda")
        o32 = _outs(hs[0].step(a))
        hs[1].step(a)
        torch.cuda.synchronize()
        r32 = _np(o32["reward"])
        assert _np(o32["truncated"]).any() == (k == 1), k
        if k == 1:
            assert _np(o32["truncated"]).all()
            assert np.array_equal(hs[0].get_state("fin_sum"), ep + r32)
        ep += r32
    outs = [_outs(fb.autoreset_finish()) for fb in hs]
    torch.cuda.synchronize()
    for name in ("yaw", "acc", "acc_prev", "num_iter", "num_moves", "episode", "ws", "wd", "ws_norm", "ep_return", "ep_len",
                 "fin_n", "fin_len", "order", "shaper_ref"):
        assert np.array_equal(hs[0].get_state(name), hs[1].get_state(name)), name
    flag = hs[0].get_state("ambiguous").astype(bool)
    _enough(flag.sum(), B // 16, ("autoreset", T))
    _assert_rows(outs[0], outs[1], flag, "env", "autoreset")
    assert np.array_equal(_np(outs[0]["freewind"]), _np(outs[1]["freewind"]).astype(np.float32))
    rows = _pick(np.random.default_rng(T), np.flatnonzero(flag))
    # the drawn winds were rotated with the device's cosd / sind, which the state keeps
    ws2, wd2, cs2 = (hs[1].get_state(name)[rows] for name in ("ws", "wd", "cs"))
    _oracle_check({k: outs[0][k][torch.as_tensor(rows, device="cuda")] for k in PER_TURBINE}, lx, ly, ws2, wd2,
                  np.zeros((len(rows), T)), "env", "autoreset", warmup=True, order=hs[0].get_state("order")[rows], cs=cs2)
    for fb in hs:
        fb.close()


# ---- 5. the evaluation re-solve at every width -------------------------------------------------------------------------
# (W, B, K of evaluate_yaw / evaluate_actions, K of evaluate_rollouts with H = 4); B * K * H selects W on 80 turbines
EVAL_CASES = [(8, 256, 8, 2), (4, 1024, 12, 3), (2, 1024, 24, 6), (1, 1024, 40, 10)]
H = 4


@pytest.mark.parametrize("W,B,K,KR", EVAL_CASES)
def test_evaluation_resolve_matches_fp64(cuda_device, wide_band, W, B, K, KR):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layout("HornsRev1_")
    T = len(lx)
    assert _resolve_warps(T, B * K) == W and _resolve_warps(T, B * KR * H) == W
    hs = [FlorisBatch(lx, ly, B, precision=p, kernel="fast", max_iter=50, reward_shaper="reference",
                      shaper_reference=0.5) for p in ("f32", "f64")]
    rng = np.random.default_rng(50 + W)
    ws, wd = _winds(rng, B)
    a = torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda")
    for fb in hs:
        fb.reset(ws, wd, host_trig=True)
        fb.step(a)  # a yaw state away from 0
    sub = np.random.default_rng(W)

    # evaluate_yaw: power of every candidate yaw setting (interface units)
    yaw = torch.as_tensor(rng.uniform(-30, 30, (B, K, T)).astype(np.float32).astype(np.float64), device="cuda")
    e32, e64 = (_outs(fb.evaluate_yaw(yaw)) for fb in hs)
    torch.cuda.synchronize()
    flag = e32["ambiguous"].cpu().numpy()
    _enough(flag.sum(), B * K // 2, ("evaluate_yaw", W))
    _assert_f32_of(_np(e32["power"])[flag], _np(e64["power"])[flag], FLOORS["interface"]["power"], "evaluate_yaw")
    b, k = np.nonzero(flag)
    pick = _pick(sub, np.arange(len(b)))
    b, k = b[pick], k[pick]
    ref, _ = _oracle(lx, ly, ws[b], wd[b], yaw.cpu().numpy()[b, k], "interface")
    _assert_f32_of(_np(e32["power"])[b, k], ref["power"], FLOORS["interface"]["power"], ("evaluate_yaw", "oracle"))

    # evaluate_actions (H = 1) and evaluate_rollouts (H = 4): every step output of every flagged row
    for name, shape in (("evaluate_actions", (B, K, T)), ("evaluate_rollouts", (B, KR, H, T))):
        act = torch.as_tensor(rng.uniform(-5, 5, shape).astype(np.float32), device="cuda")
        e32, e64 = (_outs(getattr(fb, name)(act)) for fb in hs)
        torch.cuda.synchronize()
        flag = e32["ambiguous"].cpu().numpy()
        _enough(flag.sum(), flag.size // 2, (name, W))
        if name == "evaluate_rollouts":
            _enough(flag[:, :, 1:].sum(), flag[:, :, 1:].size // 2, (name, "h > 0", W))
        _assert_rows(e32, e64, flag, "env", name)
        r32, r64 = _np(e32["reward"])[flag], _np(e64["reward"])[flag]
        assert np.all(np.abs(r32 - r64) <= _ulp32(r64)), name
        for key in ("truncated", "freewind", "yaw"):
            assert np.array_equal(_np(e32[key]), _np(e64[key]).astype(np.float32)), (name, key)
        idx = np.argwhere(flag)
        idx = idx[_pick(sub, np.arange(len(idx)))]
        rows = tuple(idx.T)
        bb = idx[:, 0]
        _oracle_check({key: _np(e32[key])[rows] for key in PER_TURBINE}, lx, ly, ws[bb], wd[bb], _np(e64["yaw"])[rows],
                      "env", (name, "oracle"), order=hs[0].get_state("order")[bb])
    for fb in hs:
        fb.close()


# ---- 6. the staged host path past its record capacity ------------------------------------------------------------------
@pytest.mark.parametrize("route", ["staged", "zero_copy"])
def test_host_path_with_more_resolved_envs_than_records(cuda_device, wide_band, route):
    """2048 envs, most at low winds: more envs are re-solved than the staged path keeps records for (1024), so it copies
    their rows from the device arrays.  The zero-copy route (pinned action and outputs, mapped into one step launch and its
    re-solve) has the re-solve write its rows straight into host memory.  Either route must equal the device-resident step
    bit for bit."""
    import torch

    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layout("Turb32_Row5_")
    B, T = 2048, len(lx)
    rng = np.random.default_rng(60)
    ws, wd = _winds(rng, B, low_frac=0.9)
    dev, host = (FlorisBatch(lx, ly, B, precision="f32", kernel="fast", max_iter=100) for _ in range(2))
    for fb in (dev, host):
        fb.reset(ws, wd, host_trig=True)
    wide_band.setenv("WFCRL_B200_HOST_PATH", route)
    for k in range(3):
        a = rng.uniform(-2, 2, (B, T)).astype(np.float32)
        want = dev.step(torch.as_tensor(a, device="cuda"))
        n0 = host.launch_count()
        got = host.step_host(torch.as_tensor(a).pin_memory())  # a pageable buffer would send zero_copy down the staged route
        torch.cuda.synchronize()
        # zero-copy: one step launch and the re-solve; staged: one step launch per chunk of envs and the re-solve
        assert host.launch_count() - n0 == (2 if route == "zero_copy" else 7), (k, route)
        resolved = host.get_state("ambiguous")
        _enough(resolved.sum(), 1025, ("host", route, k))
        assert np.array_equal(resolved, dev.get_state("ambiguous")), k
        for key, v in want.items():
            assert torch.equal(v.cpu(), got[key]), (k, key)
    for name in ("yaw", "ep_return", "num_iter", "acc"):
        assert np.array_equal(dev.get_state(name), host.get_state(name)), name
    dev.close()
    host.close()
