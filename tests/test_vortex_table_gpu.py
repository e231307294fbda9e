"""The FP64 warp-per-env kernels evaluate the transverse (vortex) velocities either directly from the positions or through
the per-env vortex table built at reset (wf_vortex_table_kernel; DESIGN.md section 5).  Both routes must reproduce the oracle;
x-ties (wd = 270 on the row layouts) always take the direct route inside a table-enabled launch.  On an FP64 handle the
table route is the gather form of the step kernel and the direct route its scatter form.  The FP32 step kernel always
evaluates directly; on a strict FP32 handle the two routes are those of the FP64 re-solve of the flagged envs, which reads
source-major double rows."""
import numpy as np
import pytest

from tests._util import host_trig, layout, rel_err, sample_winds

pytestmark = pytest.mark.gpu


def _solve(name, precision, B, seed, monkeypatch, table):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    if table:  # FP64 and strict FP32 handles build the table by default
        monkeypatch.delenv("WFCRL_B200_NO_VTAB", raising=False)
    else:
        monkeypatch.setenv("WFCRL_B200_NO_VTAB", "1")
    lx, ly = layout(name)
    T = len(lx)
    ws, wd = sample_winds(B, seed, tie_every=4)
    rng = np.random.default_rng(seed + 1)
    yaw = rng.uniform(-40, 40, (B, T)).astype(np.float32).astype(np.float64)
    yaw[1] = 0.0
    yaw[2, ::2] = 0.0
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=10)
    fb.reset(ws, wd, host_trig=True, warmup_solves=0)
    out = fb.update_command(torch.as_tensor(yaw, device="cuda"))
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in out.items()}
    fb.close()
    return got, (lx, ly, ws, wd, yaw)


@pytest.mark.parametrize("name", ["Turb6_Row2_", "Turb32_Row5_", "Turb_TCRWP_", "HornsRev1_"])
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_table_and_direct_routes_match_oracle(cuda_device, monkeypatch, name, precision):
    from oracle import c_oracle

    B = 32
    tab, (lx, ly, ws, wd, yaw) = _solve(name, precision, B, 21, monkeypatch, table=True)
    direct, _ = _solve(name, precision, B, 21, monkeypatch, table=False)
    c, s = host_trig(wd)
    ref = c_oracle.solve_batch(lx, ly, ws, wd, yaw, cs=np.stack([c, s], 1))
    tol = 1e-9 if precision == "f64" else 1e-4
    loads_ref = np.stack([ref["ti"], ref["std_u"], ref["std_v"], ref["std_w"]], -1) * 1e7
    for got in (tab, direct):
        assert rel_err(got["power"], ref["power_W"], 1.0) <= tol
        assert rel_err(got["wind_speed"], ref["ws_local"], 1e-3) <= tol
        assert rel_err(got["wind_direction"], ref["wd_local"], 1.0) <= tol
        assert rel_err(got["load"], loads_ref, 1e4) <= (tol if precision == "f64" else 2e-3)
    # the two routes agree with each other far inside the tolerance
    assert rel_err(tab["power"], direct["power"], 1.0) <= (1e-11 if precision == "f64" else 2e-5)


def test_moving_wind_falls_back_to_direct_route(cuda_device):
    """wf_update_wind every step (time-series mode) leaves the table stale: the step must not use it."""
    import torch

    from oracle import c_oracle
    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layout("Turb16_TCRWP_")
    B, T = 8, len(lx)
    ws, wd = sample_winds(B, 5)
    fb = FlorisBatch(lx, ly, B, precision="f64", kernel="fast", max_iter=50)
    fb.reset(ws, wd, host_trig=True, warmup_solves=0)
    rng = np.random.default_rng(9)
    for step in range(12):
        ws2 = np.clip(ws + rng.normal(0, 0.3, B), 3, 28)
        wd2 = (wd + rng.normal(0, 3.0, B)) % 360
        fb.update_wind(torch.as_tensor(ws2, device="cuda"), torch.as_tensor(wd2, device="cuda"), host_trig=True)
        yaw = rng.uniform(-30, 30, (B, T)).astype(np.float32).astype(np.float64)
        out = fb.update_command(torch.as_tensor(yaw, device="cuda"))
        torch.cuda.synchronize()
        c, s = host_trig(wd2)
        ref = c_oracle.solve_batch(lx, ly, ws2, wd2, yaw, cs=np.stack([c, s], 1))
        assert rel_err(out["power"].cpu().numpy(), ref["power_W"], 1.0) <= 1e-9, step
    fb.close()
