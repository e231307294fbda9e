"""Candidate evaluation (wf_evaluate_yaw / FlorisBatch.evaluate_yaw): K yaw settings per env solved in the env's current
wind without changing the handle's state.  Candidate (b, k) must equal, bit for bit, the power row of wf_update_command with
that yaw on the same handle in the same state, and nothing a step or get_state can see may change."""
import ctypes as C

import numpy as np
import pytest

from tests._util import layout, sample_winds

pytestmark = pytest.mark.gpu

# (precision, strict, vortex table)
MODES = {
    "f64_table": ("f64", True, True),
    "f64_direct": ("f64", True, False),
    "f32_strict": ("f32", True, True),
    "f32_relaxed": ("f32", False, True),
}
STATE = ("yaw", "acc", "acc_prev", "num_iter", "num_moves", "nonfinite", "episode", "ambiguous", "ep_return", "ep_len",
         "fin_sum", "fin_sumsq", "fin_n", "fin_len", "ws", "wd", "ws_norm", "shaper_ref", "ti_ambient", "order", "xs", "ys",
         "xi", "yi", "cs", "layout_id", "turbine_count")


def _table(monkeypatch, table):
    if table:
        monkeypatch.delenv("WFCRL_B200_NO_VTAB", raising=False)
    else:
        monkeypatch.setenv("WFCRL_B200_NO_VTAB", "1")


def _check_against_interface(fb, yaw, strict_f32):
    """The reference loop: state_dict -> update_command(yaw[:, k]) -> power -> load_state_dict, with an evaluation in the
    same state before each update_command (load_state_dict leaves the vortex table stale: both routes are covered)."""
    import torch

    K = yaw.shape[1]
    flagged = 0
    for k in range(K):
        ev = fb.evaluate_yaw(yaw)
        power, amb = ev["power"].clone(), ev["ambiguous"].clone()
        sd = fb.state_dict()
        out = fb.update_command(yaw[:, k].contiguous())
        torch.cuda.synchronize()
        assert torch.equal(power[:, k], out["power"]), k
        ref_amb = fb.get_state("ambiguous").astype(bool)
        if strict_f32:
            assert np.array_equal(amb[:, k].cpu().numpy(), ref_amb), k
            flagged += int(ref_amb.sum())
        else:
            assert not bool(amb.any())
        fb.load_state_dict(sd)
    return flagged


@pytest.mark.parametrize("K", [1, 7])
@pytest.mark.parametrize("name", ["Ablaincourt_", "Turb32_Row5_", "HornsRev1_"])
@pytest.mark.parametrize("mode", list(MODES))
def test_equals_interface_mode(cuda_device, monkeypatch, mode, name, K):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table = MODES[mode]
    _table(monkeypatch, table)
    lx, ly = layout(name)
    T, B = len(lx), 64
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, strict=strict)
    ws, wd = sample_winds(B, seed=T + K, tie_every=5)
    fb.reset(ws, wd, host_trig=True)
    yaw = torch.as_tensor(np.random.default_rng(K).uniform(-40, 40, (B, K, T)), device="cuda")
    _check_against_interface(fb, yaw, precision == "f32" and strict)
    fb.close()


def test_strict_flagged_candidates_equal_the_resolve(cuda_device):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layout("Turb32_Row5_")
    T, B, K = len(lx), 512, 4
    rng = np.random.default_rng(3)
    ws, wd = sample_winds(B, seed=3)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # over-sample the foot of the power curve
    fb = FlorisBatch(lx, ly, B, precision="f32", kernel="fast", max_iter=1000)
    fb.reset(ws, wd, host_trig=True)
    yaw = torch.as_tensor(rng.uniform(-40, 40, (B, K, T)), device="cuda")
    amb = fb.evaluate_yaw(yaw)["ambiguous"].clone()
    assert int(amb.sum()) > 0
    assert _check_against_interface(fb, yaw, True) == int(amb.sum())
    fb.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_state_untouched(cuda_device, monkeypatch, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table = MODES[mode]
    _table(monkeypatch, table)
    lx, ly = layout("Turb32_Row5_")
    T, B, K = len(lx), 512, 3
    rng = np.random.default_rng(8)
    ws, wd = sample_winds(B, seed=8)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # a strict handle flags envs at the foot of the power curve
    kw = dict(precision=precision, kernel="fast", max_iter=20, strict=strict, reward_shaper="step")
    twins = [FlorisBatch(lx, ly, B, **kw) for _ in range(2)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
        fb.set_autoreset(True, seed=5)
    acts = [torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda") for _ in range(4)]
    for fb in twins:
        fb.step(acts[0])
    torch.cuda.synchronize()
    if precision == "f32":
        assert twins[0].get_state("ambiguous").sum() > 0  # the previous step re-solved envs
    before = {name: twins[0].get_state(name).tobytes() for name in STATE}
    yaw = torch.as_tensor(rng.uniform(-40, 40, (B, K, T)), device="cuda")
    twins[0].evaluate_yaw(yaw)
    torch.cuda.synchronize()
    for name in STATE:
        assert twins[0].get_state(name).tobytes() == before[name], name
    for act in acts[1:]:
        outs = [{k: v.clone() for k, v in fb.step(act).items()} for fb in twins]
        twins[0].evaluate_yaw(yaw)
        torch.cuda.synchronize()
        for key in outs[0]:
            assert torch.equal(outs[0][key], outs[1][key]), key
        for name in STATE:
            assert np.array_equal(twins[0].get_state(name), twins[1].get_state(name)), name
    for fb in twins:
        fb.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_first_call_on_a_non_blocking_stream(cuda_device, monkeypatch, mode):
    """The first call allocates and zeroes the scratch (the re-solve counters, the gather rows); issued on a side stream
    that does not wait for the legacy default stream, its results still equal a call on the default stream."""
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table = MODES[mode]
    _table(monkeypatch, table)
    lx, ly = layout("Turb32_Row5_")
    T, B, K = len(lx), 1024, 5
    rng = np.random.default_rng(12)
    ws, wd = sample_winds(B, seed=12)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # flagged candidates on a strict handle
    twins = [FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, strict=strict) for _ in range(2)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
    yaw = torch.as_tensor(rng.uniform(-40, 40, (B, K, T)), device="cuda")
    ref = {k: v.clone() for k, v in twins[1].evaluate_yaw(yaw).items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = {k: v.clone() for k, v in twins[0].evaluate_yaw(yaw).items()}
    torch.cuda.synchronize()
    if precision == "f32":
        assert int(ref["ambiguous"].sum()) > 0
    for key in ref:
        assert torch.equal(got[key], ref[key]), key
    for fb in twins:
        fb.close()


@pytest.mark.parametrize("precision,strict", [("f64", True), ("f32", True)])
def test_mixed_pool_padding(cuda_device, monkeypatch, precision, strict):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    monkeypatch.delenv("WFCRL_B200_NO_VTAB", raising=False)
    farms = [layout("Ablaincourt_"), layout("Turb32_Row5_")]
    counts = [len(f[0]) for f in farms]
    T, B, K = max(counts), 128, 5
    kw = dict(precision=precision, kernel="fast", max_iter=1000, strict=strict)
    pool = FlorisBatch(*farms[-1], B, **kw)
    pool.set_mixed_layouts([f[0] for f in farms], [f[1] for f in farms])
    ids = np.arange(B) % 2
    pool.assign_layouts(None, ids)
    refs = [FlorisBatch(lx, ly, B, **kw) for lx, ly in farms]
    ws, wd = sample_winds(B, seed=2)
    for fb in [pool] + refs:
        fb.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(2)
    yaw = rng.uniform(-40, 40, (B, K, T))
    for b in range(B):
        yaw[b, :, counts[ids[b]]:] = np.nan  # ignored
    power = pool.evaluate_yaw(torch.as_tensor(yaw, device="cuda"))["power"].clone()
    torch.cuda.synchronize()
    for lay, n in enumerate(counts):
        rows = torch.as_tensor(np.flatnonzero(ids == lay), device="cuda")
        assert not bool(power[rows][:, :, n:].any())
        for k in range(K):
            out = refs[lay].update_command(torch.as_tensor(np.ascontiguousarray(yaw[:, k, :n]), device="cuda"))
            assert torch.equal(power[rows, k, :n], out["power"][rows]), (lay, k)
    for fb in [pool] + refs:
        fb.close()


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_multi_agent_handle(cuda_device, precision):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layout("Turb6_Row2_")
    T, B, K = len(lx), 64, 4
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, multi_agent=True)
    ws, wd = sample_winds(B, seed=6)
    fb.reset(ws, wd, host_trig=True)
    fb.step(torch.as_tensor(np.random.default_rng(0).uniform(-5, 5, (B, T)).astype(np.float32), device="cuda"))
    yaw = torch.as_tensor(np.random.default_rng(1).uniform(-40, 40, (B, K, T)), device="cuda")
    _check_against_interface(fb, yaw, precision == "f32")
    fb.close()


def test_launch_count_and_refusals(cuda_device):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layout("Turb6_Row2_")
    T, B = len(lx), 64
    yaw = torch.zeros(B, 3, T, dtype=torch.float64, device="cuda")
    for precision, strict, launches in (("f64", True, 1), ("f32", True, 2), ("f32", False, 1)):
        fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, strict=strict)
        fb.evaluate_yaw(yaw)  # (allocates the scratch)
        for K in (3, 1, 2):
            n0 = fb.launch_count()
            fb.evaluate_yaw(yaw[:, :K].contiguous())
            assert fb.launch_count() - n0 == launches, (precision, strict, K)
        lib, h, st = fb.lib, fb.handle, fb._stream()
        p = C.c_void_p(yaw.data_ptr())
        out = torch.zeros(B * 8 * T, dtype=torch.float64, device="cuda")
        q = C.c_void_p(out.data_ptr())
        n0 = fb.launch_count()
        assert lib.wf_evaluate_yaw(h, p, 0, q, None, st) == 1 and b"K" in lib.wf_last_error()
        assert lib.wf_evaluate_yaw(h, p, -1, q, None, st) == 1
        assert lib.wf_evaluate_yaw(h, None, 1, q, None, st) == 1 and b"NULL" in lib.wf_last_error()
        assert lib.wf_evaluate_yaw(h, p, 1, None, None, st) == 1
        assert lib.wf_evaluate_yaw(h, p, 2**31 // B + 1, q, None, st) == 1 and b"2^31" in lib.wf_last_error()
        assert fb.launch_count() == n0
        with pytest.raises(ValueError):
            fb.evaluate_yaw(torch.zeros(B, 0, T, dtype=torch.float64, device="cuda"))
        with pytest.raises(TypeError):
            fb.evaluate_yaw(yaw.float())
        fb.close()
    basic = FlorisBatch(lx, ly, B, precision="f64", kernel="basic", max_iter=1000)
    n0 = basic.launch_count()
    with pytest.raises(Exception, match="WF_KERNEL_FAST"):
        basic.evaluate_yaw(yaw)
    assert basic.launch_count() == n0
    basic.close()
    grid5 = FlorisBatch(lx, ly, B, precision="f64", kernel="basic", max_iter=1000,
                        config_overrides={"turbine_grid_points": 5})
    with pytest.raises(Exception, match="WF_KERNEL_FAST"):
        grid5.evaluate_yaw(yaw)
    grid5.close()
