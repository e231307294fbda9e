"""serial_refine on the GPU: the same choices as the oracle restatement (oracle/yaw_sr.py) in FP64, a result consistent with
the evaluation, gains where wake steering pays, batch independence, and the strict FP32 result judged in FP64."""
import numpy as np
import pytest

from tests._util import layout

pytestmark = pytest.mark.gpu


def _winds(n, seed):
    rng = np.random.default_rng(seed)
    ws = rng.uniform(6.0, 11.0, n)
    wd = np.clip(rng.normal(270.0, 12.0, n), 0.0, 360.0)
    ws[0], wd[0] = 8.0, 270.0
    return ws, wd


def _batch(lx, ly, ws, wd, precision, **kw):
    from wfcrl_b200.backend import FlorisBatch

    fb = FlorisBatch(lx, ly, len(ws), precision=precision, kernel="fast", max_iter=1000, **kw)
    fb.reset(ws, wd, host_trig=True)
    return fb


@pytest.mark.parametrize("name", ["Turb6_Row2_", "Ablaincourt_", "Turb32_Row5_"])
def test_fp64_matches_the_oracle_restatement(cuda_device, name):
    from oracle import yaw_sr
    from wfcrl_b200.yaw_optimization import serial_refine

    lx, ly = layout(name)
    ws, wd = _winds(16, seed=len(lx))
    fb = _batch(lx, ly, ws, wd, "f64")
    got = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in serial_refine(fb).items()}
    ref = yaw_sr.serial_refine(lx, ly, ws, wd)
    assert got["evaluations"] == 1 + len(lx) * 15
    compared = ref["min_gap"] >= 1e-9  # near-ties may go either way at the solver's 1e-12
    assert compared.mean() >= 0.9, ref["min_gap"]
    assert np.array_equal(got["yaw"][compared], ref["yaw"][compared])
    for key in ("farm_power", "start_power"):
        assert np.max(np.abs(got[key] - ref[key]) / ref[key]) <= 1e-9, key
    fb.close()


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_consistency_and_gain(cuda_device, precision):
    import torch

    from wfcrl_b200.yaw_optimization import farm_power, serial_refine

    for name in ("Turb6_Row2_", "Turb32_Row5_"):
        lx, ly = layout(name)
        ws, wd = _winds(16, seed=1)
        fb = _batch(lx, ly, ws, wd, precision)
        res = serial_refine(fb, passes=(5, 3))
        assert bool((res["farm_power"] >= res["start_power"]).all())
        again = farm_power(fb.evaluate_yaw(res["yaw"][:, None, :].contiguous())["power"][:, 0])
        assert torch.equal(again, res["farm_power"])
        assert float(res["farm_power"][0]) > float(res["start_power"][0]), name  # 8 m/s, 270 deg
        assert bool((res["yaw"].abs() <= 40.0).all())
        fb.close()


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_batch_independence(cuda_device, precision):
    import torch

    from wfcrl_b200.backend import FlorisBatch
    from wfcrl_b200.yaw_optimization import serial_refine

    small, big = layout("Turb6_Row2_"), layout("Turb32_Row5_")
    n = len(small[0])
    ws, wd = _winds(24, seed=4)
    handles = [_batch(*small, ws[i:i + 1], wd[i:i + 1], precision) for i in (0, 5)]
    alone = [serial_refine(fb, passes=(5, 3)) for fb in handles]
    handles.append(_batch(*small, ws, wd, precision))
    batch = serial_refine(handles[-1], passes=(5, 3))
    pool = FlorisBatch(*big, len(ws), precision=precision, kernel="fast", max_iter=1000)
    handles.append(pool)
    pool.set_mixed_layouts([small[0], big[0]], [small[1], big[1]])
    ids = np.arange(len(ws)) % 2
    ids[[0, 5]] = 0
    pool.assign_layouts(None, ids)
    pool.reset(ws, wd, host_trig=True)
    mixed = serial_refine(pool, passes=(5, 3))
    for j, i in enumerate((0, 5)):
        for other in (batch, mixed):
            assert torch.equal(other["yaw"][i, :n], alone[j]["yaw"][0]), (precision, i)
            assert torch.equal(other["farm_power"][i], alone[j]["farm_power"][0]), (precision, i)
        assert not bool(mixed["yaw"][i, n:].any())
    for fb in handles:
        fb.close()


def test_through_a_vector_env(cuda_device):
    """serial_refine(env) on a VecWindFarmEnv goes through env.backend, takes the env's yaw control bounds and leaves the
    env where it was."""
    import torch

    from wfcrl_b200 import environments as envs
    from wfcrl_b200.yaw_optimization import serial_refine

    B = 8
    env = envs.make_vec("Turb6_Row2_Floris", B, precision="f64", controls={"yaw": (-30, 30, 5)}, max_num_steps=50)
    env.reset(seed=3)
    env.step(torch.as_tensor(np.random.default_rng(3).uniform(-5, 5, (B, 6)).astype(np.float32), device=env.device))
    torch.cuda.synchronize()
    names = ("yaw", "acc", "num_iter", "num_moves", "ep_return", "ws", "wd", "ambiguous")
    before = {k: env.backend.get_state(k).tobytes() for k in names}
    res = serial_refine(env, passes=(5, 3))
    torch.cuda.synchronize()
    assert all(env.backend.get_state(k).tobytes() == before[k] for k in names)
    assert bool((res["yaw"].abs() <= 30.0).all())
    assert bool((res["farm_power"] >= res["start_power"]).all())
    explicit = serial_refine(env.backend, passes=(5, 3), bounds=(-30.0, 30.0))
    for key in ("yaw", "farm_power", "start_power"):
        assert torch.equal(res[key], explicit[key]), key
    env.close()


def test_fp32_strict_result_judged_in_fp64(cuda_device):
    from wfcrl_b200.yaw_optimization import farm_power, serial_refine

    lx, ly = layout("Turb32_Row5_")
    ws, wd = _winds(16, seed=9)
    fb64, fb32 = _batch(lx, ly, ws, wd, "f64"), _batch(lx, ly, ws, wd, "f32")
    opt64, opt32 = serial_refine(fb64), serial_refine(fb32)
    p32 = farm_power(fb64.evaluate_yaw(opt32["yaw"][:, None, :].contiguous())["power"][:, 0])
    zero64 = opt64["start_power"]
    assert bool((p32 >= zero64 * (1.0 - 1e-4)).all())
    gap = ((opt64["farm_power"] - p32) / opt64["farm_power"]).cpu().numpy()
    print("FP32-strict optimum vs FP64 optimum, relative gap: min %.3g median %.3g max %.3g" %
          (gap.min(), np.median(gap), gap.max()))
