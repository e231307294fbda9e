"""CPU tests of the serial-refine yaw optimiser: its schedule, restated on the C oracle (oracle/yaw_sr.py), and the argument
validation of wfcrl_b200.yaw_optimization.serial_refine (which happens before any device work)."""
import numpy as np
import pytest

from tests._util import layout


def test_schedule_on_the_oracle():
    from oracle import yaw_sr

    lx, ly = layout("Turb6_Row2_")
    ws, wd = np.array([8.0, 9.5, 7.0]), np.array([270.0, 262.0, 281.0])
    res = yaw_sr.serial_refine(lx, ly, ws, wd, passes=(5, 3), bounds=(-30.0, 30.0))
    T = len(lx)
    assert res["choices"].shape == (3, 2 * T)
    assert np.all(res["farm_power"] >= res["start_power"])  # monotone by construction
    assert res["farm_power"][0] > res["start_power"][0]  # wake steering pays in the aligned row at 270 deg
    assert np.all(np.abs(res["yaw"]) <= 30.0)
    # every value is on the grid the schedule allows: pass 0 on linspace(-30, 30, 5), pass 1 a step of 0 or +-15
    allowed = {a + d for a in np.linspace(-30.0, 30.0, 5) for d in (-15.0, 0.0, 15.0)}
    assert set(np.unique(res["yaw"])) <= {v for v in allowed if -30.0 <= v <= 30.0} | {0.0}
    # the returned power is the power of the returned yaw
    from oracle import c_oracle

    cs = [(np.cos(np.radians((w - 270.0) % 360.0)), np.sin(np.radians((w - 270.0) % 360.0))) for w in wd]
    out = c_oracle.solve_batch(lx, ly, ws, wd, res["yaw"], cs=cs)
    assert np.array_equal(yaw_sr.farm_power(out["power_W"]), res["farm_power"])


def test_start_is_zero_clipped_into_the_bounds():
    from oracle import yaw_sr

    lx, ly = layout("Turb6_Row2_")
    res = yaw_sr.serial_refine(lx, ly, [8.0], [270.0], passes=(2,), bounds=(5.0, 20.0))
    assert np.all((res["yaw"] >= 5.0) & (res["yaw"] <= 20.0))
    from oracle import c_oracle

    out = c_oracle.solve_batch(lx, ly, [8.0], [270.0], np.full((1, len(lx)), 5.0), cs=[(1.0, 0.0)])
    assert np.array_equal(yaw_sr.farm_power(out["power_W"]), res["start_power"])


@pytest.mark.parametrize("passes,exc", [((), ValueError), ((5, 1), ValueError), ((0,), ValueError), (5, TypeError)])
def test_serial_refine_rejects_bad_passes(passes, exc):
    from wfcrl_b200.yaw_optimization import serial_refine

    with pytest.raises(exc):
        serial_refine(object(), passes=passes)


@pytest.mark.parametrize("bounds", [(5.0, -5.0), (1.0, 1.0), (float("nan"), 10.0), (-40.0, float("inf"))])
def test_serial_refine_rejects_bad_bounds(bounds):
    from wfcrl_b200.yaw_optimization import serial_refine

    with pytest.raises(ValueError):
        serial_refine(object(), bounds=bounds)


def test_serial_refine_needs_a_batch():
    from wfcrl_b200.yaw_optimization import serial_refine

    with pytest.raises(TypeError):
        serial_refine(object())

