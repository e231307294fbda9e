"""CPU tests of the layout pool's Python front end: batches over several farms are refused before any device work when
their layouts cannot share one handle."""
import numpy as np
import pytest


def test_env_ids_of_different_turbine_counts_are_refused():
    from wfcrl_b200 import environments as envs

    with pytest.raises(ValueError, match="num_turbines"):
        envs.make_vec(["Turb6_Row2_Floris", "Ablaincourt_Floris"], 4)


def test_centralised_and_decentralised_ids_are_refused():
    from wfcrl_b200 import environments as envs

    with pytest.raises(ValueError, match="Dec_"):
        envs.make_vec(["Turb6_Row2_Floris", "Dec_Turb6_Row1_Floris"], 4)


def test_layout_sampling_with_a_time_series_is_refused():
    from wfcrl_b200.vector_env import VecWindFarmEnv

    series = np.array([[8.0, 270.0], [9.0, 260.0]])
    with pytest.raises(ValueError, match="time-series"):
        VecWindFarmEnv(["Turb6_Row2_", "Turb6_Row1_"], 4, wind_time_series=series, layout_assignment="sample")


def test_layouts_must_share_dt_and_t_init():
    from wfcrl_b200.layouts import get_layout
    from wfcrl_b200.vector_env import VecWindFarmEnv

    a = get_layout("Turb6_Row2_")
    b = dict(get_layout("Turb6_Row1_"), dt=30)
    with pytest.raises(ValueError, match="dt"):
        VecWindFarmEnv([a, b], 4)
    with pytest.raises(ValueError, match="t_init"):
        VecWindFarmEnv([a, dict(a, t_init=120)], 4)
    with pytest.raises(ValueError, match="layout_assignment"):
        VecWindFarmEnv([a, a], 4, layout_assignment="random")
