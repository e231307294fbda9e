"""CPU tests of the ``pad_turbines`` argument (layout pools of mixed turbine counts): the cases it does not cover are
refused before any device work, and the layouts must still share ``dt`` and ``t_init``."""
import pytest


def test_pad_turbines_accepts_mixed_counts_before_device_work():
    from wfcrl_b200.vector_env import layout_pool

    cases = layout_pool(["Turb1_Row1_", "Ablaincourt_", "HornsRev1_"], pad_turbines=True)
    assert [c["num_turbines"] for c in cases] == [1, 7, 80]
    with pytest.raises(ValueError, match="num_turbines"):
        layout_pool(["Turb1_Row1_", "Ablaincourt_"])


def test_decentralised_ids_are_refused():
    from wfcrl_b200 import environments as envs

    with pytest.raises(ValueError, match="pad_turbines"):
        envs.make_vec(["Dec_Turb6_Row1_Floris", "Dec_Ablaincourt_Floris"], 4, pad_turbines=True)
    with pytest.raises(ValueError, match="pad_turbines"):
        envs.make_vec("Dec_Ablaincourt_Floris", 4, pad_turbines=True)


def test_multi_agent_class_is_refused():
    from wfcrl_b200.vector_env import VecMAWindFarmEnv, VecWindFarmEnv

    with pytest.raises(ValueError, match="pad_turbines"):
        VecMAWindFarmEnv(["Turb6_Row1_", "Ablaincourt_"], 4, pad_turbines=True)
    with pytest.raises(ValueError, match="pad_turbines"):
        VecWindFarmEnv(["Turb6_Row1_", "Ablaincourt_"], 4, pad_turbines=True, multi_agent=True)


def test_mismatched_dt_and_t_init_are_still_refused():
    from wfcrl_b200.layouts import get_layout
    from wfcrl_b200.vector_env import VecWindFarmEnv

    a = get_layout("Ablaincourt_")
    b = get_layout("Turb6_Row1_")
    with pytest.raises(ValueError, match="dt"):
        VecWindFarmEnv([a, dict(b, dt=30)], 4, pad_turbines=True)
    with pytest.raises(ValueError, match="t_init"):
        VecWindFarmEnv([a, dict(b, t_init=120)], 4, pad_turbines=True)


def test_without_the_flag_mixed_counts_are_refused():
    from wfcrl_b200 import environments as envs

    with pytest.raises(ValueError, match="num_turbines"):
        envs.make_vec(["Turb6_Row2_Floris", "Ablaincourt_Floris"], 4, pad_turbines=False)
