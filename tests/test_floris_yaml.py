"""The FLORIS input file the reference passes to its backend (wfcrl/interface.py:462-479): parsed into layout, wind and
WfConfig overrides; unsupported model selections are refused, never ignored."""
import copy
import os

import numpy as np
import pytest
import yaml

from wfcrl_b200.floris_yaml import load_floris_yaml, parse_floris_config

# same schema as the reference's template (wfcrl/simulators/floris/inputs/template/case.yaml), different numbers
CASE = {
    "name": "GCH", "floris_version": "v3.0.0",
    "solver": {"type": "turbine_grid", "turbine_grid_points": 3},
    "farm": {"layout_x": [0.0, 700.0, 1400.0, 350.0], "layout_y": [0.0, 50.0, -30.0, 600.0], "turbine_type": ["nrel_5MW"]},
    "flow_field": {"air_density": 1.2, "reference_wind_height": -1, "turbulence_intensity": 0.08, "wind_directions": [262.0],
                   "wind_shear": 0.14, "wind_speeds": [9.5], "wind_veer": 0.0},
    "wake": {
        "model_strings": {"combination_model": "sosfs", "deflection_model": "gauss", "turbulence_model": "crespo_hernandez",
                          "velocity_model": "gauss"},
        "enable_secondary_steering": True, "enable_yaw_added_recovery": True, "enable_transverse_velocities": True,
        "wake_deflection_parameters": {"gauss": {"ad": 0.0, "alpha": 0.58, "bd": 0.0, "beta": 0.077, "dm": 1.0, "ka": 0.38,
                                                 "kb": 0.004}, "jimenez": {"ad": 0.0, "bd": 0.0, "kd": 0.05}},
        "wake_velocity_parameters": {"gauss": {"alpha": 0.58, "beta": 0.077, "ka": 0.38, "kb": 0.004}, "jensen": {"we": 0.05}},
        "wake_turbulence_parameters": {"crespo_hernandez": {"initial": 0.1, "constant": 0.5, "ai": 0.8, "downstream": -0.32}},
    },
}


def test_parse_reads_layout_wind_and_parameters(tmp_path):
    path = tmp_path / "case.yaml"
    path.write_text(yaml.safe_dump(CASE))
    parsed = load_floris_yaml(str(path))
    assert parsed["xcoords"] == CASE["farm"]["layout_x"] and parsed["ycoords"] == CASE["farm"]["layout_y"]
    assert (parsed["wind_speed"], parsed["wind_direction"]) == (9.5, 262.0)
    ov = parsed["overrides"]
    assert ov["turbulence_intensity"] == 0.08 and ov["air_density"] == 1.2 and ov["wind_shear"] == 0.14
    assert ov["alpha"] == 0.58 and ov["ka"] == 0.38 and ov["ch_downstream"] == -0.32 and ov["dm"] == 1.0


def test_reference_template_parses_to_the_library_defaults():
    """The FLORIS v3 GCH input the reference's template follows (tests/golden/floris_case_template.yaml, every section
    on the template's lines that SURVEY.md cites) must map onto wf_default_config exactly."""
    template = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "floris_case_template.yaml")
    from wfcrl_b200.backend import default_config

    cfg, parsed = default_config(), load_floris_yaml(template)
    for field, value in parsed["overrides"].items():
        assert getattr(cfg, field) == value, field
    assert (parsed["wind_speed"], parsed["wind_direction"]) == (8.0, 270.0)


def test_five_point_grid_is_accepted_and_routed():
    case = copy.deepcopy(CASE)
    case["solver"]["turbine_grid_points"] = 5
    assert parse_floris_config(case)["overrides"]["turbine_grid_points"] == 5   # FlorisInterface then picks the basic kernels
    assert parse_floris_config(CASE)["overrides"]["turbine_grid_points"] == 3


@pytest.mark.parametrize("mutate,needle", [
    (lambda c: c["wake"]["model_strings"].__setitem__("velocity_model", "jensen"), "velocity_model"),
    (lambda c: c["wake"]["model_strings"].__setitem__("deflection_model", "jimenez"), "deflection_model"),
    (lambda c: c["wake"].__setitem__("enable_secondary_steering", False), "enable_secondary_steering"),
    (lambda c: c["solver"].__setitem__("turbine_grid_points", 7), "turbine_grid_points"),
    (lambda c: c["farm"].__setitem__("turbine_type", ["iea_10MW"]), "turbine_type"),
    (lambda c: c["wake"]["wake_velocity_parameters"]["gauss"].__setitem__("ka", 0.5), "share ka"),
    (lambda c: c["flow_field"].__setitem__("wind_speeds", [8.0, 9.0]), "exactly one wind speed"),
])
def test_unsupported_selections_are_refused(mutate, needle):
    case = copy.deepcopy(CASE)
    mutate(case)
    with pytest.raises(ValueError, match=needle):
        parse_floris_config(case)


@pytest.mark.gpu
def test_interface_from_floris_yaml_matches_oracle(cuda_device, tmp_path):
    """FlorisInterface(num_turbines, simul_file=<yaml>) as in the reference; the file's turbulence intensity reaches the
    kernels (oracle run with the same ambient TI)."""
    from oracle import c_oracle
    from wfcrl_b200.interface import FlorisInterface

    path = tmp_path / "case.yaml"
    case = copy.deepcopy(CASE)
    case["flow_field"].update(air_density=1.225, wind_shear=0.12)   # the oracle checker exposes the ambient TI only
    path.write_text(yaml.safe_dump(case))
    iface = FlorisInterface(4, str(path), max_iter=10)
    assert (iface.wind_speed, iface.wind_dir) == (9.5, 262.0)
    yaw = np.array([12.0, -8.0, 0.0, 20.0], dtype=np.float32)
    iface.update_command(yaw=yaw)
    ref = c_oracle.solve(np.array(case["farm"]["layout_x"]), np.array(case["farm"]["layout_y"]), 9.5, 262.0,
                         yaw.astype(np.float64), ti_ambient=0.08)
    assert np.max(np.abs(iface.avg_powers() - ref.power_W) / ref.power_W) < 1e-9
    assert np.allclose(iface.get_measure("wind_speed"), ref.ws_local, rtol=1e-9)
    base = c_oracle.solve(np.array(case["farm"]["layout_x"]), np.array(case["farm"]["layout_y"]), 9.5, 262.0,
                          yaw.astype(np.float64))
    assert np.max(np.abs(base.power_W - ref.power_W) / ref.power_W) > 1e-4   # the TI of the file does matter
