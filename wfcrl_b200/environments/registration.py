"""Environment registry with the reference's id grammar ``[Dec_]<Layout>_<Simulator>`` (wfcrl/environments/
registration.py:17-28) and factory ``make`` (:81-113), restricted to the Floris simulator -- the FAST.Farm/MPI backend is
out of scope (BASELINE.json north_star).  ``make_vec`` is the batched addition."""
from __future__ import annotations

import math
import re
from typing import List, Union

from ..layouts import ALIASES
from .data_cases import DefaultControl, floris_case, registered_layouts as _layouts

env_pattern = r"(Dec_)*(\w+\d*_)(\w+)"
registered_simulators = ["Floris"]
registered_layouts = _layouts() + list(ALIASES.keys())
control_types = ["", "Dec_"]
registered_envs = [c + lay + sim for c in control_types for lay in registered_layouts for sim in registered_simulators]


def get_default_control(controls):
    defaults = DefaultControl()
    return {name: getattr(defaults, name) for name in ("yaw", "pitch", "torque") if name in controls}


def get_case(name: str, simulator: str = "Floris"):
    if simulator != "Floris":
        raise ValueError("only the Floris simulator is available in wfcrl_b200 (FAST.Farm is out of scope)")
    return floris_case(name)


def validate_case(env_id, case):
    if len(case.xcoords) != len(case.ycoords):
        raise ValueError(f"Invalid configuration for case {env_id}: xcoords and ycoords layout coordinates must have "
                         "the same length")


def _parse(env_id: str):
    if env_id not in registered_envs:
        hint = " (the FAST.Farm backend is out of scope here)" if env_id.endswith("Fastfarm") else ""
        raise ValueError(f"{env_id} is not a registered WFCRL benchmark environment.{hint}")
    match = re.match(env_pattern, env_id)
    return match.group(1) == "Dec_", match.group(2), match.group(3)


def make(env_id: str, controls: Union[dict, list] = ["yaw"], log=True, **env_kwargs):
    """Return a single wind-farm environment exactly like the reference's ``envs.make`` (Gymnasium ``WindFarmEnv`` or
    PettingZoo-AEC ``MAWindFarmEnv``, wrapped in a history logger unless ``log=False``), backed by the B200 kernels."""
    from ..interface import FlorisInterface
    from ..multiagent_env import MAWindFarmEnv
    from ..simple_env import WindFarmEnv
    from ..wrappers import AECLogWrapper, LogWrapper

    decentralized, name, simulator = _parse(env_id)
    case = get_case(name, simulator)
    validate_case(env_id, case)
    if not isinstance(controls, dict):
        controls = get_default_control(controls)
    if "wind_time_series" in env_kwargs:
        case.wind_time_series = env_kwargs.pop("wind_time_series")
    env_kwargs.pop("path_to_simulator", None)
    env_class = MAWindFarmEnv if decentralized else WindFarmEnv
    env = env_class(interface=FlorisInterface, farm_case=case, controls=controls,
                    start_iter=math.ceil(case.t_init / case.dt), **env_kwargs)
    if log:
        env = (AECLogWrapper if decentralized else LogWrapper)(env)
    return env


def make_vec(env_id: Union[str, List[str]], num_envs: int, controls: Union[dict, list] = ["yaw"], log: int = 0,
             **env_kwargs):
    """Batched counterpart of ``make``: ``num_envs`` independent copies of ``env_id`` on one GPU, stepped by one kernel
    launch (``VecWindFarmEnv`` / ``VecMAWindFarmEnv``).  Extra kwargs: device, precision ("f32" fast / "f64" bit-check),
    auto_reset, env_id_offset (global id of env 0 when the batch is sharded over ranks), layout_assignment; ``log=N``
    wraps the env in a ``VecLogWrapper`` keeping the last N steps in device-side ring buffers.

    A list of env ids gives one batch over several farms (the layout pool of ``VecWindFarmEnv``): the ids must be all
    centralised or all ``Dec_``, and their layouts must share the turbine count, ``dt`` and ``t_init``.  With
    ``pad_turbines=True`` (centralised ids only) the turbine counts may differ: see ``VecWindFarmEnv``."""
    from ..vector_env import VecMAWindFarmEnv, VecWindFarmEnv, layout_pool

    env_ids = [env_id] if isinstance(env_id, str) else list(env_id)
    if not env_ids:
        raise ValueError("env_id list is empty")
    parsed = [_parse(e) for e in env_ids]
    decentralized = parsed[0][0]
    if any(p[0] != decentralized for p in parsed):
        raise ValueError(f"cannot batch centralised and decentralised (Dec_) envs together: {env_ids}")
    pad_turbines = bool(env_kwargs.get("pad_turbines", False))
    if pad_turbines and decentralized:
        raise ValueError(f"pad_turbines is not supported by the decentralised (Dec_) envs: {env_ids}")
    layouts = []
    for e, (_dec, name, simulator) in zip(env_ids, parsed):
        case = get_case(name, simulator)
        validate_case(e, case)
        layouts.append({"num_turbines": case.num_turbines, "xcoords": case.xcoords, "ycoords": case.ycoords,
                        "dt": case.dt, "t_init": case.t_init})
    layout_pool(layouts, pad_turbines)  # same turbine count (unless padded), dt and t_init, checked before any device work
    if not isinstance(controls, dict):
        controls = get_default_control(controls)
    case = layouts[0]
    layout = case if len(layouts) == 1 else layouts
    cls = VecMAWindFarmEnv if decentralized else VecWindFarmEnv
    env = cls(layout, num_envs, controls=controls, start_iter=math.ceil(case["t_init"] / case["dt"]), **env_kwargs)
    if log:
        from ..wrappers import VecLogWrapper

        env = VecLogWrapper(env, capacity=int(log))
    return env


def list_envs():
    return registered_envs
