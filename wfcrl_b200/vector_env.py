"""Batched vector environments: thousands of independent ``*_Floris`` envs stepped by ONE kernel launch.

``VecWindFarmEnv`` keeps the reference's Gymnasium step/reset contract (wfcrl/simple_env.py:49-96) with a leading
batch dimension and torch CUDA tensors instead of numpy arrays:

    obs = env.reset(seed=..)                         # dict: yaw, freewind_measurements, wind_speed, wind_direction
    obs, reward, terminated, truncated, info = env.step(action)     # action: float32 [B, T] (or {"yaw": ...})

Everything between action and observation -- actuation constraint, float32 yaw transition, FLORIS GCH wake solve,
measures, reward + shaper, truncation -- runs inside the fused sm_100a step kernel (``FlorisBatch.step``).
``VecMAWindFarmEnv`` is the decentralised flavour (one agent per turbine, PettingZoo parallel-API style: one call = one
full agent cycle of the reference's AEC env, wfcrl/multiagent_env.py:159-254).
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, List, Optional, Union

import numpy as np
import torch

from . import spaces
from .backend import FlorisBatch
from .layouts import get_layout
from .rewards import DoNothingReward, RewardShaper

_OBS_BOUNDS = {"wind_speed": (3.0, 28.0), "wind_direction": (0.0, 360.0)}


def layout_pool(layout, pad_turbines: bool = False) -> List[Dict]:
    """The farm cases of ``layout``: one layout name or dict, or a list of them.  The layouts of a pool must share
    ``dt`` and ``t_init`` and, unless ``pad_turbines``, the turbine count (the observation and action spaces); raises
    ValueError otherwise."""
    items = list(layout) if isinstance(layout, (list, tuple)) else [layout]
    if not items:
        raise ValueError("layout list is empty")
    cases = [get_layout(c) if isinstance(c, str) else c for c in items]
    keys = (("dt", 60), ("t_init", None)) if pad_turbines else (("num_turbines", None), ("dt", 60), ("t_init", None))
    for key, default in keys:
        values = [c.get(key, default) for c in cases]
        if any(v != values[0] for v in values):
            raise ValueError(f"the layouts of one batch must share {key}, got {values}")
    return cases


class VecWindFarmEnv:
    """``num_envs`` copies of one ``*_Floris`` env on one GPU (see the module docstring).

    ALIASING: ``reset`` / ``step`` return observation, reward, ``info["power"]`` and ``info["load"]`` as VIEWS of the
    backend's output buffers, which the next ``step`` overwrites in place (and, on auto-reset steps, the warm-up solve of
    the restarted envs already has).  A rollout buffer must ``.clone()`` what it keeps, or construct the env with
    ``copy_outputs=True`` to get fresh tensors from every call (one extra device copy of ~10 floats per turbine).

    LAYOUT POOL: ``layout`` may be a list of layouts (names or dicts) of one turbine count, ``dt`` and ``t_init``.  With
    ``layout_assignment="cycle"`` the env of global id ``g = env_id_offset + b`` runs layout ``g % L`` for good; with
    ``"sample"`` every reset draws the env's layout uniformly (in the library for ``reset(seed=None)`` and auto-resets,
    with numpy's ``default_rng((seed + g, 2))`` for ``reset(seed=seed)``).  ``reset(options={"layout": ids})`` sets the
    layout of the reset envs explicitly; ``layout_ids`` returns the current ones.

    MIXED TURBINE COUNTS: with ``pad_turbines=True`` the layouts may differ in turbine count.  ``T`` is then the largest
    count; an env whose farm has n turbines uses columns 0..n-1 of every [B, T] array, and the other columns are padding:
    actions there are ignored and observations, power and load read 0.  The observation gains ``"turbine_mask"`` (bool
    [B, T], True on the env's turbines), ``turbine_counts`` gives the counts per env, and each env's reward is its own
    farm's (the mean over its n turbines).  Not available with ``multi_agent``."""

    metadata = {"name": "vectorized-windfarm"}

    def __init__(self, layout: Union[str, Dict, List], num_envs: int, *, device: int = 0, precision: str = "f32",
                 kernel: Optional[str] = None, controls: Optional[dict] = None, continuous_control: bool = True,
                 reward_shaper: Optional[RewardShaper] = None, max_num_steps: int = 500, load_coef: float = 0.1,
                 start_iter: int = 0, auto_reset: bool = True, multi_agent: bool = False, env_id_offset: int = 0,
                 wind_time_series: Optional[Union[str, np.ndarray]] = None, exact_host_trig: Optional[bool] = None,
                 turbulence_intensity_range: Optional[tuple] = None, copy_outputs: bool = False,
                 layout_assignment: str = "cycle", pad_turbines: bool = False):
        if pad_turbines and multi_agent:
            raise ValueError("pad_turbines is not supported by the multi-agent (Dec_) envs: their agents are the turbines")
        cases = layout_pool(layout, pad_turbines)
        if layout_assignment not in ("cycle", "sample"):
            raise ValueError(f"layout_assignment must be 'cycle' or 'sample', got {layout_assignment!r}")
        if layout_assignment == "sample" and wind_time_series is not None:
            raise ValueError("layout_assignment='sample' draws layouts at library-sampled resets, which time-series mode "
                             "does not use; assign layouts with 'cycle' or reset(options={'layout': ...})")
        case = cases[0]
        self.copy_outputs = bool(copy_outputs)
        self.farm_case = case
        self.farm_cases = cases
        self.layout_assignment = layout_assignment
        self.num_envs = int(num_envs)
        self.pad_turbines = bool(pad_turbines)
        if self.pad_turbines:
            case = max(cases, key=lambda c: c["num_turbines"])  # the handle is created with the largest farm
        self.num_turbines = case["num_turbines"]
        self.dt = case.get("dt", 60)
        controls = dict(controls or {"yaw": (-40, 40, 5)})
        if set(controls) != {"yaw"}:
            raise ValueError(f"Cannot control {sorted(set(controls) - {'yaw'})}. Interface FlorisInterface only allows "
                             "for the following: ['yaw']")
        lo, hi, *rest = controls["yaw"]
        if not lo < hi:
            raise ValueError("Wrong bounds for actuator yaw: ensure that lower_bound < upper_bound")
        step = rest[0] if rest else 1
        self.controls = {"yaw": (lo, hi, step)}
        self.continuous_control = continuous_control
        self.max_num_steps = max_num_steps
        self.start_iter = start_iter
        self.load_coef = load_coef
        self.auto_reset = auto_reset
        self.env_id_offset = int(env_id_offset)
        self.reward_shaper = reward_shaper if reward_shaper is not None else DoNothingReward()
        code = getattr(self.reward_shaper, "kernel_code", None)
        if code is None:
            raise ValueError("the batched path supports DoNothingReward, ReferencePercentage and StepPercentage")
        precision = {"fp32": "f32", "fp64": "f64"}.get(precision, precision)
        kernel = kernel or "fast"  # warp-per-env kernels: FP32 fast mode or its FP64 instantiation (bit-check mode)
        self.precision = precision
        self.exact_host_trig = (precision == "f64") if exact_host_trig is None else exact_host_trig
        self.backend = FlorisBatch(case["xcoords"], case["ycoords"], self.num_envs, device=device, precision=precision,
                                   kernel=kernel, max_iter=start_iter + max_num_steps, yaw_bounds=(lo, hi, step),
                                   load_coef=load_coef, reward_shaper=code,
                                   shaper_reference=float(getattr(self.reward_shaper, "reference", 0.0)),
                                   continuous_control=continuous_control, multi_agent=multi_agent)
        self.device = self.backend.device
        if len(cases) > 1:
            if self.pad_turbines:
                self.backend.set_mixed_layouts([c["xcoords"] for c in cases], [c["ycoords"] for c in cases])
            else:
                self.backend.set_layouts([c["xcoords"] for c in cases], [c["ycoords"] for c in cases])
            if layout_assignment == "cycle":
                self.backend.assign_layouts(None, (self.env_id_offset + np.arange(self.num_envs)) % len(cases))
        if layout_assignment == "sample":
            self.backend.set_layout_sampling(True)
        T = self.num_turbines
        self.single_action_space = spaces.Dict({"yaw": spaces.Box(-step, step, shape=(T,))}) if continuous_control \
            else spaces.Dict({"yaw": spaces.MultiDiscrete([3] * T)})
        ones = np.ones(T, dtype=np.float32)
        self.single_observation_space = spaces.Dict(OrderedDict([
            ("yaw", spaces.Box(ones * lo, ones * hi, shape=(T,))),
            ("freewind_measurements", spaces.Box(np.array([3, 0], np.float32), np.array([28, 360], np.float32), shape=(2,))),
            # padding columns read 0
            ("wind_speed", spaces.Box(ones * (0 if self.pad_turbines else 3), ones * 28, shape=(T,))),
            ("wind_direction", spaces.Box(ones * 0, ones * 360, shape=(T,))),
        ] + ([("turbine_mask", spaces.MultiDiscrete([2] * T))] if self.pad_turbines else [])))
        self.action_space = self.single_action_space
        self.observation_space = self.single_observation_space
        self._gen = torch.Generator(device=self.device)  # time-series start offsets of in-loop resets only
        self._gen.manual_seed(0x5EED + self.env_id_offset)
        self._seed = int(np.random.SeedSequence().entropy) & 0xFFFFFFFFFFFFFFFF  # replaced by reset(seed=...)
        # Episodes have a fixed length, so the host knows WHEN envs truncate without looking at the device: one countdown per
        # cohort of envs that were reset together (a handful of python ints, no per-env mirror)
        self._countdowns = []
        self._series = None
        if wind_time_series is not None:
            if isinstance(wind_time_series, str):  # csv path: first column speed, second direction (interface.py:473-474, 514)
                import pandas as pd

                wind_time_series = pd.read_csv(wind_time_series).values
            series = np.asarray(wind_time_series, dtype=np.float64)
            assert series.ndim == 2 and series.shape[1] >= 2, "time series rows are [speed, direction]"
            self._series = torch.as_tensor(series[:, :2], device=self.device)
            self._series_pos = torch.zeros(self.num_envs, dtype=torch.long, device=self.device)
        # extension (BASELINE.json configs[2]): ambient TI sampled per env at reset, U(lo, hi); the reference fixes 0.06
        self.turbulence_intensity_range = turbulence_intensity_range
        self._arm_autoreset()
        self._zeros_bool = torch.zeros(self.num_envs, dtype=torch.bool, device=self.device)
        self._needs_reset = True
        self._turbine_mask = None
        if self.pad_turbines:
            self._refresh_turbine_mask()

    def _refresh_turbine_mask(self):
        """Rebuild ``"turbine_mask"`` from the envs' turbine counts; called where layouts can change (construction, reset,
        and auto-resets that draw layouts), so that a plain step costs no host round trip."""
        counts = torch.as_tensor(self.backend.get_state("turbine_count"), device=self.device)
        self._turbine_mask = torch.arange(self.num_turbines, device=self.device)[None, :] < counts[:, None]

    def _arm_autoreset(self):
        """In-kernel auto-reset (wf_set_autoreset): the truncating step itself zeroes the env's state and marks it; one
        geometry + warm-up launch pair (``autoreset_finish``) completes the reset.  Time-series mode restarts the series at
        a host-drawn row and keeps the explicit reset path."""
        self._fused_autoreset = bool(self.auto_reset and self._series is None)
        self.backend.set_autoreset(self._fused_autoreset, self._seed, self.env_id_offset, self.turbulence_intensity_range)

    def _tick(self) -> bool:
        """Advance the cohort countdowns by one step; True when some cohort's episode ends at this step."""
        fired = False
        nxt = set()
        for c in self._countdowns:
            c -= 1
            if c == 0:
                fired = True
                if self.auto_reset:
                    nxt.add(self.max_num_steps - 1)
            else:
                nxt.add(c)
        self._countdowns = sorted(nxt)
        return fired

    # -- wind sampling ------------------------------------------------------------------------------------------
    def sample_wind_host(self, seed: Optional[int], env_ids: np.ndarray, need_speed: bool = True,
                         need_direction: bool = True):
        """The reference's reset distribution with numpy's Generator, one stream per GLOBAL env id
        (wfcrl/mdp.py:235-258): bit-identical to what ``WindFarmMDP.reset(seed + env_id)`` would draw.  A component the
        caller supplies through ``options`` is not drawn at all, so the other one keeps its place in the stream."""
        ws = np.empty(len(env_ids))
        wd = np.empty(len(env_ids))
        for k, b in enumerate(env_ids):
            rng = np.random.default_rng(None if seed is None else seed + self.env_id_offset + int(b))
            if need_speed:
                ws[k] = np.clip(8 * rng.weibull(8), 3, 28)
            if need_direction:
                wd[k] = np.clip(rng.normal(270, 20) % 360, 0, 360)
        return ws, wd

    # -- API ------------------------------------------------------------------------------------------------------
    def _obs(self, out):
        c = (lambda t: t.clone()) if self.copy_outputs else (lambda t: t)
        obs = OrderedDict([("yaw", c(out["yaw"])), ("freewind_measurements", c(out["freewind"])),
                           ("wind_speed", c(out["wind_speed"])), ("wind_direction", c(out["wind_direction"]))])
        if self.pad_turbines:
            obs["turbine_mask"] = self._turbine_mask  # replaced, never written in place, by _refresh_turbine_mask
        return obs

    def reset(self, seed: Optional[int] = None, options: Optional[dict] = None, env_ids=None):
        """Reset all (or ``env_ids``) envs.  ``options`` may carry ``wind_speed`` / ``wind_direction`` (scalars or
        per-env arrays) exactly like the reference; otherwise both are sampled per env.  ``options["layout"]`` (a scalar or
        per-env pool index) sets the layout of the reset envs; otherwise ``layout_assignment="sample"`` draws it.

        ``seed=s`` draws env ``g``'s wind with numpy exactly as the reference's ``reset(seed=s + g)`` would and makes
        ``s`` the key of all later in-loop resets; ``seed=None`` draws on the device (``wf_reset_sampled``).  Either way
        an env's winds depend on its GLOBAL id and episode index only, not on the sharding."""
        ids = np.arange(self.num_envs) if env_ids is None else np.asarray(env_ids)
        idt = torch.as_tensor(ids, device=self.device)
        options = options or {}
        warm = self.start_iter + 1
        if seed is not None:
            self._seed = int(seed) & 0xFFFFFFFFFFFFFFFF
            episode = self.backend.get_state("episode")
            episode[ids] = 0
            self.backend.set_state("episode", episode)
        given = "wind_speed" in options and "wind_direction" in options
        any_given = "wind_speed" in options or "wind_direction" in options
        if self._series is not None:
            start = np.random.randint(0, self._series.shape[0], size=len(ids))  # interface.py:517
            self._series_pos[idt] = torch.as_tensor(start, device=self.device)
        in_library = seed is None and not any_given and self._series is None
        sampling = self.layout_assignment == "sample"
        if "layout" in options:
            self.backend.assign_layouts(ids, options["layout"])
        elif sampling and not in_library:  # as the sampled TI below: one numpy stream per (seed + global id, 2)
            n_layouts = len(self.farm_cases)
            self.backend.assign_layouts(ids, [np.random.default_rng(
                None if seed is None else (seed + self.env_id_offset + int(b), 2)).integers(n_layouts) for b in ids])
        if in_library:
            # nothing to reproduce on the host: winds (and TI, layouts) drawn by the library for the selected envs
            mask = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
            mask[idt] = 1
            keep_layouts = sampling and "layout" in options  # the layouts given in options are not redrawn
            if keep_layouts:
                self.backend.set_layout_sampling(False)
            out = self.backend.reset_sampled(mask, self._seed, self.env_id_offset, warm, self.turbulence_intensity_range)
            if keep_layouts:
                self.backend.set_layout_sampling(True)
        else:
            if self._series is not None:
                first = self._series[self._series_pos[idt]].cpu().numpy()
                ws, wd = first[:, 0], first[:, 1]
            else:
                ws_s, wd_s = (None, None) if given else self.sample_wind_host(
                    seed, ids, "wind_speed" not in options, "wind_direction" not in options)
                ws = np.broadcast_to(np.asarray(options.get("wind_speed", ws_s), dtype=np.float64), ids.shape)
                wd = np.broadcast_to(np.asarray(options.get("wind_direction", wd_s), dtype=np.float64), ids.shape)
            if self.turbulence_intensity_range is not None:
                lo_ti, hi_ti = self.turbulence_intensity_range
                ti = self.backend.get_state("ti_ambient")
                ti[ids] = [np.random.default_rng(None if seed is None else (seed + self.env_id_offset + int(b), 1))
                           .uniform(lo_ti, hi_ti) for b in ids]
                self.backend.set_turbulence_intensity(torch.as_tensor(ti, device=self.device))
            out = self.backend.reset(ws, wd, env_ids=ids.astype(np.int32), host_trig=self.exact_host_trig,
                                     warmup_solves=warm)
        self._arm_autoreset()  # (re)arm with the current seed: in-loop resets are keyed by it
        if len(ids) == self.num_envs:
            self._countdowns = []
        self._countdowns = sorted(set(self._countdowns) | {self.max_num_steps - 1})
        self._needs_reset = False
        if self.pad_turbines:
            self._refresh_turbine_mask()
        return self._obs(out)

    def step(self, action):
        assert not self._needs_reset, "Call reset before `step`"
        if isinstance(action, dict):
            action = action["yaw"]
        if not torch.is_tensor(action):
            action = torch.as_tensor(np.asarray(action, dtype=np.float32), device=self.device)
        action = action.to(device=self.device, dtype=torch.float32).contiguous()
        if self._series is not None:  # time-series mode: the wind moves before every solve (interface.py:563).
            # Extension: the series is cyclic here; the reference's generator stops after one pass over the rows.
            self._series_pos = (self._series_pos + 1) % self._series.shape[0]
            row = self._series[self._series_pos]
            self.backend.update_wind(row[:, 0].contiguous(), row[:, 1].contiguous(), host_trig=self.exact_host_trig)
        out = self.backend.step(action)
        # nothing else per step on this side: episode returns / lengths and the finished-episode sums are kept by the step
        # kernel's epilogue (state arrays "ep_return", "ep_len", "fin_*"), `truncated` is the kernel's flag viewed as bool
        reward = out["reward"]
        truncated = out["truncated"].view(torch.bool)
        if self.copy_outputs:
            reward, truncated = reward.clone(), truncated.clone()
            info = {"power": out["power"].clone(), "load": out["load"].clone()}
        else:
            info = {"power": out["power"], "load": out["load"]}
        obs = self._obs(out)
        if self._tick() and self.auto_reset:
            # same-step autoreset: final observation is preserved in info, obs rows of finished envs restart
            info["final_observation"] = OrderedDict((k, v.clone()) for k, v in obs.items())
            info["final_info"] = {"power": out["power"].clone(), "load": out["load"].clone()}
            truncated = truncated.clone()
            reward = reward.clone()
            if self._fused_autoreset:
                # the step kernel has already reset the truncated envs' state and marked them: wind draw + geometry +
                # warm-up solve of the marked envs, no host round trip
                out = self.backend.autoreset_finish(self.start_iter + 1)
                if self.pad_turbines and self.layout_assignment == "sample":
                    self._refresh_turbine_mask()
            else:  # time series: the wind generator restarts at a random row (interface.py:517)
                start = torch.randint(0, self._series.shape[0], (self.num_envs,), device=self.device, generator=self._gen)
                self._series_pos = torch.where(truncated, start, self._series_pos)
                row = self._series[self._series_pos]
                out = self.backend.reset_masked(truncated.view(torch.uint8).clone(), row[:, 0].contiguous(),
                                                row[:, 1].contiguous(), warmup_solves=self.start_iter + 1)
            obs = self._obs(out)
        self.last_info = info  # joint (un-split) info of this step, incl. final_observation on auto-reset steps
        return obs, reward, self._zeros_bool, truncated, info

    def evaluate_actions(self, action):
        """One-step lookahead: what ``step`` would return for each of K candidate actions per env, from where each env is
        now, without stepping (``FlorisBatch.evaluate_actions``).  ``action``: [B, K, T] (or ``{"yaw": ...}``).  Returns
        ``(obs, reward, terminated, truncated, info)`` with a K axis after the batch axis, exactly as ``step`` would return
        them for each candidate, without the auto-reset handling: a candidate that truncates reports ``truncated`` and its
        final observation, and nothing is reset.  The env's state, its cohort countdowns included, does not change.
        Views of buffers the next call overwrites unless ``copy_outputs``.  Not available in wind-time-series mode, where a
        step moves the wind before it solves."""
        assert not self._needs_reset, "Call reset before `evaluate_actions`"
        if self._series is not None:
            raise ValueError("evaluate_actions is not available in wind-time-series mode: a step there moves the wind (and "
                             "the geometry) before it solves, which an evaluation cannot do without changing the state")
        if isinstance(action, dict):
            action = action["yaw"]
        if not torch.is_tensor(action):
            action = torch.as_tensor(np.asarray(action, dtype=np.float32), device=self.device)
        out = self.backend.evaluate_actions(action.to(device=self.device, dtype=torch.float32).contiguous())
        c = (lambda t: t.clone()) if self.copy_outputs else (lambda t: t)
        obs = OrderedDict([("yaw", c(out["yaw"])), ("freewind_measurements", c(out["freewind"])),
                           ("wind_speed", c(out["wind_speed"])), ("wind_direction", c(out["wind_direction"]))])
        K = out["reward"].shape[1]
        if self.pad_turbines:
            obs["turbine_mask"] = self._turbine_mask[:, None, :].expand(-1, K, -1)
        terminated = torch.zeros(self.num_envs, K, dtype=torch.bool, device=self.device)
        info = {"power": c(out["power"]), "load": c(out["load"])}
        return obs, c(out["reward"]), terminated, c(out["truncated"].view(torch.bool)), info

    @property
    def layout_ids(self):
        """Index into the layout list of the layout every env currently runs (int32 [B], device copy)."""
        return torch.as_tensor(self.backend.get_state("layout_id"), device=self.device)

    @property
    def turbine_counts(self):
        """Turbine count of the layout every env currently runs (int32 [B], device copy)."""
        return torch.as_tensor(self.backend.get_state("turbine_count"), device=self.device)

    @property
    def episode_returns(self):
        """Return accumulated so far in every env's RUNNING episode (float64 [B], device copy of the kernel's accumulator)."""
        return torch.as_tensor(self.backend.get_state("ep_return"), device=self.device)

    @property
    def episode_lengths(self):
        return torch.as_tensor(self.backend.get_state("ep_len").astype(np.int64), device=self.device)

    def episode_statistics(self):
        """Global statistics of the finished episodes (all-gathered over ranks when torch.distributed is initialised), from
        the per-env sums the step kernels keep: (sum, sum of squares, count, length sum)."""
        from .dist import gather_episode_sums

        g = self.backend.get_state
        return gather_episode_sums(float(g("fin_sum").sum()), float(g("fin_sumsq").sum()), float(g("fin_n").sum()),
                                   float(g("fin_len").sum()), self.device)

    def close(self):
        self.backend.close()


class VecMAWindFarmEnv(VecWindFarmEnv):
    """Decentralised batch: agents ``turbine_1..T``; ``step`` takes the actions of ALL agents (a full AEC cycle) either
    as a float32 [B, T] tensor (column k = agent k) or as ``{agent: {"yaw": tensor[B]}}``, and returns per-agent dicts."""

    metadata = {"name": "vectorized-multiagent-windfarm", "is_parallelizable": True}

    def __init__(self, layout, num_envs, **kwargs):
        kwargs["multi_agent"] = True
        super().__init__(layout, num_envs, **kwargs)
        self.possible_agents = [f"turbine_{k + 1}" for k in range(self.num_turbines)]
        self.agents = self.possible_agents[:]
        self.agent_name_mapping = {a: k for k, a in enumerate(self.possible_agents)}
        lo, hi, step = self.controls["yaw"]
        self._obs_spaces = {a: {"yaw": spaces.Box(lo, hi), "wind_speed": spaces.Box(3, 28),
                                "wind_direction": spaces.Box(0, 360)} for a in self.possible_agents}
        self._act_spaces = {a: {"yaw": spaces.Box(-step, step)} for a in self.possible_agents}

    def observation_space(self, agent):
        return self._obs_spaces[agent]

    def action_space(self, agent):  # noqa: D102 - shadows the attribute of the centralised env on purpose
        return self._act_spaces[agent]

    def _split(self, obs):
        return {a: OrderedDict((k, v[:, i]) for k, v in obs.items() if k != "freewind_measurements")
                for a, i in self.agent_name_mapping.items()}

    def reset(self, seed=None, options=None, env_ids=None):
        return self._split(super().reset(seed, options, env_ids))

    def step(self, actions):
        if isinstance(actions, dict) and actions and next(iter(actions)) in self.agent_name_mapping:
            cols = [torch.as_tensor(actions[a]["yaw"], device=self.device).reshape(self.num_envs) for a in self.possible_agents]
            actions = torch.stack(cols, 1)
        obs, reward, terminated, truncated, info = super().step(actions)
        per_agent_info = {a: {"power": info["power"][:, i], "load": info["load"][:, i]}
                          for a, i in self.agent_name_mapping.items()}
        return (self._split(obs), {a: reward for a in self.possible_agents}, {a: terminated for a in self.possible_agents},
                {a: truncated for a in self.possible_agents}, per_agent_info)

    def evaluate_actions(self, actions):
        """``VecWindFarmEnv.evaluate_actions`` for the agents: ``actions`` is the joint float32 [B, K, T] tensor (column
        k = agent k) or ``{agent: {"yaw": tensor[B, K]}}``; returns per-agent dicts as ``step`` does, with the K axis."""
        if isinstance(actions, dict) and actions and next(iter(actions)) in self.agent_name_mapping:
            actions = torch.stack([torch.as_tensor(actions[a]["yaw"], device=self.device) for a in self.possible_agents], 2)
        obs, reward, terminated, truncated, info = super().evaluate_actions(actions)
        split = {a: OrderedDict((k, v[:, :, i]) for k, v in obs.items() if k != "freewind_measurements")
                 for a, i in self.agent_name_mapping.items()}
        per_agent_info = {a: {"power": info["power"][:, :, i], "load": info["load"][:, :, i]}
                          for a, i in self.agent_name_mapping.items()}
        return (split, {a: reward for a in self.possible_agents}, {a: terminated for a in self.possible_agents},
                {a: truncated for a in self.possible_agents}, per_agent_info)
