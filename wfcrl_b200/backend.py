"""``FlorisBatch``: thin PyTorch-facing wrapper over the C-ABI (device memory, streams; no arithmetic here).

It replaces, for ``num_envs`` environments at once, what the reference reaches through
``FlorisInterface`` (wfcrl/interface.py:444-671) plus the MDP transition / reward wrapped around it
(wfcrl/mdp.py:273-319, wfcrl/simple_env.py:58-96).  All compute happens in libwfcrl_b200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _lib

_PREC = {"f64": _lib.PREC_F64, "fp64": _lib.PREC_F64, "f32": _lib.PREC_F32, "fp32": _lib.PREC_F32}
_KERN = {"basic": _lib.KERNEL_BASIC, "fast": _lib.KERNEL_FAST}
_SHAPER = {"none": _lib.SHAPER_NONE, "reference": _lib.SHAPER_REFERENCE_PCT, "step": _lib.SHAPER_STEP_PCT}

_STATE_DTYPES = {
    "yaw": (np.float64, "BT"), "acc": (np.float32, "BT"), "acc_prev": (np.float32, "BT"),
    "num_iter": (np.int32, "B"), "num_moves": (np.int32, "B"), "nonfinite": (np.int32, "B"), "episode": (np.int32, "B"), "ambiguous": (np.uint8, "B"),
    "ep_return": (np.float64, "B"), "ep_len": (np.int32, "B"), "fin_sum": (np.float64, "B"), "fin_sumsq": (np.float64, "B"),
    "fin_n": (np.int32, "B"), "fin_len": (np.int64, "B"), "ws": (np.float64, "B"), "wd": (np.float64, "B"),
    "ws_norm": (np.float64, "B"), "shaper_ref": (np.float64, "B"), "ti_ambient": (np.float64, "B"),
    "order": (np.int32, "BT"), "xs": (np.float64, "BT"), "ys": (np.float64, "BT"), "xi": (np.float64, "BT"),
    "yi": (np.float64, "BT"), "cs": (np.float64, "B2"), "layout_id": (np.int32, "B"),
    "turbine_count": (np.int32, "B"),
}
# the step outputs (WfStepOut) and their shapes; each is "real" (the handle's precision) but the uint8 truncation flag
_OUTPUTS = {"yaw": "BT", "wind_speed": "BT", "wind_direction": "BT", "power": "BT", "load": "BT4", "reward": "B",
            "freewind": "B2", "truncated": "B"}


def default_config() -> _lib.WfConfig:
    cfg = _lib.WfConfig()
    _lib.check(_lib.load().wf_default_config(C.byref(cfg)))
    return cfg


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _out_struct(bufs: Dict[str, torch.Tensor]) -> _lib.WfStepOut:
    """The WfStepOut of the output buffers ``bufs`` (name -> tensor); the outputs it does not name are not written."""
    return _lib.WfStepOut(**{k: t.data_ptr() for k, t in bufs.items()})


class FlorisBatch:
    """``num_envs`` independent Floris-backed wind-farm envs resident on one GPU.  They share the layout given here
    unless ``set_layouts`` gives the handle a pool of layouts of the same turbine count to assign per env, or
    ``set_mixed_layouts`` a pool of layouts of 1..T turbines (an env of n turbines uses columns 0..n-1 of every [B, T]
    array; the other columns are padding and read 0)."""

    def __init__(self, layout_x: Sequence[float], layout_y: Sequence[float], num_envs: int, *, device: int = 0,
                 precision: str = "f64", kernel: str = "basic", max_iter: int = 500,
                 yaw_bounds=(-40.0, 40.0, 5.0), load_coef: float = 0.1, reward_shaper: str = "none",
                 shaper_reference: float = 0.0, continuous_control: bool = True, multi_agent: bool = False,
                 strict: bool = True, config_overrides: Optional[Dict[str, float]] = None):
        if not torch.cuda.is_available():
            raise _lib.WfError("wfcrl_b200 needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.T = len(layout_x)
        self.B = int(num_envs)
        self.device = torch.device("cuda", device)
        self.precision = precision
        self.real = torch.float64 if _PREC[precision] == _lib.PREC_F64 else torch.float32
        cfg = default_config()
        cfg.num_turbines, cfg.num_envs, cfg.device = self.T, self.B, device
        cfg.precision, cfg.kernel = _PREC[precision], _KERN[kernel]
        cfg.max_iter = int(max_iter)
        cfg.continuous_control = int(bool(continuous_control))
        cfg.multi_agent = int(bool(multi_agent))
        cfg.fp32_relaxed = int(not strict)  # FP32 fast kernel only: skip the guard band + FP64 re-solve (raw FP32 results)
        cfg.reward_shaper = _SHAPER[reward_shaper]
        cfg.shaper_reference = float(shaper_reference)
        cfg.yaw_lo, cfg.yaw_hi, cfg.yaw_step = (float(v) for v in yaw_bounds)
        cfg.load_coef = float(load_coef)
        for key, val in (config_overrides or {}).items():
            if not hasattr(cfg, key):
                raise ValueError(f"unknown config field {key}")
            setattr(cfg, key, val)
        self.cfg = cfg
        lx = np.ascontiguousarray(layout_x, dtype=np.float64)
        ly = np.ascontiguousarray(layout_y, dtype=np.float64)
        handle = C.c_void_p()
        _lib.check(self.lib.wf_create(C.byref(cfg), lx.ctypes.data_as(C.c_void_p), ly.ctypes.data_as(C.c_void_p),
                                      C.byref(handle)))
        self.handle = handle
        self.out = {k: torch.zeros(self._shape(kind), dtype=torch.uint8 if k == "truncated" else self.real,
                                   device=self.device) for k, kind in _OUTPUTS.items()}
        self._out_struct = _out_struct(self.out)
        self._host = None
        self.eval_capacity = 0  # largest K evaluate_yaw has run with (its output buffers and the library scratch hold that)
        self.act_capacity, self._act_bufs = 0, None  # the same for evaluate_actions

    # ------------------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.wf_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------------------------------------------
    def set_layouts(self, xs, ys) -> None:
        """Replace the layout pool by ``xs``, ``ys`` [L, T] (metres).  Every env gets layout 0 and its geometry is rebuilt
        with its current wind; counters and yaw are kept.  Waits for all queued work of the handle."""
        x = np.ascontiguousarray(xs, dtype=np.float64)
        y = np.ascontiguousarray(ys, dtype=np.float64)
        if x.ndim != 2 or x.shape != y.shape or x.shape[1] != self.T:
            raise ValueError(f"layout pool must be two [L, {self.T}] arrays, got {x.shape} and {y.shape}")
        _lib.check(self.lib.wf_set_layouts(self.handle, x.shape[0], x.ctypes.data_as(C.c_void_p),
                                           y.ctypes.data_as(C.c_void_p)))

    def set_mixed_layouts(self, xs, ys) -> None:
        """Replace the layout pool by layouts of different turbine counts: ``xs``, ``ys`` are lists of 1-D arrays
        (metres), layout l of ``len(xs[l])`` in [1, T] turbines.  An env of n turbines runs them in columns 0..n-1;
        columns n..T-1 of its outputs are 0, and its results equal those of a handle created with its layout alone.
        Otherwise as ``set_layouts``."""
        if len(xs) != len(ys) or len(xs) < 1:
            raise ValueError("xs and ys must be non-empty lists of the same length")
        L, T = len(xs), self.T
        counts = np.empty(L, dtype=np.int32)
        x = np.zeros((L, T), dtype=np.float64)
        y = np.zeros((L, T), dtype=np.float64)
        for l, (lx, ly) in enumerate(zip(xs, ys)):
            lx, ly = np.asarray(lx, dtype=np.float64).reshape(-1), np.asarray(ly, dtype=np.float64).reshape(-1)
            if lx.shape != ly.shape or not 1 <= lx.shape[0] <= T:
                raise ValueError(f"layout {l}: x and y must be two 1-D arrays of the same length in [1, {T}], "
                                 f"got {lx.shape} and {ly.shape}")
            counts[l] = lx.shape[0]
            x[l, :counts[l]], y[l, :counts[l]] = lx, ly
        _lib.check(self.lib.wf_set_layouts_sized(self.handle, L, counts.ctypes.data_as(C.c_void_p),
                                                 x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p)))

    def assign_layouts(self, env_ids, layout_ids) -> None:
        """Give the envs ``env_ids`` (None = all) the pool layouts ``layout_ids`` (scalar or per env) and rebuild their
        geometry with their current wind."""
        ids = None if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32).reshape(-1)
        n = self.B if ids is None else ids.shape[0]
        lids = np.ascontiguousarray(np.broadcast_to(np.asarray(layout_ids, dtype=np.int32), (n,)))
        _lib.check(self.lib.wf_assign_layouts(self.handle, None if ids is None else ids.ctypes.data_as(C.c_void_p), n,
                                              lids.ctypes.data_as(C.c_void_p), self._stream()))

    def set_layout_sampling(self, enabled: bool) -> None:
        """While enabled, ``reset_sampled`` and the in-kernel auto-reset also draw each reset env's layout id uniformly
        from the pool, with the same counter-based generator as its wind (draw word 2)."""
        _lib.check(self.lib.wf_set_layout_sampling(self.handle, int(bool(enabled))))

    def reset(self, wind_speed, wind_direction, env_ids=None, *, host_trig: bool = True, warmup_solves: int = 1):
        """WindFarmMDP.reset for the selected envs (mdp.py:260-270).  ``host_trig=True`` ships numpy's FP64 cosd/sind of
        the wind deviation so the rotated geometry is bit-identical to a host (numpy) reference (SURVEY 7.3)."""
        ids = np.arange(self.B, dtype=np.int32) if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32)
        n = ids.shape[0]
        ws = np.ascontiguousarray(np.broadcast_to(np.asarray(wind_speed, dtype=np.float64), (n,)))
        wd = np.ascontiguousarray(np.broadcast_to(np.asarray(wind_direction, dtype=np.float64), (n,)))
        hc = hs = None
        if host_trig:
            dev = (((wd % 360.0) - 270.0) % 360.0 + 360.0) % 360.0
            hc = np.ascontiguousarray(np.cos(np.radians(dev)))
            hs = np.ascontiguousarray(np.sin(np.radians(dev)))
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
        _lib.check(self.lib.wf_reset(self.handle, vp(ids), n, vp(ws), vp(wd), vp(hc), vp(hs), int(warmup_solves),
                                     C.byref(self._out_struct), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()  # host staging arrays above must outlive the copies
        return self.out

    def reset_sampled(self, mask: Optional[torch.Tensor], seed: int, env_id_offset: int = 0, warmup_solves: int = 1,
                      turbulence_intensity_range: Optional[tuple] = None):
        """Device-side reset with the winds drawn inside the library from the reference's reset distribution
        (wfcrl/mdp.py:242-258) by a counter-based generator keyed by (seed, env_id_offset + env, episode index): the
        draws do not depend on how the envs are sharded over handles / GPUs.  ``mask`` uint8 [B] or None (= all)."""
        if mask is not None and mask.dtype != torch.uint8:
            raise TypeError("mask must be a uint8 CUDA tensor of shape [B]")
        lo, hi = turbulence_intensity_range if turbulence_intensity_range is not None else (0.0, 0.0)
        _lib.check(self.lib.wf_reset_sampled(self.handle, _ptr(mask) if mask is not None else None,
                                             int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_id_offset), float(lo), float(hi),
                                             int(warmup_solves), C.byref(self._out_struct), self._stream()))
        return self.out

    def set_autoreset(self, enabled: bool, seed: int = 0, env_id_offset: int = 0,
                      turbulence_intensity_range: Optional[tuple] = None):
        """Arm / disarm the in-kernel auto-reset (``wf_set_autoreset``): a step that truncates an env also starts its next
        episode (wind from the library's counter-based sampler); ``autoreset_finish`` completes it."""
        lo, hi = turbulence_intensity_range if turbulence_intensity_range is not None else (0.0, 0.0)
        _lib.check(self.lib.wf_set_autoreset(self.handle, int(bool(enabled)), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                             int(env_id_offset), float(lo), float(hi)))

    def autoreset_finish(self, warmup_solves: int = 1):
        """Geometry + warm-up solve(s) of the envs the last step(s) reset in-kernel; their output rows become the start
        observation.  Cheap no-op launches when no env is marked."""
        _lib.check(self.lib.wf_autoreset_finish(self.handle, int(warmup_solves), C.byref(self._out_struct), self._stream()))
        return self.out

    def reset_masked(self, mask: torch.Tensor, wind_speed: torch.Tensor, wind_direction: torch.Tensor,
                     warmup_solves: int = 1):
        """Device-side reset of the envs where ``mask`` (uint8 [B]) is non-zero; no host round trip."""
        if not (mask.dtype == torch.uint8 and wind_speed.dtype == torch.float64 and wind_direction.dtype == torch.float64):
            raise TypeError("mask must be uint8, wind_speed / wind_direction float64 (CUDA tensors of shape [B])")
        _lib.check(self.lib.wf_reset_masked(self.handle, _ptr(mask), _ptr(wind_speed), _ptr(wind_direction),
                                            int(warmup_solves), C.byref(self._out_struct), self._stream()))
        return self.out

    def step(self, action: torch.Tensor):
        """One env step for every env; ``action`` float32 [B, T] on the device.  Returns the output tensor dict
        (overwritten in place every call)."""
        if not (torch.is_tensor(action) and action.dtype == torch.float32 and action.is_cuda and action.is_contiguous()):
            raise TypeError("action must be a contiguous float32 CUDA tensor")
        if tuple(action.shape) != (self.B, self.T):
            raise ValueError(f"action must have shape ({self.B}, {self.T}), got {tuple(action.shape)}")
        _lib.check(self.lib.wf_step(self.handle, _ptr(action), C.byref(self._out_struct), self._stream()))
        return self.out

    def update_command(self, yaw: Optional[torch.Tensor] = None):
        """FlorisInterface.update_command(yaw) for every env (interface.py:557-586); power in W, loads x1e7."""
        if yaw is not None:
            if not (yaw.dtype == torch.float64 and yaw.is_cuda and yaw.is_contiguous()):
                raise TypeError("yaw must be a contiguous float64 CUDA tensor")
            if tuple(yaw.shape) != (self.B, self.T):
                raise ValueError(f"yaw must have shape ({self.B}, {self.T}), got {tuple(yaw.shape)}")
        _lib.check(self.lib.wf_update_command(self.handle, _ptr(yaw), C.byref(self._out_struct), self._stream()))
        return self.out

    def evaluate_yaw(self, yaw: torch.Tensor) -> Dict[str, torch.Tensor]:
        """Per-turbine power (W) of K candidate yaw settings per env, in each env's current wind, TI and layout, without
        changing any state (``wf_evaluate_yaw``).  ``yaw``: contiguous float64 CUDA tensor [B, K, T], absolute degrees, not
        clipped; padding columns of a mixed-count pool are ignored.  Returns ``{"power": [B, K, T], "ambiguous": bool [B, K]}``
        (1 = re-solved in FP64 on a strict FP32 handle), views of buffers owned by the batch that the next call overwrites.
        Asynchronous; the first call with a larger K than before allocates, synchronously."""
        if not (torch.is_tensor(yaw) and yaw.dtype == torch.float64 and yaw.is_cuda and yaw.is_contiguous()):
            raise TypeError("yaw must be a contiguous float64 CUDA tensor of shape [B, K, T]")
        if yaw.dim() != 3 or yaw.shape[0] != self.B or yaw.shape[2] != self.T or yaw.shape[1] < 1:
            raise ValueError(f"yaw must have shape ({self.B}, K, {self.T}) with K >= 1, got {tuple(yaw.shape)}")
        K = int(yaw.shape[1])
        power_buf, amb_buf = getattr(self, "_eval_power", None), getattr(self, "_eval_amb", None)
        if K > self.eval_capacity:
            power_buf = torch.zeros(self.B * K * self.T, dtype=self.real, device=self.device)
            amb_buf = torch.zeros(self.B * K, dtype=torch.uint8, device=self.device)
        power = power_buf[: self.B * K * self.T].view(self.B, K, self.T)
        amb = amb_buf[: self.B * K].view(self.B, K)
        _lib.check(self.lib.wf_evaluate_yaw(self.handle, _ptr(yaw), K, _ptr(power), _ptr(amb), self._stream()))
        if K > self.eval_capacity:  # the library holds scratch for this K now
            self._eval_power, self._eval_amb, self.eval_capacity = power_buf, amb_buf, K
        return {"power": power, "ambiguous": amb.view(torch.bool)}

    def evaluate_actions(self, action: torch.Tensor) -> Dict[str, torch.Tensor]:
        """What ``step`` would return for each of K candidate actions per env, from the current state, without stepping
        (``wf_evaluate_actions``).  ``action``: contiguous float32 CUDA tensor [B, K, T], each [T] row interpreted as
        ``step`` interprets one; padding columns of a mixed-count pool are ignored.  Returns the eight step outputs with a K
        axis after the batch axis (``yaw`` [B, K, T], ..., ``load`` [B, K, T, 4], ``reward`` / ``truncated`` [B, K],
        ``freewind`` [B, K, 2]; env-mode units) and ``"ambiguous"`` bool [B, K], views of buffers owned by the batch that
        the next call overwrites.  No state changes.  Asynchronous; the first call with a larger K than before allocates,
        synchronously."""
        if not (torch.is_tensor(action) and action.dtype == torch.float32 and action.is_cuda and action.is_contiguous()):
            raise TypeError("action must be a contiguous float32 CUDA tensor of shape [B, K, T]")
        if action.dim() != 3 or action.shape[0] != self.B or action.shape[2] != self.T or action.shape[1] < 1:
            raise ValueError(f"action must have shape ({self.B}, K, {self.T}) with K >= 1, got {tuple(action.shape)}")
        K = int(action.shape[1])
        kinds = dict(_OUTPUTS, ambiguous="B")
        bufs = self._act_bufs
        if K > self.act_capacity:
            bufs = {k: torch.zeros((self.B, K) + self._shape(kind)[1:], device=self.device,
                                   dtype=torch.uint8 if k in ("truncated", "ambiguous") else self.real)
                    for k, kind in kinds.items()}
        res = {k: bufs[k].view(-1)[: self.B * K * bufs[k][0, 0].numel()].view((self.B, K) + bufs[k].shape[2:])
               for k in kinds}
        amb = res.pop("ambiguous")
        _lib.check(self.lib.wf_evaluate_actions(self.handle, _ptr(action), K, C.byref(_out_struct(res)), _ptr(amb),
                                                self._stream()))
        if K > self.act_capacity:
            self._act_bufs, self.act_capacity = bufs, K
        res["ambiguous"] = amb.view(torch.bool)
        return res

    def _host_out(self) -> Dict[str, torch.Tensor]:
        """Pinned host mirror of ``self.out`` for the host-buffer entry points (allocated on first use)."""
        if self._host is None:
            self._host = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in self.out.items()}
        return self._host

    def step_host(self, action_host: torch.Tensor, fields=tuple(_OUTPUTS)):
        """End-to-end step from HOST memory (pinned recommended): H2D action, step, D2H of ``fields``, sync."""
        if not (action_host.dtype == torch.float32 and not action_host.is_cuda and action_host.is_contiguous()):
            raise TypeError("action_host must be a contiguous float32 HOST tensor (pinned recommended)")
        if tuple(action_host.shape) != (self.B, self.T):
            raise ValueError(f"action_host must have shape ({self.B}, {self.T})")
        host = self._host_out()
        st = _out_struct({k: host[k] for k in fields})
        up, down = C.c_uint64(), C.c_uint64()
        _lib.check(self.lib.wf_step_host(self.handle, C.c_void_p(action_host.data_ptr()), C.byref(st), C.byref(up),
                                         C.byref(down)))
        self.last_h2d_bytes, self.last_d2h_bytes = up.value, down.value
        return {k: host[k] for k in fields}

    def update_command_host(self, yaw_host: Optional[np.ndarray] = None):
        """FlorisInterface.update_command from HOST memory in one library call (wf_update_command_host): float64 [B, T]
        yaw command in (or None), measures out as numpy views of pinned buffers (overwritten by the next call)."""
        if getattr(self, "_host_np", None) is None:
            host = self._host_out()
            self._host_np = {k: v.numpy() for k, v in host.items()}
            self._host_struct = _out_struct({k: v for k, v in host.items() if k != "reward"})
            self._yaw_pin = torch.empty(self.B, self.T, dtype=torch.float64).pin_memory()
            self._yaw_pin_np = self._yaw_pin.numpy()
        ptr = None
        if yaw_host is not None:
            self._yaw_pin_np[...] = yaw_host
            ptr = C.c_void_p(self._yaw_pin.data_ptr())
        _lib.check(self.lib.wf_update_command_host(self.handle, ptr, C.byref(self._host_struct)))
        return self._host_np

    def set_turbulence_intensity(self, ti: torch.Tensor):
        if not (ti.dtype == torch.float64 and ti.is_cuda and tuple(ti.shape) == (self.B,)):
            raise TypeError("ti must be a float64 CUDA tensor of shape [B]")
        _lib.check(self.lib.wf_set_turbulence_intensity(self.handle, _ptr(ti), self._stream()))

    def update_wind(self, wind_speed: torch.Tensor, wind_direction: torch.Tensor, mask: Optional[torch.Tensor] = None,
                    host_trig: bool = False):
        """FlorisInterface.update_wind for every (or the masked) env: new free-stream wind, counters untouched.
        ``host_trig=True`` computes cosd/sind of the deviation with numpy (one host round trip) for bit-exact geometry."""
        if not (wind_speed.dtype == torch.float64 and wind_direction.dtype == torch.float64):
            raise TypeError("wind_speed / wind_direction must be float64 CUDA tensors of shape [B]")
        cs = None
        if host_trig:
            wd = wind_direction.detach().cpu().numpy()
            dev = (((wd % 360.0) - 270.0) % 360.0 + 360.0) % 360.0
            cs = torch.as_tensor(np.stack([np.cos(np.radians(dev)), np.sin(np.radians(dev))], 1), device=self.device)
            cs = cs.contiguous()
        _lib.check(self.lib.wf_update_wind(self.handle, _ptr(mask), _ptr(wind_speed), _ptr(wind_direction), _ptr(cs),
                                           self._stream()))
        if cs is not None:
            torch.cuda.current_stream(self.device).synchronize()

    # ------------------------------------------------------------------------------------------------------
    def _shape(self, kind):
        return {"BT": (self.B, self.T), "BT4": (self.B, self.T, 4), "B": (self.B,), "B2": (self.B, 2)}[kind]

    def get_state(self, name: str) -> np.ndarray:
        dt, kind = _STATE_DTYPES[name]
        arr = np.empty(self._shape(kind), dtype=dt)
        _lib.check(self.lib.wf_get_state(self.handle, name.encode(), arr.ctypes.data_as(C.c_void_p), arr.nbytes))
        return arr

    def set_state(self, name: str, value) -> None:
        dt, kind = _STATE_DTYPES[name]
        arr = np.ascontiguousarray(np.broadcast_to(np.asarray(value, dtype=dt), self._shape(kind)))
        _lib.check(self.lib.wf_set_state(self.handle, name.encode(), arr.ctypes.data_as(C.c_void_p), arr.nbytes))

    # checkpoint / resume: the complete env state is a handful of small arrays (SURVEY.md section 5)
    _CHECKPOINT = ("yaw", "acc", "acc_prev", "num_iter", "num_moves", "nonfinite", "episode", "ws", "wd", "ws_norm", "shaper_ref",
                   "ti_ambient", "ep_return", "ep_len", "fin_sum", "fin_sumsq", "fin_n", "fin_len")

    def state_dict(self) -> Dict[str, np.ndarray]:
        """Host copy of everything needed to resume the batch exactly where it is (geometry is rebuilt from wd and the
        layout ids, which also give each env's turbine count; the layout pool itself is configuration and is not saved)."""
        sd = {name: self.get_state(name) for name in self._CHECKPOINT}
        sd["cs"] = self.get_state("cs")
        sd["layout_id"] = self.get_state("layout_id")
        return sd

    def load_state_dict(self, sd: Dict[str, np.ndarray]) -> None:
        """Restore a ``state_dict``: layout ids (0 for a dict saved without them), then wind (rebuilds the rotated/sorted
        geometry with the saved cos/sin so the geometry is bit-identical), then counters, yaw and accumulators."""
        self.assign_layouts(None, sd.get("layout_id", 0))
        ws = torch.as_tensor(np.ascontiguousarray(sd["ws"]), device=self.device)
        wd = torch.as_tensor(np.ascontiguousarray(sd["wd"]), device=self.device)
        cs = torch.as_tensor(np.ascontiguousarray(sd["cs"]), device=self.device)
        _lib.check(self.lib.wf_update_wind(self.handle, None, _ptr(ws), _ptr(wd), _ptr(cs), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()
        for name in self._CHECKPOINT:
            self.set_state(name, sd[name])

    def device_info(self) -> Dict[str, int]:
        vals = [C.c_int32() for _ in range(6)]
        _lib.check(self.lib.wf_device_info(self.handle, *[C.byref(v) for v in vals]))
        keys = ("sm_count", "sm_clock_khz", "ctas_per_sm", "regs_per_thread", "threads_per_cta", "smem_per_cta")
        return {k: v.value for k, v in zip(keys, vals)}

    def launch_count(self) -> int:
        return int(self.lib.wf_launch_count(self.handle))

    def set_kernel_timing(self, enabled: bool):
        """Bracket the launches of every following ``step`` / ``update_command`` with CUDA events (measurement legs only)."""
        _lib.check(self.lib.wf_set_kernel_timing(self.handle, int(bool(enabled))))

    def kernel_timing(self) -> Dict[str, float]:
        """Average device time of the step kernel and of the FP64 re-solve kernel (0 where there is none) over the calls
        since the last query, and their number."""
        a, b, n = C.c_double(), C.c_double(), C.c_int32()
        _lib.check(self.lib.wf_get_kernel_timing(self.handle, C.byref(a), C.byref(b), C.byref(n)))
        return {"step_kernel_ms": a.value, "resolve_kernel_ms": b.value, "calls": n.value}
