"""``BmiTopoflowGlacier`` -- the BMI surface of the reference over device-resident state.

Drop-in for reference ``src/topoflow_glacier/bmi/bmi_topoflow_glacier.py:115`` (same class name, method
names, variable names/units and config schema).  What differs by design:

* state lives in HBM (``MeltEngine``); ``get_value_ptr`` returns the live ``torch`` CUDA tensor;
* one model may hold N cells (an ``ensemble:`` list in the yaml, or ``initialize_ensemble``): every BMI
  variable then has N items instead of 1;
* ``update()`` is one launch of the fused kernel with ``n_steps = 1``; ``update_until`` /
  ``update_steps`` advance many steps in one launch with the per-cell state held in registers;
* the BMI functions that raise in the reference (time, units, grid, ``get_value_at_indices`` ...,
  reference ``bmi_base.py:93-274``) are implemented.

Host<->device traffic of the per-step driver pattern (7 x set_value, update, 8 x get_value) is batched: values
set through ``set_value`` are staged in one pinned block and uploaded with a single copy at ``update()``;
the first ``get_value`` after an update downloads all outputs with a single copy.
"""

from __future__ import annotations

from pathlib import Path
from typing import Optional, Sequence

import numpy as np
import torch
import yaml

from . import _lib
from .config import CELL_PARAM_KEYS, FORCING_ADJUST_KEYS, KERNEL_CONSTANTS, TopoflowGlacierConfig
from .engine import INPUT_ROWS, MeltEngine
from .logger import configure_logging, logger
from .statics import CELL_KEYS
from .timebase import default_timezone, parse_start

try:  # the reference derives from bmipy.Bmi; keep that when the package is present
    from bmipy import Bmi as _BmiBase
except Exception:  # noqa: BLE001
    _BmiBase = object

__all__ = ["BmiTopoflowGlacier", "ensemble_cell_params"]

# (BMI name, unit, internal name) -- names and unit strings as in the reference, :18-57
_INPUTS = (
    ("land_surface_radiation~incoming~longwave__energy_flux", "W m-2", "LW_in"),
    ("land_surface_air__pressure", "Pa", "P_air"),
    ("atmosphere_air_water~vapor__relative_saturation", "kg kg-1", "Hum_sp"),
    ("atmosphere_water__liquid_equivalent_precipitation_rate", "mm h-1", "P"),
    ("land_surface_radiation~incoming~shortwave__energy_flux", "W m-2", "SW_in"),
    ("land_surface_air__temperature", "degC", "T_air"),
    ("wind_speed_UV", "m sec-1", "uz"),
)
_OUTPUTS = (
    ("snowpack__depth", "m", "h_snow"),
    ("snowpack__liquid-equivalent_depth", "m", "h_swe"),
    ("snowpack__melt_volume_flux", "m s-1", "SM"),
    ("glacier_ice__thickness", "m", "h_ice"),
    ("glacier__liquid_equivalent_depth", "m", "h_iwe"),
    ("glacier_ice__melt_volume_flux", "m s-1", "IM"),
    ("land_surface_water__runoff_volume_flux", "m s-1", "M_total"),
    ("atmosphere_bottom_air_water-vapor__relative_saturation", "-", "RH"),
)
INTERNAL_NAME_CROSSWALK = {b: i for b, _, i in _INPUTS + _OUTPUTS}
EXTERNAL_NAME_CROSSWALK = {v: k for k, v in INTERNAL_NAME_CROSSWALK.items()}
_OUT_INTERNAL = tuple(i for _, _, i in _OUTPUTS)


def ensemble_cell_params(cfgs) -> dict:
    """Per-member values of ``config.CELL_PARAM_KEYS`` (float64 ``[len(cfgs)]`` arrays) of an ensemble of validated configs.

    Every other setting the kernels read is one value per model: members that differ in ``dt``, ``start_time``,
    ``SATTERLUND`` or another ``KERNEL_CONSTANTS`` key are refused with a ``ValueError`` naming the key."""
    head = cfgs[0]
    for c in cfgs[1:]:
        if (c.dt, str(c.start_time)) != (head.dt, str(head.start_time)):
            raise ValueError("all ensemble members must share dt and start_time")
        for k in ("SATTERLUND",) + tuple(k for k in KERNEL_CONSTANTS if k not in CELL_PARAM_KEYS):
            if getattr(c, k) != getattr(head, k):
                raise ValueError(f"all ensemble members must share {k} (only {', '.join(CELL_PARAM_KEYS)} may differ "
                                 f"per member): {getattr(head, k)!r} != {getattr(c, k)!r}")
    return {k: np.array([getattr(c, k) for c in cfgs], dtype=np.float64) for k in CELL_PARAM_KEYS}


class BmiTopoflowGlacier(_BmiBase):
    """BMI model of the snow / glacier-ice energy-balance melt path on one B200."""

    def __init__(self) -> None:
        self._engine: Optional[MeltEngine] = None
        self._units = {b: u for b, u, _ in _INPUTS + _OUTPUTS}
        self._in_names = tuple(b for b, _, _ in _INPUTS)
        self._out_names = tuple(b for b, _, _ in _OUTPUTS)
        configure_logging()

    # ------------------------------------------------------------------ initialise / finalise
    def initialize(self, config_file) -> None:
        """Read ``config_file`` (reference yaml schema) and place the model on the GPU (``:274-411``)."""
        path = Path(config_file)
        with open(path) as f:
            raw = yaml.safe_load(f)
        self.cfg = TopoflowGlacierConfig.model_validate(raw)
        cfgs = [self.cfg]
        for extra in self.cfg.ensemble or []:
            p = Path(extra)
            with open(p if p.is_absolute() else path.parent / p) as f:
                cfgs.append(TopoflowGlacierConfig.model_validate(yaml.safe_load(f)))
        self._build(cfgs)

    def initialize_ensemble(self, configs: Sequence, **engine_kw) -> None:
        """Extension: N catchments (config paths, dicts or validated objects) as one device-resident model.

        ``engine_kw`` reaches ``MeltEngine``: e.g. ``mode="f64_fast"``, ``basin_id=..., n_basin=...`` or
        ``forcing_index=..., n_forcing_cols=M`` (members that share a forcing series: the input variables then hold
        ``M`` values, one per series).  Each member keeps its own ``dust_atten, canopy_factor, cloud_factor, z0_air,
        em_surf`` and its own forcing adjustments ``T_air_offset`` / ``P_multiplier``; members that differ in any other
        physical constant are refused (``ensemble_cell_params``)."""
        cfgs = []
        for c in configs:
            if isinstance(c, (str, Path)):
                with open(c) as f:
                    c = yaml.safe_load(f)
            cfgs.append(c if isinstance(c, TopoflowGlacierConfig) else TopoflowGlacierConfig.model_validate(c))
        self.cfg = cfgs[0]
        self._build(cfgs, **engine_kw)

    def initialize_cells(self, base_config, cells, zones=None, tz_idx=None, **engine_kw) -> None:
        """Extension: N cells given as arrays (a raster, elevation bands ...) instead of N yaml files.

        ``base_config`` (path, dict or validated object) supplies ``dt``, the time window and the physical constants;
        ``cells`` maps the per-catchment yaml keys (``statics.CELL_KEYS``: ``da, slope, aspect, lon, lat, elev,
        h0_snow, h0_ice, h0_swe, h0_iwe, T_rain_snow``) to float64 ``[N]`` arrays, and may also give per-cell values
        of ``config.CELL_PARAM_KEYS`` (``dust_atten`` ... ``em_surf``; the others come from ``base_config``) and of the
        forcing adjustments ``T_air_offset`` / ``P_multiplier`` (``MeltEngine.set_forcing_adjust``; keys not given take
        ``base_config``'s values).  ``zones`` / ``tz_idx`` as for
        ``MeltEngine``; ``engine_kw`` reaches it too (``mode``, ``basin_id``, ``n_basin``, ``forcing_index`` ...).
        With ``shard=True`` under an initialised ``torch.distributed`` group every rank keeps only its own
        128-aligned block of the cells (``sharding.shard_bounds``) -- see ``ShardedMeltEngine``."""
        c = base_config
        if isinstance(c, (str, Path)):
            with open(c) as f:
                c = yaml.safe_load(f)
        self.cfg = c if isinstance(c, TopoflowGlacierConfig) else TopoflowGlacierConfig.model_validate(c)
        par = {k: np.atleast_1d(np.asarray(cells[k], dtype=np.float64)) for k in CELL_PARAM_KEYS if k in cells}
        adj = {k: np.atleast_1d(np.asarray(cells[k] if k in cells else getattr(self.cfg, k), dtype=np.float64))
               for k in FORCING_ADJUST_KEYS}
        cells = {k: np.atleast_1d(np.asarray(cells[k], dtype=np.float64)) for k in CELL_KEYS}
        n = cells["lat"].size
        if par:
            engine_kw.setdefault("cell_params", {k: np.broadcast_to(v, (n,)) for k, v in par.items()})
        engine_kw.setdefault("forcing_adjust", {k: np.broadcast_to(v, (n,)) for k, v in adj.items()})
        if zones is None:
            h = self.cfg
            zones = [h.utc_offset_hours if h.utc_offset_hours is not None else
                     (h.tz_name or default_timezone(float(cells["lat"].mean()), float(cells["lon"].mean())))]
        self._build_from_cells(self.cfg, cells, list(zones), tz_idx, **engine_kw)

    def _build(self, cfgs, **engine_kw) -> None:
        head = cfgs[0]
        engine_kw.setdefault("cell_params", ensemble_cell_params(cfgs))
        engine_kw.setdefault("forcing_adjust", {k: np.array([getattr(c, k) for c in cfgs], dtype=np.float64)
                                                for k in FORCING_ADJUST_KEYS})
        cells = {k: np.array([getattr(c, k) for c in cfgs], dtype=np.float64) for k in CELL_KEYS}
        zones, tz_idx = [], np.zeros(len(cfgs), dtype=np.uint8)
        for i, c in enumerate(cfgs):
            z = c.utc_offset_hours if c.utc_offset_hours is not None else (c.tz_name or default_timezone(c.lat, c.lon))
            if z not in zones:
                zones.append(z)
            tz_idx[i] = zones.index(z)
        for z in zones:  # the zone is data here (the reference looks it up): say which one was taken
            logger.info(f"time zone / UTC offset in use: {z}")
        self._build_from_cells(head, cells, zones, tz_idx if len(zones) > 1 else None, **engine_kw)

    def _build_from_cells(self, head, cells, zones, tz_idx, shard: bool = False, **engine_kw) -> None:
        n_total = int(cells["lat"].size)
        # reference scalars drivers rely on (:286-294)
        self.dt = head.dt
        self.C_to_K = 273.15
        self.K_to_C = -273.15
        self.da_km2 = head.da if n_total == 1 else cells["da"]
        self.da_m2 = self.da_km2 * 1e6
        self._start = parse_start(head.start_time)
        try:
            self._end_s = (parse_start(head.end_time) - self._start).total_seconds()
        except ValueError:
            self._end_s = float("inf")
        horizon = int(min(max(self._end_s / 3600.0 / max(head.dt, 1) + 2, 48), 24 * 366 * 4))
        engine_kw.setdefault("mode", head.precision)
        engine_kw.setdefault("device", head.device)
        engine_kw.setdefault("horizon_steps", horizon)
        if shard:
            from .sharding import ShardedMeltEngine

            # every rank keeps its block of the cells; BMI variables then hold this rank's cells only, and
            # `model.sharded.run(...)` returns the global basin aggregates (sharding.ShardedMeltEngine)
            self.sharded = ShardedMeltEngine(cells, head.model_dump(), head.start_time, dt_hours=head.dt, zones=zones,
                                             tz_idx=tz_idx, **engine_kw)
            self._engine = self.sharded.engine
            lo, hi = self.sharded.bounds
            self.da_km2 = cells["da"][lo:hi]
            self.da_m2 = self.da_km2 * 1e6
        else:
            self._engine = MeltEngine(cells, head.model_dump(), head.start_time, dt_hours=head.dt, zones=zones,
                                      tz_idx=tz_idx, **engine_kw)
        e = self._engine
        self._n = e.N
        # pinned staging: inputs (upload at update) and outputs (download at first get after update)
        # (one column per cell, or per forcing column when the ensemble was built with forcing_index=...)
        self._in_host = torch.zeros(len(INPUT_ROWS), e.n_cols, dtype=e.dtype).pin_memory()
        self._in_dirty = np.zeros(len(INPUT_ROWS), dtype=bool)
        self._in_uploaded = None  # CUDA event: the last asynchronous upload has finished reading _in_host
        self._out_host = torch.zeros(len(_OUT_INTERNAL), e.N, dtype=e.dtype).pin_memory()
        self._out_rows = torch.tensor([self._state_row(k) for k in _OUT_INTERNAL], device=e.device)
        self._out_valid = False
        self._forcing_block = None
        self._forcing_pos = 0

    def finalize(self) -> None:
        """Release the device context (the reference's is a no-op, ``:467``)."""
        if self._engine is not None:
            self._engine.close()

    # ------------------------------------------------------------------ time stepping
    def _flush_inputs(self) -> None:
        if self._in_dirty.any():
            e = self._engine
            if self._in_dirty.all():
                e.inputs.copy_(self._in_host, non_blocking=True)
            else:
                for r in np.flatnonzero(self._in_dirty):
                    e.inputs[r].copy_(self._in_host[r], non_blocking=True)
            self._in_dirty[:] = False
            # the DMA reads the pinned block asynchronously: the next host write into it must wait for this event
            self._in_uploaded = torch.cuda.Event()
            self._in_uploaded.record(torch.cuda.current_stream(e.device))

    def _wait_upload(self) -> None:
        """Block until the pinned input block may be overwritten (a driver that calls set_value / update in a loop
        without reading outputs would otherwise overwrite values an upload in flight has not read yet)."""
        if self._in_uploaded is not None:
            self._in_uploaded.synchronize()
            self._in_uploaded = None

    def update(self) -> None:
        """Advance one timestep from the current inputs (reference ``update()``, ``:413-465``)."""
        self._flush_inputs()
        self._engine.step()
        self._out_valid = False

    def update_steps(self, n_steps: int, forcing: Optional[torch.Tensor] = None, **run_kw):
        """Extension: ``n_steps`` fused timesteps in ONE kernel launch.

        ``forcing`` is a device tensor ``[n_steps, 5, N]`` (P [m/h], T_air [degC], P_air [Pa], Hum_sp, uz);
        when omitted the current inputs are held constant over the interval, as the reference's
        ``update_until`` loop does (``:489-490``).
        """
        e = self._engine
        n_steps = int(n_steps)
        if n_steps <= 0:
            raise ValueError("n_steps must be positive")
        if forcing is not None and (forcing.dim() != 3 or forcing.shape[0] < n_steps or
                                    tuple(forcing.shape[1:]) != (5, e.n_cols)):
            # checked BEFORE the launch: a bad block must not leave the model advanced
            raise ValueError(f"forcing must be [>= {n_steps}, 5, {e.n_cols}] (one column per "
                             f"{'forcing series' if e.forcing_index is not None else 'cell'}), got {tuple(forcing.shape)}")
        self._flush_inputs()
        self._out_valid = False
        if forcing is not None:
            out = e.run(forcing, n_steps, **run_kw)
            e.inputs[:5].copy_(forcing[n_steps - 1])  # inputs reflect the last step
            return out
        out, done = {}, 0
        chunk = max(1, min(n_steps, (64 << 20) // max(1, 5 * e.n_cols * e.inputs.element_size())))
        block = e.inputs[:5].unsqueeze(0).expand(chunk, 5, e.n_cols).contiguous()
        while done < n_steps:
            k = min(chunk, n_steps - done)
            part = e.run(block, k, **run_kw)
            for name, v in part.items():
                out.setdefault(name, []).append(v)
            done += k
        return {k: torch.cat(v) for k, v in out.items()}

    def load_forcing(self, forcing: torch.Tensor) -> None:
        """Extension: queue a device-resident ``[T, 5, N]`` block (``[T, 5, n_series]`` for an ensemble built with
        ``forcing_index``) that ``update_until`` consumes step by step."""
        e = self._engine
        if forcing.dim() != 3 or tuple(forcing.shape[1:]) != (5, e.n_cols):
            raise ValueError(f"forcing must be [T, 5, {e.n_cols}], got {tuple(forcing.shape)}")
        self._forcing_block, self._forcing_pos = forcing, 0

    def update_until(self, time: float) -> None:
        """Advance to model time ``time`` [s] (intended behaviour of reference ``:471-490``, which raises)."""
        now = self.get_current_time()
        if time <= now:
            logger.warning(f"no update performed: {time=} <= current_time={now}")
            return None
        n_steps, remainder = divmod(time - now, self.get_time_step())
        if remainder != 0:
            logger.warning(f"time is not multiple of time step size. updating until: {time - remainder}")
        n_steps = int(n_steps)
        if n_steps <= 0:
            return None
        fb = self._forcing_block
        if fb is None:
            self.update_steps(n_steps)   # inputs held constant, as the reference's loop of update() calls (:489-490)
            return None
        left = fb.shape[0] - self._forcing_pos
        k = min(left, n_steps)
        if k > 0:
            self.update_steps(k, fb[self._forcing_pos:self._forcing_pos + k])
            self._forcing_pos += k
        if k < n_steps:  # never fall back silently to constant inputs in the middle of a queued series
            raise RuntimeError(f"update_until({time}): the block queued by load_forcing held {left} more steps, "
                               f"{n_steps} were requested; the model stopped at t = {self.get_current_time()} s")

    # ------------------------------------------------------------------ checkpoint / resume (extension)
    def save_state(self, path) -> None:
        self._flush_inputs()
        torch.save(self._engine.state_dict(), path)

    def load_state(self, path) -> None:
        self._engine.load_state_dict(torch.load(path, weights_only=False))
        self._wait_upload()
        self._in_host.copy_(self._engine.inputs)
        self._in_dirty[:] = False
        self._out_valid = False

    # ------------------------------------------------------------------ time queries
    def get_start_time(self) -> float:
        return 0

    def get_current_time(self) -> float:
        return self._engine.step_index * self.get_time_step()

    def get_time_step(self) -> float:
        return float(self.dt) * 3600.0

    def get_time_units(self) -> str:
        return "s"

    def get_end_time(self) -> float:
        return self._end_s

    # ------------------------------------------------------------------ variable info
    def get_component_name(self) -> str:
        return "Topoflow-Glacier"

    def get_input_item_count(self) -> int:
        return len(self._in_names)

    def get_output_item_count(self) -> int:
        return len(self._out_names)

    def get_input_var_names(self) -> tuple:
        return self._in_names

    def get_output_var_names(self) -> tuple:
        return self._out_names

    def get_var_units(self, name: str) -> str:
        self._internal(name)
        return self._units[name]

    def get_var_itemsize(self, name: str) -> int:
        return self.get_value_ptr(name).itemsize

    def get_var_nbytes(self, name: str) -> int:
        return self.get_value_ptr(name).nbytes

    def get_var_type(self, name: str) -> str:
        return str(self.get_value_ptr(name).dtype)

    def get_var_grid(self, name: str) -> int:
        self._internal(name)
        return 0

    def get_var_location(self, name: str) -> str:
        self._internal(name)
        return "node"

    # one grid: N unconnected points (cells / catchments)
    def get_grid_rank(self, grid: int) -> int:
        return 1

    def get_grid_size(self, grid: int) -> int:
        return self._n

    def get_grid_type(self, grid: int) -> str:
        return "scalar" if self._n == 1 else "points"

    def get_grid_shape(self, grid: int, shape: np.ndarray) -> np.ndarray:
        shape[:] = self._n
        return shape

    def get_grid_node_count(self, grid: int) -> int:
        return self._n

    # ------------------------------------------------------------------ get / set
    def _internal(self, name: str) -> str:
        try:
            return INTERNAL_NAME_CROSSWALK[name]
        except KeyError:
            raise KeyError(f"unknown name: {name!s}") from None

    def _state_row(self, internal: str) -> int:
        from .engine import STATE_ROWS

        return STATE_ROWS.index(internal)

    def get_value_ptr(self, name: str) -> torch.Tensor:
        """Live device tensor of the variable (the reference returns the live ndarray, ``:1826-1828``)."""
        internal = self._internal(name)
        if internal in INPUT_ROWS:
            self._flush_inputs()
        return self._engine.row(internal)

    def _host_view(self, name: str) -> np.ndarray:
        internal = self._internal(name)
        if internal in INPUT_ROWS:
            r = INPUT_ROWS.index(internal)
            if not self._in_dirty[r]:
                self._wait_upload()
                self._in_host[r].copy_(self._engine.inputs[r])
            return self._in_host[r].numpy()
        if not self._out_valid:
            e = self._engine
            self._out_host.copy_(e.state.index_select(0, self._out_rows), non_blocking=True)
            torch.cuda.current_stream(e.device).synchronize()
            self._out_valid = True
        return self._out_host[_OUT_INTERNAL.index(internal)].numpy()

    def get_value(self, name: str, dest: np.ndarray) -> np.ndarray:
        """Copy the variable into ``dest`` and return it (``:1810-1824``)."""
        src = self._host_view(name)
        try:
            dest[:] = src.flatten()
        except Exception as e:  # noqa: BLE001
            raise RuntimeError(f"Could not return value {name} as flattened array") from e
        return dest

    def get_value_at_indices(self, name: str, dest: np.ndarray, inds: np.ndarray) -> np.ndarray:
        dest[:] = self._host_view(name)[np.asarray(inds)]
        return dest

    def set_value(self, name: str, src) -> None:
        """``value[:] = src`` with NumPy broadcasting (reference ``Context.set_value``, ``context.py:44``)."""
        internal = self._internal(name)
        if internal in INPUT_ROWS:
            r = INPUT_ROWS.index(internal)
            self._wait_upload()
            self._in_host[r].numpy()[:] = src
            self._in_dirty[r] = True
        else:
            host = np.empty(self._n, dtype=np.float64)
            host[:] = src
            self._engine.row(internal).copy_(torch.as_tensor(host).to(self._engine.dtype))
            lo = getattr(self._engine, "mass_lo", None)
            if lo is not None and internal in ("h_swe", "h_iwe"):   # float32 mode: the low part belongs to the old value
                lo[("h_swe", "h_iwe").index(internal)].zero_()
            self._out_valid = False

    def set_value_at_indices(self, name: str, inds: np.ndarray, src: np.ndarray) -> None:
        cur = np.array(self._host_view(name), dtype=np.float64)
        src = np.atleast_1d(np.asarray(src))
        for i in range(np.asarray(inds).shape[0]):
            cur[inds[i]] = src[i]
        self.set_value(name, cur)

    # internal-name attribute access used by drivers / tests of the reference (model.SM, model.h_swe ...)
    def __getattr__(self, item):
        if item in EXTERNAL_NAME_CROSSWALK and self.__dict__.get("_engine") is not None:
            return self.get_value_ptr(EXTERNAL_NAME_CROSSWALK[item])
        if item in ("vol_P", "vol_PR", "vol_PS", "vol_SM", "vol_IM", "P_max", "Eccs", "Ecci", "albedo") \
                and self.__dict__.get("_engine") is not None:
            return self._engine.row(item)
        raise AttributeError(item)
