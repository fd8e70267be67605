"""Device-resident ensemble of melt cells driven through the C ABI.

``MeltEngine`` owns every per-cell array as a ``torch`` CUDA tensor (PyTorch is used for device memory and
streams only), binds their raw pointers into a ``tfg_ctx`` and advances all cells with ``tfg_run``.  One
engine = one shard of cells on one GPU.  It is the N-cell counterpart of what one reference instance keeps
in ``Context`` (reference ``physics/context.py:18-71``) and in the attributes set up by
``BmiTopoflowGlacier.initialize`` (reference ``bmi_topoflow_glacier.py:274-411``).
"""

from __future__ import annotations

import ctypes as C
import os
from typing import Iterable, Mapping, Optional, Sequence

import numpy as np
import pandas as pd
import torch

from . import _lib
from .config import (CELL_PARAM_KEYS, FORCING_ADJUST_IDENTITY, FORCING_ADJUST_KEYS, KERNEL_CONSTANTS, check_cell_params,
                     check_forcing_adjust, check_forcing_noise)
from .statics import cell_tables
from .timebase import parse_start, time_tables, utc_offsets

__all__ = ["MeltEngine", "INPUT_ROWS", "STATE_ROWS"]

# rows of the input block; the first five are the live forcings in kernel order (TFG_N_FORCING)
INPUT_ROWS = ("P", "T_air", "P_air", "Hum_sp", "uz", "LW_in", "SW_in")
# rows of the state block (order of tfg_state, minus the ring)
STATE_ROWS = ("h_snow", "h_swe", "h_ice", "h_iwe", "Eccs", "Ecci", "albedo", "n", "SM", "IM", "M_total", "RH",
              "vol_P", "vol_PR", "vol_PS", "vol_SM", "vol_IM", "P_max")
_STATE_FIELD = dict(zip(STATE_ROWS, _lib.STATE_FIELDS))  # python name -> C field


def _require_cuda(device: int) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("topoflow_glacier_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", device)


class MeltEngine:
    """All cells of one shard, resident in HBM.

    Parameters
    ----------
    cells : mapping with float64 ``[N]`` arrays ``lat, lon, slope, aspect, elev, da, h0_snow, h0_ice, h0_swe,
        h0_iwe, T_rain_snow`` (names of the yaml keys; ``da`` in km2)
    consts : mapping holding the physical constants (``config.KERNEL_CONSTANTS`` keys, ``SATTERLUND``)
    start_time : ``YYYYMMDDHH`` string; ``dt_hours`` : timestep [h]
    zones : list of IANA names / fixed offsets; ``tz_idx`` : per-cell index into it (uint8) or None
    forcing_index : optional per-cell int32 column of the forcing blocks (``n_forcing_cols`` columns): the cells of
        one catchment share the catchment's forcing series, so forcing is ``[T, 5, n_forcing_cols]`` instead of
        ``[T, 5, N]`` -- nothing is replicated per cell on the host or over PCIe (``tfg_bind_forcing_map``)
    basin_id : per-cell int32 basin index in ``[0, n_basin)`` or None
    cell_params : optional mapping of any of ``config.CELL_PARAM_KEYS`` (``dust_atten, canopy_factor, cloud_factor,
        z0_air, em_surf``) to per-cell ``[N]`` arrays or device tensors: every cell runs with its own values (a
        parameter ensemble, e.g. one calibration candidate per cell); keys it does not name take the value of
        ``consts``.  See ``set_cell_params``.
    forcing_adjust : optional mapping of ``T_air_offset`` [K] and/or ``P_multiplier`` [-] to per-cell ``[N]`` arrays or
        device tensors: every cell adds its offset to the air temperature and multiplies the precipitation rate it
        reads (its own forcing column or, with ``forcing_index``, its catchment's).  See ``set_forcing_adjust``.
    forcing_noise : optional mapping of stochastic forcing perturbations for ensemble members: temporally correlated
        air-temperature and log-normal precipitation noise per stream of cells, generated on the device.  See
        ``set_forcing_noise``.
    mode : ``"f64"`` (strict), ``"f64_fast"`` or ``"f32"``
    horizon_steps : number of steps the host time tables are prepared for (extended on demand)
    """

    def __init__(self, cells: Mapping[str, np.ndarray], consts: Mapping[str, float], start_time, dt_hours: int = 1,
                 zones: Sequence = ("America/Los_Angeles",), tz_idx: Optional[np.ndarray] = None,
                 basin_id: Optional[np.ndarray] = None, n_basin: int = 0, mode: str = "f64", device: int = 0,
                 horizon_steps: int = 24 * 366, diag_integrals: bool = True, device_statics: Optional[dict] = None,
                 tma_staging: Optional[bool] = None, forcing_index=None, n_forcing_cols: Optional[int] = None,
                 column_terms: Optional[bool] = None, cell_params: Optional[Mapping] = None,
                 forcing_adjust: Optional[Mapping] = None, forcing_noise: Optional[Mapping] = None):
        self.lib = _lib.load()
        self.device = _require_cuda(device)
        self.mode = _lib.MODE_NAMES[mode] if isinstance(mode, str) else int(mode)
        self.dtype = torch.float32 if self.mode == _lib.F32 else torch.float64
        self.dt_hours = dt_hours
        self.start = parse_start(start_time) if not isinstance(start_time, pd.Timestamp) else start_time
        self.zones = list(zones)
        if not 1 <= len(self.zones) <= _lib.MAX_TZ:
            raise ValueError(f"between 1 and {_lib.MAX_TZ} time zones per engine")
        self.consts = {k: float(consts[k]) for k in KERNEL_CONSTANTS}
        self.satterlund = bool(consts.get("SATTERLUND", False))
        self.ring_slots = int(3 * 24 / dt_hours)
        if not 1 <= self.ring_slots <= _lib.RING_SLOTS_MAX:
            raise ValueError("dt must give between 1 and 72 snowfall-window slots")
        self.step_index = 0
        self.n_basin = int(n_basin)
        self._exact_agg, self._agg_exp = 0, None

        with torch.cuda.device(self.device):
            ctx = C.c_void_p()
            _lib.check(self.lib.tfg_create(C.byref(ctx), self.device.index, self.mode), "tfg_create")
            self.ctx = ctx
            if tma_staging is None:
                tma_staging = os.environ.get("TFG_TMA_STAGING", "0") == "1"
            self.tma_staging = bool(tma_staging)
            _lib.check(self.lib.tfg_set_option(ctx, _lib.OPT_TMA_STAGING, int(self.tma_staging)), "tfg_set_option")
            if column_terms is None:  # TFG_OPT_COLUMN_TERMS: forcing-only terms once per forcing column (default on)
                column_terms = os.environ.get("TFG_COLUMN_TERMS", "1") != "0"
            self.column_terms = bool(column_terms)
            _lib.check(self.lib.tfg_set_option(ctx, _lib.OPT_COLUMN_TERMS, int(self.column_terms)), "tfg_set_option")
            self._set_constants()
            if device_statics is not None:  # synthetic grids: tables already on the device
                self.N = int(next(iter(device_statics.values())).numel())
                self.static = {k: device_statics[k].to(self.device, self.dtype).contiguous() for k in _lib.STATIC_FIELDS}
                init = {k: device_statics[k].to(self.device, self.dtype) for k in ("h0_snow", "h0_ice", "h0_swe", "h0_iwe")}
            else:
                tabs = cell_tables(cells["lat"], cells["lon"], cells["slope"], cells["aspect"], cells["elev"],
                                   cells["da"], cells["T_rain_snow"], M_mass_air=self.consts["M_mass_air"],
                                   g=self.consts["g"])
                self.N = int(tabs["lon"].size)
                self.static = {k: torch.as_tensor(tabs[k]).to(self.device, self.dtype).contiguous()
                               for k in _lib.STATIC_FIELDS}
                init = {k: torch.as_tensor(np.broadcast_to(np.asarray(cells[k], dtype=np.float64), (self.N,)).copy())
                        .to(self.device, self.dtype) for k in ("h0_snow", "h0_ice", "h0_swe", "h0_iwe")}
            N = self.N
            if basin_id is None:
                self.basin_id = None
            elif torch.is_tensor(basin_id):
                self.basin_id = basin_id.to(self.device, torch.int32).contiguous()
            else:
                self.basin_id = torch.as_tensor(np.ascontiguousarray(basin_id, dtype=np.int32)).to(self.device)
            self.tz_idx = None if tz_idx is None else torch.as_tensor(
                np.ascontiguousarray(tz_idx, dtype=np.uint8)).to(self.device)
            self._bind_static()
            self.objective = None
            self.cell_params = None
            if cell_params is not None:
                self.set_cell_params(cell_params)
            self.forcing_adjust = None
            if forcing_adjust is not None:
                self.set_forcing_adjust(forcing_adjust)
            self.forcing_noise = None
            if forcing_noise is not None:
                self.set_forcing_noise(forcing_noise)
            self.n_cols, self.forcing_index = N, None
            if forcing_index is not None:
                self.set_forcing_map(forcing_index, n_forcing_cols, _alloc_inputs=False)

            self.inputs = torch.zeros(len(INPUT_ROWS), self.n_cols, dtype=self.dtype, device=self.device)
            self.state = torch.zeros(len(STATE_ROWS), N, dtype=self.dtype, device=self.device)
            self.ring = torch.zeros(self.ring_slots, N, dtype=self.dtype, device=self.device)
            self.diag_integrals = diag_integrals
            self._init_state(init)
            self._bind_state()
            self._n_time = 0
            self.ensure_horizon(horizon_steps)

    # ---- binding -----------------------------------------------------------------------------------------
    def _set_constants(self):
        c = _lib.Constants()
        for k, v in self.consts.items():
            setattr(c, k, v)
        c.dt_hours = float(self.dt_hours)
        c.z_wind = 10.0  # reference bmi_topoflow_glacier.py:301
        c.satterlund = int(self.satterlund)
        c.ring_slots = self.ring_slots
        _lib.check(self.lib.tfg_set_constants(self.ctx, C.byref(c)), "tfg_set_constants")

    def _bind_static(self):
        s = _lib.Statics()
        for k in _lib.STATIC_FIELDS:
            setattr(s, k, self.static[k].data_ptr())
        s.basin_id = self.basin_id.data_ptr() if self.basin_id is not None else None
        s.tz_idx = self.tz_idx.data_ptr() if self.tz_idx is not None else None
        _lib.check(self.lib.tfg_bind_static(self.ctx, self.N, C.byref(s)), "tfg_bind_static")

    def set_cell_params(self, params: Optional[Mapping]) -> None:
        """Bind per-cell surface parameters (``None`` unbinds them); may be called between launches.

        ``params`` maps any of ``config.CELL_PARAM_KEYS`` to ``[N]`` arrays or tensors; unnamed keys take the engine's
        constants.  Values are range-checked with the schema's bounds (``ValueError``).  A key whose values all equal
        the constant is not bound, and with no key left the engine runs exactly as without parameters.  A calibration
        loop: ``run``, score, ``set_cell_params(next_candidates)``, ``load_state_dict(initial)``, ``run`` again."""
        tensors = {k: (v if torch.is_tensor(v) else torch.as_tensor(np.asarray(v, dtype=np.float64)))
                   .to(self.device, torch.float64).contiguous().reshape(-1) for k, v in (params or {}).items()}
        bound = {}
        for k, t in check_cell_params(tensors).items():
            if t.numel() != self.N:
                raise ValueError(f"{k}: one value per cell ({self.N}) expected, got {t.numel()}")
            if not bool((t == self.consts[k]).all()):
                bound[k] = t
        with torch.cuda.device(self.device):
            if not bound:
                _lib.check(self.lib.tfg_bind_cell_params(self.ctx, None, self.stream_ptr), "tfg_bind_cell_params")
                self.cell_params = None
                return
            p = _lib.CellParams()
            for k in CELL_PARAM_KEYS:
                setattr(p, k, bound[k].data_ptr() if k in bound else None)
            # the library derives its own copy on the current stream and waits for its range check
            _lib.check(self.lib.tfg_bind_cell_params(self.ctx, C.byref(p), self.stream_ptr), "tfg_bind_cell_params")
        self.cell_params = bound

    def set_forcing_adjust(self, adjust: Optional[Mapping]) -> None:
        """Bind per-cell forcing adjustments (``None`` unbinds them); may be called between launches.

        ``adjust`` maps ``T_air_offset`` (K, in [-30, 30]) and/or ``P_multiplier`` (in [0, 10]) to ``[N]`` arrays or
        tensors.  At every step cell ``i`` then uses ``T_air + T_air_offset[i]`` and ``P * P_multiplier[i]`` of the
        forcing it reads, one operation each in the engine's float type -- the bits of a per-cell forcing adjusted in
        advance.  ``P_air``, ``Hum_sp`` and ``uz`` are not adjusted, and the input block keeps what the caller set.
        Values are range-checked (``ValueError``).  A key whose values are all the identity (0, 1) is not bound, and
        with no key left the engine runs exactly as without adjustments.  Elevation bands that share a catchment's
        series: ``T_air_offset = -T_lapse_rate * (elev_cell - elev_series)``.  Adjustments are bindings, like
        ``set_cell_params``: ``state_dict`` does not hold them."""
        tensors = {k: (v if torch.is_tensor(v) else torch.as_tensor(np.array(v, dtype=np.float64)))
                   .to(self.device, torch.float64).contiguous().reshape(-1) for k, v in (adjust or {}).items()}
        bound = {}
        for k, t in check_forcing_adjust(tensors).items():
            if t.numel() != self.N:
                raise ValueError(f"{k}: one value per cell ({self.N}) expected, got {t.numel()}")
            if not bool((t == FORCING_ADJUST_IDENTITY[k]).all()):
                bound[k] = t
        with torch.cuda.device(self.device):
            if not bound:
                _lib.check(self.lib.tfg_bind_forcing_adjust(self.ctx, None, self.stream_ptr), "tfg_bind_forcing_adjust")
                self.forcing_adjust = None
                return
            a = _lib.ForcingAdjust()
            for k in FORCING_ADJUST_KEYS:
                setattr(a, k, bound[k].data_ptr() if k in bound else None)
            # the library copies the values on the current stream and waits for its range check
            _lib.check(self.lib.tfg_bind_forcing_adjust(self.ctx, C.byref(a), self.stream_ptr), "tfg_bind_forcing_adjust")
        self.forcing_adjust = bound

    def set_forcing_noise(self, noise: Optional[Mapping]) -> None:
        """Bind stochastic forcing perturbations (``None`` unbinds them); may be called between launches.

        ``noise`` maps ``T_air_sd`` (K, in [0, 5]), ``T_air_rho`` ([0, 1]), ``P_sd`` (sd of ln of the precipitation
        factor, [0, 1.5]), ``P_rho`` ([0, 1]) and ``seed`` (an integer in [0, 2^64)); optionally ``stream``, one global
        stream id >= 0 per cell (default: the cell index), and ``step0``, the absolute step the noise starts at
        (default: ``step_index``, which ``load_state_dict`` restores).  Cells with the same stream id get the same noise
        -- one stream per ensemble member perturbs a member spread over several cells coherently -- and every stream
        is independent of the others.  At every step ``s >= step0`` cell ``i`` uses ``(T_air + T_air_offset[i]) + dT``
        and ``(P * P_multiplier[i]) * fP`` of its stream: ``dT`` an AR(1) series of standard deviation ``T_air_sd`` and
        lag-1 correlation ``T_air_rho``, ``fP = exp(P_sd z - P_sd^2 / 2)`` of an AR(1) series ``z`` of unit variance and
        correlation ``P_rho``, so that ``E[fP] = 1`` (include/tfglacier.h states the definition).  The noise is a pure
        function of (seed, stream id, step0, step): results do not depend on how a run is split into launches, on the
        per-step path, on sharding or on a checkpoint rewind.  ``P_air``, ``Hum_sp`` and ``uz`` are not perturbed, and
        the input block keeps what the caller set.  Values are range-checked (``ValueError``).  ``T_air_sd = P_sd = 0``
        is not bound: the engine then runs exactly as without noise.  The noise is a binding, like
        ``set_forcing_adjust``: ``state_dict`` does not hold it.  ``forcing_noise_series`` returns the series."""
        if noise is None:
            _lib.check(self.lib.tfg_bind_forcing_noise(self.ctx, None, self.stream_ptr), "tfg_bind_forcing_noise")
            self.forcing_noise = None
            return
        nz = check_forcing_noise(noise)
        stream = nz.pop("stream", None)
        if stream is None:
            stream = torch.arange(self.N, dtype=torch.int64, device=self.device)
        else:
            stream = (stream if torch.is_tensor(stream) else torch.as_tensor(np.asarray(stream, dtype=np.int64)))
            stream = stream.to(self.device, torch.int64).reshape(-1)
            if stream.numel() != self.N:
                raise ValueError(f"stream: one value per cell ({self.N}) expected, got {stream.numel()}")
        nz.setdefault("step0", self.step_index)
        with torch.cuda.device(self.device):
            if nz["T_air_sd"] == 0.0 and nz["P_sd"] == 0.0:
                _lib.check(self.lib.tfg_bind_forcing_noise(self.ctx, None, self.stream_ptr), "tfg_bind_forcing_noise")
                self.forcing_noise = None
                return
            ids, inv = torch.unique(stream, return_inverse=True)
            ids, inv = ids.contiguous(), inv.to(torch.int32).contiguous()
            b = _lib.ForcingNoise(seed=nz["seed"], step0=nz["step0"], T_air_sd=nz["T_air_sd"], T_air_rho=nz["T_air_rho"],
                                  P_sd=nz["P_sd"], P_rho=nz["P_rho"], n_streams=ids.numel(), stream_id=ids.data_ptr(),
                                  cell_stream=inv.data_ptr())
            # the library copies both arrays on the current stream and waits for its range check
            _lib.check(self.lib.tfg_bind_forcing_noise(self.ctx, C.byref(b), self.stream_ptr), "tfg_bind_forcing_noise")
        self.forcing_noise = {**nz, "stream_id": ids, "cell_stream": inv}

    def forcing_noise_series(self, step0: int, n_steps: int):
        """``(dT, fP, stream_id)`` of the bound noise for absolute steps ``[step0, step0 + n_steps)``: ``[n_steps,
        n_streams]`` device tensors of the engine dtype -- the values the kernel applies -- and the ``[n_streams]``
        global ids of their columns.  Cell ``i`` reads column ``forcing_noise["cell_stream"][i]``."""
        if self.forcing_noise is None:
            raise RuntimeError("no forcing noise bound (set_forcing_noise)")
        ids = self.forcing_noise["stream_id"]
        dT = torch.empty(int(n_steps), ids.numel(), dtype=self.dtype, device=self.device)
        fP = torch.empty_like(dT)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.tfg_forcing_noise_series(self.ctx, int(step0), int(n_steps), dT.data_ptr(), fP.data_ptr(),
                                                         self.stream_ptr), "tfg_forcing_noise_series")
        return dT, fP, ids

    # ---- objective: scores of every cell against observations, accumulated inside the melt kernel ----------------
    def set_objective(self, quantity: Optional[str], obs=None, obs_step0: int = 0, obs_index=None) -> None:
        """Score one BMI output of every cell against observations in every later ``run`` (``tfg_bind_objective``).

        ``quantity`` is one of the eight BMI outputs (``REC_NAMES[:8]``: ``h_snow, h_swe, SM, h_ice, h_iwe, IM,
        M_total, RH``); ``None`` unbinds.  ``obs`` is ``[T_obs, n_obs_cols]`` (host or device), row ``j`` the observation
        of absolute step ``obs_step0 + j``; NaN = not observed (daily values of an hourly run, a spin-up period).
        Cell ``i`` reads column ``obs_index[i]``; the default is the forcing map when one is bound (one column per
        catchment), else the identity (``n_obs_cols == N``).  The sums start at zero; ``scores()`` reads them and
        ``reset_objective()`` zeroes them (after ``load_state_dict`` in a calibration loop)."""
        if quantity is None:
            _lib.check(self.lib.tfg_bind_objective(self.ctx, None, self.stream_ptr), "tfg_bind_objective")
            self.objective = None
            return
        q = _lib.REC_BIT.get(quantity, -1)
        if not 0 <= q < 8:
            raise ValueError(f"quantity must be one of the eight BMI outputs {_lib.REC_NAMES[:8]}, got {quantity!r}")
        o = (obs if torch.is_tensor(obs) else torch.as_tensor(np.asarray(obs, dtype=np.float64)))
        if o.dim() != 2 or o.shape[0] < 1 or o.shape[1] < 1:
            raise ValueError(f"obs must be [T_obs, n_obs_cols] with both > 0, got shape {tuple(o.shape)}")
        o = o.to(self.device, torch.float64).contiguous()
        if obs_index is None:
            obs_index = self.forcing_index
        idx = None
        if obs_index is not None:
            idx = (obs_index if torch.is_tensor(obs_index) else torch.as_tensor(np.ascontiguousarray(obs_index)))
            idx = idx.to(self.device, torch.int32).contiguous().reshape(-1)
            if idx.numel() != self.N:
                raise ValueError(f"obs_index must have one entry per cell ({self.N}), got {idx.numel()}")
        elif o.shape[1] != self.N:
            raise ValueError(f"obs must have one column per cell ({self.N}) without obs_index, got {o.shape[1]}")
        acc = torch.zeros(_lib.N_OBJ, self.N, dtype=torch.float64, device=self.device)
        b = _lib.Objective(quantity=q, obs=o.data_ptr(), obs_step0=int(obs_step0), n_obs_steps=o.shape[0],
                           n_obs_cols=o.shape[1], obs_col=idx.data_ptr() if idx is not None else None, acc=acc.data_ptr())
        with torch.cuda.device(self.device):
            _lib.check(self.lib.tfg_bind_objective(self.ctx, C.byref(b), self.stream_ptr), "tfg_bind_objective")
        self.objective = {"quantity": quantity, "obs": o, "obs_step0": int(obs_step0), "obs_index": idx, "acc": acc,
                          "row_counts": np.zeros(o.shape[0], dtype=np.int64), "moments": None}

    def reset_objective(self) -> None:
        """Zero the objective's sums and the count of scored observation rows (e.g. after ``load_state_dict``)."""
        ob = self._objective_or_raise()
        ob["acc"].zero_()
        ob["row_counts"][:] = 0
        ob["moments"] = None

    def objective_sums(self):
        """The kernel's four ``[N]`` float64 sums ``(S_s, S_ss, S_so, S_ee)`` (views of the accumulators)."""
        acc = self._objective_or_raise()["acc"]
        return acc[0], acc[1], acc[2], acc[3]

    def objective_moments(self):
        """``(n, S_o, S_oo)`` of the observations each cell was scored against, ``[N]`` float64 each.

        Formed from ``obs`` and the count of launches that scored each row: rows in time order, each added as often as
        it was scored, with the kernel's operations -- so after one pass over the window they are the bits the kernel
        would form from the observations themselves."""
        from .objective import accumulate_step

        ob = self._objective_or_raise()
        if ob["moments"] is None:
            mom = torch.zeros(3, ob["obs"].shape[1], dtype=torch.float64, device=self.device)
            for j in np.nonzero(ob["row_counts"])[0]:
                for _ in range(int(ob["row_counts"][j])):
                    accumulate_step(None, mom, None, ob["obs"][j])
            ob["moments"] = mom
        m = ob["moments"] if ob["obs_index"] is None else ob["moments"][:, ob["obs_index"].to(torch.int64)]
        return m[0], m[1], m[2]

    def scores(self) -> dict:
        """``{n, nse, kge, r, alpha, beta, rmse, bias}``: ``[N]`` float64 device tensors (``objective.skill_scores``).
        Observation rows scored twice (a rewind without ``reset_objective``) count twice on both sides."""
        from .objective import skill_scores

        return skill_scores(self.objective_sums(), self.objective_moments())

    def _objective_or_raise(self) -> dict:
        if getattr(self, "objective", None) is None:
            raise RuntimeError("no objective bound (set_objective)")
        return self.objective

    def _count_scored_rows(self, step0: int, n_steps: int) -> None:
        """Count the observation rows a run of [step0, step0 + n_steps) scored (for objective_moments)."""
        ob = self.objective
        w0 = ob["obs_step0"]
        lo, hi = max(step0, w0), min(step0 + n_steps, w0 + ob["obs"].shape[0])
        if lo < hi:
            ob["row_counts"][lo - w0:hi - w0] += 1
            ob["moments"] = None

    def _init_state(self, init):
        """Initial state of reference ``initialize()`` (``:350-395``): depths from the config, albedo 0.3,
        cold contents ``max(rho*Cp*h*(T0 - T_surf), 0)`` with ``T_surf = 0``."""
        c = self.consts
        st = self.state
        st.zero_()
        self.row("h_snow").copy_(init["h0_snow"])
        self.row("h_ice").copy_(init["h0_ice"])
        self.row("h_swe").copy_(init["h0_swe"])
        self.row("h_iwe").copy_(init["h0_iwe"])
        self.row("albedo").fill_(0.3)
        del_T = c["T0"] - 0.0
        h_snow64 = init["h0_snow"].to(torch.float64)
        self.row("Eccs").copy_(torch.clamp_min((c["rho_snow"] * c["Cp_snow"]) * h_snow64 * del_T, 0.0).to(self.dtype))
        self.row("Ecci").fill_(max((c["rho_ice"] * c["Cp_ice"]) * c["h_active_layer"] * del_T, 0.0))
        self.ring.zero_()

    def _bind_state(self):
        s = _lib.State()
        for name in STATE_ROWS:
            is_vol = name.startswith("vol_") or name == "P_max"
            ptr = self.row(name).data_ptr() if (self.diag_integrals or not is_vol) else None
            setattr(s, _STATE_FIELD[name], ptr)
        s.ring = self.ring.data_ptr()
        _lib.check(self.lib.tfg_bind_state(self.ctx, C.byref(s)), "tfg_bind_state")
        # running sum of the snowfall window carried between launches (tfg_bind_window_carry); NaN count = re-seed
        self.window_carry = torch.full((3, self.N), float("nan"), dtype=self.dtype, device=self.device)
        _lib.check(self.lib.tfg_bind_window_carry(self.ctx, self.window_carry.data_ptr()), "tfg_bind_window_carry")
        # float32 mode: low parts of h_swe / h_iwe, so that the water-equivalent balances run in float64 (tfg_bind_mass_residual)
        self.mass_lo = None
        if self.mode == _lib.F32:
            self.mass_lo = torch.zeros(2, self.N, dtype=self.dtype, device=self.device)
            _lib.check(self.lib.tfg_bind_mass_residual(self.ctx, self.mass_lo.data_ptr()), "tfg_bind_mass_residual")

    def invalidate_window_sum(self):
        """Call after writing to ``ring`` from outside the kernels: the next launch re-sums the window."""
        self.window_carry[2].fill_(float("nan"))

    def ensure_horizon(self, n_steps: int):
        """Make sure host time tables cover absolute steps ``[0, n_steps)``."""
        if n_steps <= self._n_time:
            return
        n = max(n_steps, 2 * self._n_time)
        tt = time_tables(self.start, self.dt_hours, n)
        rows = np.ascontiguousarray(np.stack([tt[k] for k in ("clock_hour", "TE", "sin_decl", "cos_decl", "tan_decl",
                                                                "isc_e0", "cos_hour", "sin_hour")], axis=1),
                                    dtype=np.float64)
        gmt = utc_offsets(tt["when"], self.zones)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.tfg_bind_time(self.ctx, rows.ctypes.data, gmt.ctypes.data, n, gmt.shape[1], stream),
                   "tfg_bind_time")
        self._n_time = n

    # ---- access ------------------------------------------------------------------------------------------
    def row(self, name: str) -> torch.Tensor:
        """Live ``[N]`` tensor of an input or state variable (internal names)."""
        if name in STATE_ROWS:
            return self.state[STATE_ROWS.index(name)]
        return self.inputs[INPUT_ROWS.index(name)]

    @property
    def stream_ptr(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- the hot path --------------------------------------------------------------------------------------
    def run(self, forcing: torch.Tensor, n_steps: Optional[int] = None, record: Optional[Iterable[str]] = None,
            basin_agg: Optional[torch.Tensor] = None):
        """Advance every cell ``n_steps`` timesteps with ``forcing[T, 5, N]`` (device, engine dtype).

        Returns ``{name: [T, N] tensor}`` for the recorded quantities (empty dict if none).  ``basin_agg``
        (float64 ``[T, n_basin, 3]``) is accumulated into.
        """
        T = int(n_steps if n_steps is not None else forcing.shape[0])
        if forcing.dtype != self.dtype or not forcing.is_cuda or not forcing.is_contiguous():
            raise ValueError("forcing must be a contiguous device tensor of the engine dtype")
        if forcing.numel() < T * _lib.N_FORCING * self.n_cols:
            raise ValueError("forcing block smaller than [n_steps, 5, N]  (N = n_forcing_cols with a forcing map)")
        if self.forcing_index is not None and forcing.dim() == 3 and forcing.shape[2] != self.n_cols:
            raise ValueError(f"forcing must have {self.n_cols} columns (forcing map)")
        self.ensure_horizon(self.step_index + T)
        rec_t, mask, names = None, 0, []
        if record:
            names = sorted(set(record), key=lambda k: _lib.REC_BIT[k])
            for k in names:
                mask |= 1 << _lib.REC_BIT[k]
            rec_t = torch.empty(T, len(names), self.N, dtype=self.dtype, device=self.device)
        if basin_agg is not None:
            if self.basin_id is None or self.n_basin <= 0:
                raise RuntimeError("basin aggregates requested but the engine was built without basin_id / n_basin")
            exact = 0
            if basin_agg.dtype == torch.int64:  # order-independent fixed-point accumulators (sharding.BasinAggregates)
                if basin_agg.numel() < T * self.n_basin * _lib.N_AGG * 2 + 1:
                    raise ValueError("exact basin_agg must be int64 [n_steps * n_basin * 3 * 2 + 1]")
                exact = self.exact_agg_option()
            elif basin_agg.dtype != torch.float64 or basin_agg.numel() < T * self.n_basin * _lib.N_AGG:
                raise ValueError("basin_agg must be float64 [n_steps, n_basin, 3]")
            if exact != self._exact_agg:
                _lib.check(self.lib.tfg_set_option(self.ctx, _lib.OPT_EXACT_AGG, exact), "tfg_set_option")
                self._exact_agg = exact
        with torch.cuda.device(self.device):
            _lib.check(self.lib.tfg_run(
                self.ctx, forcing.data_ptr(), self.step_index, T, rec_t.data_ptr() if rec_t is not None else None,
                mask, basin_agg.data_ptr() if basin_agg is not None else None, self.n_basin, self.stream_ptr),
                "tfg_run")
            if self.objective is not None:
                self._count_scored_rows(self.step_index, T)
        self.step_index += T
        return {k: rec_t[:, i] for i, k in enumerate(names)} if rec_t is not None else {}

    def snapshot_outputs(self, names: Sequence[str], dtype=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``[len(names), N]`` device copy of the named state rows, cast to ``dtype`` (e.g. ``torch.float32`` to halve the
        device->host traffic of a hydrograph product); ``out`` (pinned host tensor) receives it asynchronously on the
        current stream -- synchronise the stream (or record an event) before reading it."""
        rows = torch.tensor([STATE_ROWS.index(k) for k in names], device=self.device)
        snap = self.state.index_select(0, rows)
        if dtype is not None and dtype != snap.dtype:
            snap = snap.to(dtype)
        if out is not None:
            out.copy_(snap, non_blocking=True)
        return snap

    def set_forcing_map(self, forcing_index, n_forcing_cols: Optional[int] = None, _alloc_inputs: bool = True):
        """(Re)bind the cell -> forcing-column map (``None`` restores one column per cell); the input block of the
        per-step path is re-allocated with one column per forcing column."""
        if forcing_index is None:
            self.n_cols, self.forcing_index = self.N, None
            _lib.check(self.lib.tfg_bind_forcing_map(self.ctx, None, 0), "tfg_bind_forcing_map")
        else:
            fi = forcing_index if torch.is_tensor(forcing_index) else torch.as_tensor(np.ascontiguousarray(forcing_index))
            fi = fi.to(self.device, torch.int32).contiguous()
            if fi.numel() != self.N:
                raise ValueError("forcing_index must have one entry per cell")
            n_cols = int(n_forcing_cols) if n_forcing_cols is not None else int(fi.max().item()) + 1
            if int(fi.min().item()) < 0 or int(fi.max().item()) >= n_cols:
                raise ValueError("forcing_index entries must lie in [0, n_forcing_cols)")
            self.n_cols, self.forcing_index = n_cols, fi
            _lib.check(self.lib.tfg_bind_forcing_map(self.ctx, fi.data_ptr(), n_cols), "tfg_bind_forcing_map")
        if _alloc_inputs:
            torch.cuda.synchronize(self.device)
            self.inputs = torch.zeros(len(INPUT_ROWS), self.n_cols, dtype=self.dtype, device=self.device)

    # ---- order-independent basin aggregates (TFG_OPT_EXACT_AGG, include/tfglacier.h) ---------------------------
    def agg_exponents(self):
        """Scaling of the exact aggregates, ``(E0, E1, E2, L)`` (``sharding.agg_scaling``): binary exponents E_q with
        |32-cell partial of aggregate q| < 2^E_q for physically possible values -- M_total < 2^-8 m/s (10 m/h of rain
        is 2.8e-3), water-equivalent depths < 2^17 m -- and the fraction bits L of the low word, chosen from the count
        of contributions to one basin so that neither word can leave the int64 range.  Under ``torch.distributed``
        the largest cell area and the per-basin counts are agreed over all ranks (collective: call on all ranks).
        ``set_agg_exponents`` pins other values instead."""
        if self._agg_exp is None:
            self._agg_exp = self._agg_scaling(reduce=True)
        return self._agg_exp

    def _agg_scaling(self, reduce: bool):
        from .sharding import agg_contributions, agg_scaling

        da_max_t = self.static["da_m2"].max().to(torch.float64)
        counts = torch.stack(agg_contributions(self.basin_id, self.n_basin))
        if reduce:
            try:  # every rank must scale with the SAME exponents, or the integer all-reduce adds apples and pears
                import torch.distributed as dist

                if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                    dist.all_reduce(da_max_t, op=dist.ReduceOp.MAX)   # collective: call on all ranks
                    dist.all_reduce(counts, op=dist.ReduceOp.SUM)
            except ImportError:
                pass
        counts = counts.cpu().numpy()
        return agg_scaling(float(da_max_t.item()), counts[0], counts[1])

    def set_agg_exponents(self, exps) -> None:
        """Scale this engine's exact aggregates with ``exps`` (``(E0, E1, E2)`` or ``(E0, E1, E2, L)``; 3 values mean
        L = 42) instead of its own ``agg_exponents()``.  For engines in one process whose words are added together: all
        must scale alike, e.g. with the exponents of an engine over all their cells.  Exponents smaller than this
        engine's cells need, or an L larger than its own basin counts allow, are refused (ValueError); the caller
        answers for the sum of the counts over the engines it adds."""
        e = tuple(int(x) for x in exps)
        if len(e) == 3:
            e += (42,)
        if len(e) != 4:
            raise ValueError(f"exponents must be (E0, E1, E2) or (E0, E1, E2, L), got {exps!r}")
        need = self._agg_scaling(reduce=False)
        if any(e[q] < need[q] for q in range(3)) or not 1 <= e[3] <= need[3]:
            raise ValueError(f"exact aggregates of this engine need exponents >= {need[:3]} and 1 <= L <= {need[3]}, "
                             f"got {e}")
        self._agg_exp = e

    def exact_agg_option(self) -> int:
        e = self.agg_exponents()
        if not all(-128 <= x < 128 for x in e[:3]):
            raise ValueError("cell areas out of range for exact aggregates")
        return (e[3] << 32) | (1 << 24) | ((e[2] + 128) << 16) | ((e[1] + 128) << 8) | (e[0] + 128)

    def step(self, record: Optional[Iterable[str]] = None):
        """One literal ``update()`` from the current input block."""
        return self.run(self.inputs, 1, record=record)

    def synth_forcing(self, out: torch.Tensor, step0: int, n_steps: int, elev: torch.Tensor, seed: int,
                      storm_cells: int = 1):
        _lib.check(self.lib.tfg_synth_forcing(self.ctx, out.data_ptr(), step0, n_steps, int(out.shape[-1]), elev.data_ptr(), seed,
                                              int(storm_cells), self.stream_ptr), "tfg_synth_forcing")

    # ---- hydrograph routing stand-in (SURVEY.md 8f rank 2) --------------------------------------------------
    def route_fir(self, series: torch.Tensor, weights=None) -> torch.Tensor:
        """Causal FIR along time of float64 ``series[T, M]`` on the device; default = the reference example's
        20-tap 0.05 box "mock routing" (reference ``examples/run_topoflow_glacier.py:129-131``)."""
        w = torch.full((20,), 0.05, dtype=torch.float64) if weights is None else torch.as_tensor(weights, dtype=torch.float64)
        w = w.to(self.device).contiguous()
        x = series.to(self.device, torch.float64).contiguous()
        x2 = x.reshape(x.shape[0], -1)
        out = torch.empty_like(x2)
        _lib.check(self.lib.tfg_route_fir(self.ctx, x2.data_ptr(), out.data_ptr(), w.data_ptr(), w.numel(), x2.shape[0],
                                          x2.shape[1], self.stream_ptr), "tfg_route_fir")
        return out.reshape(x.shape)

    # ---- checkpoint / resume (SURVEY.md 8f rank 3; the reference has none, finalize() is a no-op) ---------------
    def state_dict(self) -> dict:
        """Everything that evolves: state block, snowfall window, inputs and the step counter (CPU tensors)."""
        torch.cuda.synchronize(self.device)
        return {"format": 1, "n_cells": self.N, "dtype": str(self.dtype), "mode": self.mode, "step_index": self.step_index,
                "start": str(self.start), "dt_hours": self.dt_hours, "ring_slots": self.ring_slots,
                "state": self.state.cpu(), "ring": self.ring.cpu(), "inputs": self.inputs.cpu(),
                "mass_lo": None if self.mass_lo is None else self.mass_lo.cpu()}

    def load_state_dict(self, sd: dict) -> None:
        if sd.get("format") != 1:
            raise ValueError("unknown checkpoint format")
        for k, mine in (("n_cells", self.N), ("dtype", str(self.dtype)), ("start", str(self.start)),
                        ("dt_hours", self.dt_hours), ("ring_slots", self.ring_slots)):
            if sd[k] != mine:
                raise ValueError(f"checkpoint {k}={sd[k]!r} does not match this engine ({mine!r})")
        self.state.copy_(sd["state"])
        self.ring.copy_(sd["ring"])
        self.invalidate_window_sum()
        self.inputs.copy_(sd["inputs"])
        if self.mass_lo is not None:
            if sd.get("mass_lo") is not None:
                self.mass_lo.copy_(sd["mass_lo"])
            else:
                self.mass_lo.zero_()
        self.step_index = int(sd["step_index"])
        self.ensure_horizon(self.step_index + 1)

    def measure_fp64_peak(self) -> float:
        """Measured DFMA rate of this GPU in thread-level operations per second (x2 = FP64 FLOP/s)."""
        v = C.c_double()
        _lib.check(self.lib.tfg_measure_fp64_peak(self.ctx, C.byref(v), self.stream_ptr), "tfg_measure_fp64_peak")
        return float(v.value)

    @property
    def column_term_launches(self) -> int:
        """Launches that evaluated the forcing-only terms once per forcing column (``TFG_OPT_COLUMN_TERMS``)."""
        return int(self.lib.tfg_column_term_launches(self.ctx))

    def close(self):
        if getattr(self, "ctx", None):
            torch.cuda.synchronize(self.device)
            self.lib.tfg_destroy(self.ctx)
            self.ctx = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
