"""Schema of ``config/cat-*.yaml`` (drop-in for reference ``src/topoflow_glacier/bmi/config.py:6-115``).

Field names, types, defaults and range checks are the reference's; the model is generated from one
table so that the constants the kernels consume and the schema cannot drift apart.  Differences, all
backwards compatible:

* ``start_time`` / ``end_time`` given as YAML integers are coerced to ``str`` (three of the five shipped
  configs hold unquoted integers, which the reference's ``str`` field rejects);
* optional extension keys (ignored by the reference): ``tz_name`` / ``utc_offset_hours`` (the reference looks
  the zone up with ``timezonefinder``; here the zone is data), ``precision``, ``device``, ``ensemble``,
  and the per-cell forcing adjustments ``T_air_offset`` [K] / ``P_multiplier`` [-] (``FORCING_ADJUST_RANGES``).  The
  schema's legacy ``P_factor`` stays parsed and ignored, as in the reference.
"""

from __future__ import annotations

from typing import Any, Optional

from pydantic import ConfigDict, Field, create_model, field_validator

__all__ = ["TopoflowGlacierConfig", "KERNEL_CONSTANTS", "CELL_PARAM_KEYS", "CELL_PARAM_RANGES", "check_cell_params",
           "FORCING_ADJUST_KEYS", "FORCING_ADJUST_RANGES", "FORCING_ADJUST_IDENTITY", "check_forcing_adjust",
           "default_constants"]

_REQ = ...  # pydantic's "required" marker

# name: (type, default, constraints, description)
_TABLE: dict[str, tuple[type, Any, dict, str]] = {
    # -- required per-catchment configuration ----------------------------------------------------------
    "site_prefix": (str, _REQ, {}, "File prefix for the study site"),
    "forcing_file": (str, _REQ, {}, "Forcing .csv file"),
    "dt": (int, _REQ, {"ge": 0}, "Timestep of the snowmelt process [h]"),
    "start_time": (str, _REQ, {}, "Start of the run, YYYYMMDDHH"),
    "end_time": (str, _REQ, {}, "End of the run, YYYYMMDDHH"),
    "da": (float, _REQ, {}, "Drainage area [km2]"),
    "slope": (float, _REQ, {}, "Catchment slope [m km-1]"),
    "lat": (float, _REQ, {}, "Centroid latitude [deg]"),
    "lon": (float, _REQ, {}, "Centroid longitude [deg east]"),
    "h0_snow": (float, _REQ, {}, "Initial snow depth [m]"),
    "h0_ice": (float, _REQ, {}, "Initial ice thickness [m]"),
    "h0_swe": (float, _REQ, {}, "Initial snow water equivalent [m]"),
    "h0_iwe": (float, _REQ, {}, "Initial ice water equivalent [m]"),
    "elev": (float, _REQ, {}, "Mean elevation [m]"),
    "T_rain_snow": (float, 1.0, {}, "Rain/snow air-temperature threshold [degC]"),
    "aspect": (float, 0.0, {}, "Aspect angle"),
    "dust_atten": (float, 0.08, {"ge": 0.0, "le": 0.2}, "Aerosol/dust attenuation of transmittance"),
    "canopy_factor": (float, 0.0, {"ge": 0.0, "le": 1.0}, "Canopy factor"),
    "cloud_factor": (float, 0.0, {"ge": 0.0, "le": 1.0}, "Cloud fraction"),
    # -- physical constants ---------------------------------------------------------------------------
    "rho_air": (float, 1.2614, {}, "[kg m-3]"),
    "rho_snow": (float, 50.0, {}, "[kg m-3]"),
    "rho_ice": (float, 917.0, {}, "[kg m-3]"),
    "rho_H2O": (float, 1000.0, {}, "[kg m-3]"),
    "h_active_layer": (float, 0.125, {}, "Active ice layer [m]"),
    "T0": (float, -0.2, {}, "Reference temperature [degC]"),
    "Cp_air": (float, 1005.7, {}, "[J kg-1 K-1]"),
    "Cp_ice": (float, 2060.0, {}, "[J kg-1 K-1]"),
    "Cp_snow": (float, 2090.0, {}, "[J kg-1 K-1]"),
    "g": (float, 9.81, {}, "[m s-2]"),
    "Lf": (float, 334000.0, {}, "Latent heat of fusion [J kg-1]"),
    "eps": (float, 0.622, {}, "Ratio of gas constants"),
    "kappa": (float, 0.408, {}, "von Karman constant"),
    "latent_heat_constant": (float, 0.622, {}, "Dingman (2002, p. 273)"),
    "Lv": (float, 2500000, {}, "Latent heat of vaporisation [J kg-1]"),
    "sigma": (float, 5.67 * 10 ** (-8), {}, "Stefan-Boltzmann [W m-2 K-4]"),
    "sea_level_p0": (float, 101325.0, {}, "[Pa]"),
    "sea_level_T0": (float, 288.15, {}, "[K]"),
    "T_lapse_rate": (float, 0.0065, {}, "[K m-1]"),
    "uni_gas_const": (float, 8.3144598, {}, "[J mol-1 K-1]"),
    "M_mass_air": (float, 0.0289644, {}, "[kg mol-1]"),
    # -- glacier-dynamics keys: parsed, never read by the melt path --------------------------------------
    "min_glacier_thick": (float, 1.0, {}, ""), "glens_A": (float, 2.142e-16, {}, ""), "B": (float, 0.0012, {}, ""),
    "char_sliding_vel": (float, 10.0, {}, ""), "char_tau_bed": (float, 100000.0, {}, ""),
    "depth_to_water_table": (float, 20.0, {}, ""), "max_float_fraction": (float, 80.0, {}, ""),
    "Hp_eff": (float, 20.0, {}, ""), "init_ELA": (float, 3350.0, {}, ""), "ELA_step_size": (float, -10.0, {}, ""),
    "ELA_step_interval": (float, 500.0, {}, ""), "grad_Bz": (float, 0.01, {}, ""), "max_Bz": (float, 2.0, {}, ""),
    "spinup_time": (float, 200.0, {}, ""), "sea_level": (float, -100.0, {}, ""),
    "z0_air": (float, 0.01, {"ge": 0.0001, "le": 0.1}, "Surface roughness length [m]"),
    "em_surf": (float, 0.985, {"ge": 0.9, "le": 1}, "Surface emissivity"),
    "geothermal_heat_flux": (float, 1575000.0, {}, ""), "geothermal_gradient": (float, -0.0255, {}, ""),
    # -- legacy toggles ---------------------------------------------------------------------------------
    "PRECIP_ONLY": (bool, False, {}, ""), "P_factor": (float, 1.0, {}, ""),
    "SATTERLUND": (bool, False, {}, "Satterlund (1979) e_sat / em_air"),
    # -- extensions (optional) --------------------------------------------------------------------------
    "tz_name": (Optional[str], None, {}, "IANA zone of the catchment (replaces the timezonefinder lookup)"),
    "utc_offset_hours": (Optional[float], None, {}, "Fixed UTC offset [h]; overrides tz_name"),
    "precision": (str, "f64", {}, "f64 | f64_fast | f32"),
    "device": (int, 0, {}, "CUDA device ordinal"),
    "ensemble": (Optional[list], None, {}, "Further config files advanced as extra cells of the same model"),
    "T_air_offset": (float, 0.0, {"ge": -30.0, "le": 30.0}, "Added to the forcing's air temperature [K]"),
    "P_multiplier": (float, 1.0, {"ge": 0.0, "le": 10.0}, "Multiplies the forcing's precipitation rate [-]"),
}

# constants handed to the kernels (tfg_constants in include/tfglacier.h)
KERNEL_CONSTANTS = ("T0", "h_active_layer", "rho_air", "rho_snow", "rho_ice", "rho_H2O", "Cp_air", "Cp_snow",
                    "Cp_ice", "g", "Lf", "Lv", "eps", "kappa", "latent_heat_constant", "sigma", "sea_level_p0",
                    "uni_gas_const", "M_mass_air", "z0_air", "em_surf", "dust_atten", "canopy_factor", "cloud_factor")


# per-catchment tunables that may also be given per cell (MeltEngine(cell_params=...), tfg_bind_cell_params)
CELL_PARAM_KEYS = ("dust_atten", "canopy_factor", "cloud_factor", "z0_air", "em_surf")
CELL_PARAM_RANGES = {k: (_TABLE[k][2]["ge"], _TABLE[k][2]["le"]) for k in CELL_PARAM_KEYS}


def check_cell_params(params) -> dict:
    """Validate per-cell parameter arrays (NumPy arrays or torch tensors, any device) against the schema's ranges.

    Returns ``params`` as a plain dict; raises ``ValueError`` naming the first unknown key, or the first key holding a
    value that is not finite or outside its range."""
    params = dict(params)
    for k, v in params.items():
        if k not in CELL_PARAM_RANGES:
            raise ValueError(f"{k!r} is not a per-cell parameter (one of {', '.join(CELL_PARAM_KEYS)})")
        lo, hi = CELL_PARAM_RANGES[k]
        if not bool(((v >= lo) & (v <= hi)).all()):   # NaN and +-inf compare false
            raise ValueError(f"{k}: every value must be finite and within [{lo}, {hi}]")
    return params


# per-cell adjustments of the forcing a cell reads (MeltEngine(forcing_adjust=...), tfg_bind_forcing_adjust)
FORCING_ADJUST_KEYS = ("T_air_offset", "P_multiplier")
FORCING_ADJUST_RANGES = {k: (_TABLE[k][2]["ge"], _TABLE[k][2]["le"]) for k in FORCING_ADJUST_KEYS}
FORCING_ADJUST_IDENTITY = {k: _TABLE[k][1] for k in FORCING_ADJUST_KEYS}


def check_forcing_adjust(adjust) -> dict:
    """Validate per-cell forcing adjustments (NumPy arrays or torch tensors, any device) against their ranges.

    Returns ``adjust`` as a plain dict; raises ``ValueError`` naming the first unknown key, or the first key holding a
    value that is not finite or outside its range."""
    adjust = dict(adjust)
    for k, v in adjust.items():
        if k not in FORCING_ADJUST_RANGES:
            raise ValueError(f"{k!r} is not a forcing adjustment (one of {', '.join(FORCING_ADJUST_KEYS)})")
        lo, hi = FORCING_ADJUST_RANGES[k]
        if not bool(((v >= lo) & (v <= hi)).all()):   # NaN and +-inf compare false
            raise ValueError(f"{k}: every value must be finite and within [{lo}, {hi}]")
    return adjust


def _coerce_time(cls, v):  # noqa: ANN001
    return str(v) if isinstance(v, int) and not isinstance(v, bool) else v


TopoflowGlacierConfig = create_model(
    "TopoflowGlacierConfig",
    __config__=ConfigDict(arbitrary_types_allowed=True),
    __validators__={"_coerce_time": field_validator("start_time", "end_time", mode="before")(_coerce_time)},
    **{name: (tp, Field(default, description=desc, **cons)) for name, (tp, default, cons, desc) in _TABLE.items()},
)
TopoflowGlacierConfig.__doc__ = "Validates a topoflow-glacier catchment configuration."


def default_constants() -> dict:
    """Every defaulted field of the schema as a plain dict (the physical constants of a stock run)."""
    return {k: v[1] for k, v in _TABLE.items() if v[1] is not _REQ}
