"""ctypes binding of libtfglacier.so (the C ABI declared in include/tfglacier.h).

There is no fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

F64_STRICT, F64_FAST, F32 = 0, 1, 2
MODE_NAMES = {"f64": F64_STRICT, "f64_strict": F64_STRICT, "strict": F64_STRICT, "f64_fast": F64_FAST,
              "fast": F64_FAST, "f32": F32, "fp32": F32, "fp64": F64_STRICT}
OPT_TMA_STAGING = 1
OPT_EXACT_AGG = 2
OPT_COLUMN_TERMS = 3
N_FORCING = 5
N_AGG = 3
MAX_TZ = 8
RING_SLOTS_MAX = 72

# bit positions of recordable quantities (enum tfg_rec)
REC_NAMES = [
    "h_snow", "h_swe", "SM", "h_ice", "h_iwe", "IM", "M_total", "RH", "p0", "e_sat_air", "e_air", "T_dew", "T_surf",
    "e_sat_surf", "Ri", "Dn", "Dh", "Qh", "W_p", "e_surf", "Qe", "TSN_offset", "albedo", "n", "Qn_SW", "em_air",
    "Qn_LW", "Q_sum", "Eccs", "Ecci", "snow3day", "P_rain", "P_snow",
]
REC_BIT = {n: i for i, n in enumerate(REC_NAMES)}


class Constants(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "dt_hours", "T0", "h_active_layer", "rho_air", "rho_snow", "rho_ice", "rho_H2O", "Cp_air", "Cp_snow", "Cp_ice",
        "g", "Lf", "Lv", "eps", "kappa", "latent_heat_constant", "sigma", "sea_level_p0", "uni_gas_const",
        "M_mass_air", "z0_air", "em_surf", "dust_atten", "canopy_factor", "cloud_factor", "z_wind")] + [
        ("satterlund", C.c_int32), ("ring_slots", C.c_int32)]


CELL_PARAM_FIELDS = ("dust_atten", "canopy_factor", "cloud_factor", "z0_air", "em_surf")


class CellParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in CELL_PARAM_FIELDS]


FORCING_ADJUST_FIELDS = ("T_air_offset", "P_multiplier")


class ForcingAdjust(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in FORCING_ADJUST_FIELDS]


class ForcingNoise(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("step0", C.c_int64), ("T_air_sd", C.c_double), ("T_air_rho", C.c_double),
                ("P_sd", C.c_double), ("P_rho", C.c_double), ("n_streams", C.c_int64), ("stream_id", C.c_void_p),
                ("cell_stream", C.c_void_p)]


N_OBJ = 4  # rows of Objective.acc: S_s, S_ss, S_so, S_ee


class Objective(C.Structure):
    _fields_ = [("quantity", C.c_int32), ("obs", C.c_void_p), ("obs_step0", C.c_int64), ("n_obs_steps", C.c_int64),
                ("n_obs_cols", C.c_int64), ("obs_col", C.c_void_p), ("acc", C.c_void_p)]


class TimeRow(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("clock_hour", "TE", "sin_decl", "cos_decl", "tan_decl", "isc_e0",
                                              "cos_hour", "sin_hour")]


STATIC_FIELDS = ("a_elev", "sin_lat", "cos_lat", "neg_tan_lat", "lon", "sin_lat_eq", "cos_lat_eq", "neg_tan_lat_eq",
                 "dlon", "t_noon", "da_m2", "t_rain_snow")


class Statics(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in STATIC_FIELDS] + [("basin_id", C.c_void_p), ("tz_idx", C.c_void_p)]


STATE_FIELDS = ("h_snow", "h_swe", "h_ice", "h_iwe", "eccs", "ecci", "albedo", "n_days", "SM", "IM", "M_total", "RH",
                "vol_P", "vol_PR", "vol_PS", "vol_SM", "vol_IM", "P_max", "ring")


class State(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in STATE_FIELDS]


# name -> (restype, argtypes); every symbol include/tfglacier.h declares
PROTOTYPES = {
    "tfg_abi_version": (C.c_int, []),
    "tfg_last_error": (C.c_char_p, []),
    "tfg_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int]),
    "tfg_destroy": (None, [C.c_void_p]),
    "tfg_mode": (C.c_int, [C.c_void_p]),
    "tfg_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t, C.c_int]),
    "tfg_host_free": (C.c_int, [C.c_void_p]),
    "tfg_host_is_pinned": (C.c_int, [C.c_void_p]),
    "tfg_column_term_launches": (C.c_int64, [C.c_void_p]),
    "tfg_elem_size": (C.c_size_t, [C.c_void_p]),
    "tfg_set_option": (C.c_int, [C.c_void_p, C.c_int, C.c_int64]),
    "tfg_set_constants": (C.c_int, [C.c_void_p, C.POINTER(Constants)]),
    "tfg_bind_static": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(Statics)]),
    "tfg_bind_state": (C.c_int, [C.c_void_p, C.POINTER(State)]),
    "tfg_bind_forcing_map": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "tfg_bind_cell_params": (C.c_int, [C.c_void_p, C.POINTER(CellParams), C.c_void_p]),
    "tfg_bind_objective": (C.c_int, [C.c_void_p, C.POINTER(Objective), C.c_void_p]),
    "tfg_bind_forcing_adjust": (C.c_int, [C.c_void_p, C.POINTER(ForcingAdjust), C.c_void_p]),
    "tfg_bind_forcing_noise": (C.c_int, [C.c_void_p, C.POINTER(ForcingNoise), C.c_void_p]),
    "tfg_forcing_noise_series": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tfg_bind_window_carry": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tfg_bind_mass_residual": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tfg_bind_time": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "tfg_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_uint64, C.c_void_p,
                          C.c_int32, C.c_void_p]),
    "tfg_ingest_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "tfg_convert_forcing": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "tfg_convert_forcing_packed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                             C.c_void_p]),
    "tfg_stream_wait_event": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tfg_route_fir": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int64,
                                C.c_void_p]),
    "tfg_measure_fp64_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "tfg_synth_forcing": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_uint64,
                                    C.c_int64, C.c_void_p]),
}

import os

LIB_PATH = Path(os.environ.get("TFG_LIBRARY") or Path(__file__).resolve().parent / "lib" / "libtfglacier.so")
_lib = None


def load() -> C.CDLL:
    """Load libtfglacier.so (built by ``topoflow_glacier_b200.build``); raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists() and not os.environ.get("TFG_LIBRARY"):
        try:  # same image on the GPU box: nvcc is there, so a missing library can simply be built
            from . import build as _build

            _build.build()
        except Exception:  # noqa: BLE001
            pass
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m topoflow_glacier_b200.build` "
            "(there is no CPU fallback for this path)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.tfg_abi_version() != 1:
        raise RuntimeError("libtfglacier.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().tfg_last_error()
        raise RuntimeError(f"libtfglacier {what}: {msg.decode() if msg else 'unknown error'}")
