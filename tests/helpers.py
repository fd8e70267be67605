"""Shared test plumbing: golden fixtures -> oracle / device engine, and the parity tolerances."""

from __future__ import annotations

from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parent / "golden"
STATIC_KEYS = ["da", "slope", "aspect", "lon", "lat", "elev", "h0_snow", "h0_ice", "h0_swe", "h0_iwe", "T_rain_snow"]
CASES = ["sample265", "cats288", "const", "allconst", "nosnow", "rand64", "satterlund", "dt2", "year4",
         "cfgspace", "south_dt3", "polar", "dt24", "year2070"]

# |gpu - ref| <= rtol*|ref| + atol, float64 modes.  rtol and atol are SURVEY.md 8a's table; the three departures from
# it are marked and explained in DESIGN.md section 6 together with the worst error achieved per quantity
# (profiles/r2_parity.csv): a relative bound is meaningless where the reference value itself passes through zero.
RTOL = 1e-12
ATOL = {
    "p0": 0, "e_sat_air": 0, "e_air": 0, "RH": 0, "e_sat_surf": 0, "W_p": 0, "Dn": 0, "em_air": 0, "albedo": 0,
    "n": 0, "P_rain": 0, "P_snow": 0, "TSN_offset": 0, "Ri": 0, "Dh": 0, "e_surf": 0,
    "T_dew": 1e-13, "T_surf": 1e-13,      # departure 1: degC values cross 0 (survey: 0); worst achieved 1.2e-14 K
    "Qh": 1e-12, "Qe": 1e-12, "Qn_LW": 1e-12,
    "Qn_SW": 1e-11,                       # departure 2: cos Z cancels at the horizon (survey: 1e-12); worst 3.9e-12 W m-2
    "Q_sum": 1e-9,
    "SM": 3e-18, "IM": 3e-18, "M_total": 3e-18,
    "h_swe": 1e-15, "h_iwe": 1e-15, "h_snow": 1e-15, "h_ice": 1e-15, "Eccs": 1e-6, "Ecci": 1e-6,
    # not in the survey's table: the running window sum (exact only inside its guard band, by design) and the integrals
    "snow3day": 1e-13,                    # departure 3: incremental sum of 72 entries ~1e-3 m; decisions (n) are exact
    "vol_P": 1e-9, "vol_PR": 1e-9, "vol_PS": 1e-9, "vol_SM": 1e-6, "vol_IM": 1e-6, "P_max": 0,
}


def load_case(name: str) -> dict:
    z = np.load(GOLDEN / f"{name}.npz")
    statics = {k: z[f"static_{k}"] for k in STATIC_KEYS}
    N = statics["lat"].size
    forcing = z["forcing"]
    if forcing.shape[2] != N:
        forcing = np.repeat(forcing, N, axis=2)
    ref = {k[4:]: z[k] for k in z.files if k.startswith("ref_")}
    rows = z["rows"] if "rows" in z.files else None
    extra = {k: z[k] for k in z.files if k.startswith("upstream_")}
    consts = {k[6:]: z[k].item() for k in z.files if k.startswith("const_")}  # non-default config values of the case
    dt = int(consts.pop("dt", 1))
    if "SATTERLUND" in consts:
        consts["SATTERLUND"] = bool(consts["SATTERLUND"])
    tz = str(z["tz_name"]) if "tz_name" in z.files else "America/Los_Angeles"
    if "generated_year" in z.files:  # vectors that depend on the year they were generated in (see make_golden.py)
        from datetime import datetime

        if int(z["generated_year"]) != datetime.now().year:
            ref = {}
    return {"name": name, "tz": tz, "statics": statics, "N": N, "forcing": np.ascontiguousarray(forcing), "dt": dt,
            "consts": consts, "start_time": str(z["start_time"]), "ref": ref, "rows": rows, **extra}


def make_oracle(case: dict, strict_pow: bool = False, consts: dict | None = None):
    from oracle.np_ref import CellStatics, Constants, OracleModel

    s = case["statics"]
    cells = CellStatics(**{k: s[k].astype(np.float64) for k in STATIC_KEYS}, tz=[case.get("tz", "America/Los_Angeles")])
    kw = dict(case.get("consts", {}), dt=case.get("dt", 1))
    kw.update(consts or {})
    return OracleModel(cells, Constants(**kw), start_time=case["start_time"], strict_pow=strict_pow)


def default_constants() -> dict:
    from topoflow_glacier_b200.config import default_constants as dc

    return dc()


def make_engine(case: dict, mode: str = "f64", **kw):
    from topoflow_glacier_b200.engine import MeltEngine

    consts = default_constants()
    consts.update(case.get("consts", {}))
    consts.update(kw.pop("consts", {}))
    return MeltEngine(case["statics"], consts, case["start_time"], dt_hours=case.get("dt", 1),
                      zones=[case.get("tz", "America/Los_Angeles")],
                      mode=mode, horizon_steps=case["forcing"].shape[0] + 1, **kw)


def err_report(got: np.ndarray, want: np.ndarray, atol: float, rtol: float = RTOL):
    """(ok, worst ratio err/tol, max abs err, max rel err)."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    both_nan = np.isnan(got) & np.isnan(want)
    diff = np.where(both_nan, 0.0, np.abs(got - want))
    tol = np.where(both_nan, np.inf, rtol * np.abs(want) + atol)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(diff == 0, 0.0, diff / np.where(tol > 0, tol, np.finfo(float).tiny))
        rel = np.where(diff == 0, 0.0, diff / np.maximum(np.abs(want), 1e-300))
    return bool((diff <= tol).all()), float(np.nanmax(ratio)), float(np.nanmax(diff)), float(np.nanmax(rel))



# float32 mode, |gpu - ref| <= rtol*|ref| + atol as (rtol, atol) per quantity: DESIGN.md section 6, "fp32 mode"
F32_TOL = {"Qn_SW": (2e-3, 0.05), "Qn_LW": (2e-3, 0.05), "Qh": (2e-3, 0.05), "Qe": (2e-3, 0.05), "Q_sum": (2e-3, 0.2),
           "RH": (1e-4, 0), "albedo": (1e-5, 0), "T_surf": (1e-4, 1e-3), "SM": (2e-3, 2e-10), "IM": (2e-3, 2e-10),
           "M_total": (2e-3, 2e-10), "h_swe": (1e-3, 1e-5), "h_iwe": (1e-3, 1e-5), "h_snow": (1e-3, 2e-4), "h_ice": (1e-3, 2e-5)}
F32_DEPTHS = ("h_swe", "h_iwe", "h_snow", "h_ice")


def f32_bound_report(got: dict, want: dict, h0_snow: np.ndarray, z0_air: float = 0.01, z: float = 10.0):
    """The stated bound of the float32 mode against the oracle (DESIGN.md section 6): ``(report, failures)``.

    ``got`` / ``want`` map quantities to ``[T, N]`` series (float32 results widened to float64); ``h_snow``, ``h_swe`` and
    ``h_iwe`` must be among them, every other quantity of F32_TOL that both hold is checked.  NaN where both sides have it
    passes (err_report): callers that feed missing data check the NaN pattern themselves.

    (a) Cells whose packs melt out in the same step as in the oracle (or not at all): EVERY cell-step within F32_TOL.
    (b) Cells where a melt-out lands on the other side of a step boundary (a float32 flux error of 1e-3 moves the
        melt-out hour of a thin pack): fluxes and rates within F32_TOL outside +-3 steps of a disagreement of the surface
        class, depths within 1 % + 1e-4 m at the end.  There are at most as many such cells as melt-out events, and
        the surface class disagrees on at most 3 cell-steps per melt-out event.
    Melt-out knife edges (knife_edge_mask: a residue below 1e-12 of the pre-melt depth survives on one side only, DESIGN.md
    section 6) switch the cold content and the melt of the cell from then on, as between the float64 modes and the
    oracle: such cells are exempt from (b)'s depth check and the disagreement count, and there are at most
    max(5, 0.15 x melt-out events) of them.
    Cell-steps in the log-law singularity (condition number of the drag coefficient with respect to h_snow > 1000, see
    test_large_random_sample_with_knife_edges) are excluded from the step they enter it: float32 carries 6e-8 of depth
    error into it.
    """
    T, N = want["h_swe"].shape
    # surface class (snow cover / exhausted pack) disagreement, per cell-step
    same = ((got["h_snow"] > 0) == (want["h_snow"] > 0)) & ((got["h_iwe"] > 0) == (want["h_iwe"] > 0))
    event_cell = ~same.all(axis=0)
    near = ~same
    for sh in range(1, 4):
        near[sh:] |= ~same[:-sh]
        near[:-sh] |= ~same[sh:]
    hs = np.vstack([np.asarray(h0_snow, dtype=np.float64)[None, :], want["h_snow"][:-1]])   # depth the step STARTS from
    arg = (z - hs) / z0_air
    with np.errstate(divide="ignore", invalid="ignore"):
        cond = np.where(arg > 0.01, 2.0 * hs / (np.abs(z - hs) * np.abs(np.log(np.maximum(arg, 1e-300)))), 0.0)
    singular = np.maximum.accumulate(np.nan_to_num(cond, posinf=np.inf) > 1000.0, axis=0)
    w_swe, w_iwe = np.nan_to_num(want["h_swe"]), np.nan_to_num(want["h_iwe"])
    melt_outs = int(((w_swe[:-1] > 0) & (w_swe[1:] == 0)).sum() + ((w_iwe[:-1] > 0) & (w_iwe[1:] == 0)).sum())
    knife = knife_edge_mask({k: np.nan_to_num(got[k]) for k in ("h_swe", "h_iwe")},
                            {k: np.nan_to_num(want[k]) for k in ("h_swe", "h_iwe")})[-1]
    disagree = int((~same)[:, event_cell & ~knife].sum())
    rep = {"cells": N, "steps": T, "cells_with_shifted_melt_out": int(event_cell.sum()), "melt_out_events": melt_outs,
           "log_law_singular_cells": int(singular[-1].sum()), "knife_edge_cells": int(knife.sum()),
           "disagreeing_cell_steps": disagree}
    bad = []
    for k, (rt, at) in F32_TOL.items():
        if k not in got or k not in want:
            continue
        keep = ~singular & ~near
        if k in F32_DEPTHS:   # (a): every step of the cells without an event
            keep = ~singular & ~event_cell[None, :]
        ok, ratio, dabs, drel = err_report(got[k][keep], want[k][keep], at, rt)
        rep[k] = {"ok": ok, "err_over_tol": ratio, "max_abs": dabs, "max_rel": drel}
        if not ok:
            bad.append((k, ratio, dabs, drel))
    for k in F32_DEPTHS:   # (b): event cells, end of run
        sel = event_cell & ~singular[-1] & ~knife
        if k in got and k in want and sel.any():
            ok, ratio, dabs, drel = err_report(got[k][-1][sel], want[k][-1][sel], 1e-4, 1e-2)
            rep[k + "@end,event cells"] = {"ok": ok, "err_over_tol": ratio, "max_abs": dabs, "max_rel": drel}
            if not ok:
                bad.append((k + "@end", ratio, dabs, drel))
    if event_cell.sum() > max(1, melt_outs):
        bad.append(("cells_with_shifted_melt_out", int(event_cell.sum()), "> melt-out events", melt_outs))
    if knife.sum() > max(5, 0.15 * melt_outs):
        bad.append(("knife_edge_cells", int(knife.sum()), "> max(5, 0.15 x melt-out events)", melt_outs))
    if disagree > 3 * max(1, melt_outs):
        bad.append(("disagreeing_cell_steps", disagree, "> 3 x melt-out events", melt_outs))
    return rep, bad


def knife_edge_mask(got: dict, want: dict) -> np.ndarray:
    """Cells whose state left the oracle's trajectory through a melt-out knife edge (boolean ``[T, N]``).

    The reference lets SWE/IWE reach *exactly* zero through ``min(M*3600, h)/3600*dt*3600`` (reference
    ``bmi_topoflow_glacier.py:1601-1606``); whether a residue of ~1e-19 m survives depends on the last bits of
    ``h``, and a surviving residue switches albedo, the surface-temperature cap and the ice-melt gate for a step
    or two.  Two implementations whose transcendental functions differ by 1 ulp therefore disagree on a few per
    cent of melt-out events by O(1) for a step, and by the skipped melt ever after.  Such a cell is masked from
    the step where one side holds an exact zero and the other a residue below 1e-12 of the pre-melt depth.
    """
    T, N = want["h_swe"].shape
    mask = np.zeros((T, N), dtype=bool)
    for key in ("h_swe", "h_iwe"):
        g, w = got[key], want[key]
        prev = np.vstack([np.full((1, N), np.inf), np.maximum(np.abs(w[:-1]), np.abs(g[:-1]))])
        residue = ((g == 0) != (w == 0)) & (np.maximum(np.abs(g), np.abs(w)) <= 1e-12 * np.maximum(prev, 1e-6))
        mask |= np.maximum.accumulate(residue, axis=0)
    return mask
