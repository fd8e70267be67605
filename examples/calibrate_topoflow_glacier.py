"""Random-search calibration of the five surface parameters over the shipped catchments, scored on the device.

    python examples/calibrate_topoflow_glacier.py [--sets 256] [--mode f64|f64_fast|f32] [--quantity M_total] [--daily]
                                                  [--obs FILE.csv] [--write-obs FILE.csv] [--seed 0] [--forcing-params]

Every catchment of ``config/`` (``cat-*.yaml`` except the ``-const`` variant) gets ``--sets`` candidate parameter sets,
drawn uniformly from the schema's ranges of ``dust_atten, canopy_factor, cloud_factor, z0_air, em_surf``.  All
(catchment, candidate) pairs are the cells of ONE engine: the forcing map lets the candidates of a catchment share its
forcing series, the per-cell parameters give each its own values, and one objective (``MeltEngine.set_objective``)
scores every cell's ``--quantity`` against the catchment's observations inside the melt kernel.  Nothing per step
leaves the device; the result is NSE, KGE, RMSE and bias per candidate.

Observations.  The repository ships none, so without ``--obs`` the example runs a twin experiment: per catchment a
seeded "truth" parameter set is placed among the candidates at a seeded index, and the observations are the
``--quantity`` of one cell per catchment that runs with the truth's parameters (``twin_observations``).  The truth
must then score NSE = 1 exactly and rank first.  The default quantity is the melt runoff ``M_total``: over the shipped
12-day March window some catchments lose their thin snow cover early, so their ``h_swe`` does not depend on the
surface parameters at all and every candidate would tie.  ``--daily`` keeps one observation in 24 (step 12 of each
day, a once-a-day reading); the other rows are NaN.
``--obs FILE.csv`` reads real observations instead: a ``Time`` column (``YYYY-MM-DD HH:MM``) plus one column per
catchment, named after its yaml (``cat-3062784`` ...); a blank cell is a missing observation.
``--write-obs`` writes the observations in that format.
``--forcing-params`` also draws the two forcing parameters that matter most in glacier mass-balance calibration, a
temperature bias ``T_air_offset`` in [-3, 3] K and a precipitation factor ``P_multiplier`` in [0.5, 2]
(``MeltEngine(forcing_adjust=...)``): each candidate then adjusts the catchment's shared series inside the melt kernel.
The twin experiment's truth draws them from the same ranges.

``run()`` returns the best candidate per catchment and all scores, like ``run_topoflow_glacier.run``.
"""

import argparse
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from topoflow_glacier_b200.config import (CELL_PARAM_KEYS, CELL_PARAM_RANGES, KERNEL_CONSTANTS,  # noqa: E402
                                          TopoflowGlacierConfig, default_constants)
from topoflow_glacier_b200.forcing import convert_on_host, read_forcing_csv  # noqa: E402
from topoflow_glacier_b200.timebase import parse_start  # noqa: E402

STATIC_KEYS = ("lat", "lon", "slope", "aspect", "elev", "da", "h0_snow", "h0_ice", "h0_swe", "h0_iwe", "T_rain_snow")


def catchments():
    """(name, validated config) of every shipped catchment yaml."""
    import yaml

    out = []
    for p in sorted((ROOT / "config").glob("cat-*.yaml")):
        if p.stem.endswith("-const"):
            continue
        out.append((p.stem, TopoflowGlacierConfig.model_validate(yaml.safe_load(p.read_text()))))
    return out


# ranges of the forcing parameters drawn with --forcing-params (narrower than the engine accepts)
FORCING_DRAW = {"T_air_offset": (-3.0, 3.0), "P_multiplier": (0.5, 2.0)}


def draw(rng, n, forcing_params=False):
    """n parameter sets, uniform in the schema's ranges (and FORCING_DRAW's with ``forcing_params``): {key: [n]}."""
    out = {k: rng.uniform(lo, hi, n) for k, (lo, hi) in CELL_PARAM_RANGES.items()}
    if forcing_params:
        out.update({k: rng.uniform(lo, hi, n) for k, (lo, hi) in FORCING_DRAW.items()})
    return out


def read_obs_csv(path, names, start, T, dt_hours=1):
    """``[T, len(names)]`` float64 observations from a CSV (``Time`` + one column per catchment; blank = NaN)."""
    import pandas as pd

    df = pd.read_csv(path, float_precision="round_trip")   # the default parser may be off by an ulp
    missing = [n for n in names if n not in df.columns]
    if "Time" not in df.columns or missing:
        raise ValueError(f"{path}: needs a Time column and one column per catchment; missing {['Time'] + missing}")
    obs = np.full((T, len(names)), np.nan)
    step = ((pd.to_datetime(df["Time"]) - start) / pd.Timedelta(hours=dt_hours)).to_numpy()
    ok = (step >= 0) & (step < T) & (step == np.round(step))
    for j, n in enumerate(names):
        obs[step[ok].astype(np.int64), j] = pd.to_numeric(df[n], errors="coerce").to_numpy(dtype=np.float64)[ok]
    return obs


def write_obs_csv(path, obs, names, start, dt_hours=1):
    import pandas as pd

    when = start + pd.to_timedelta(np.arange(obs.shape[0]) * dt_hours, unit="h")
    df = pd.DataFrame({"Time": when.strftime("%Y-%m-%d %H:%M"), **{n: obs[:, j] for j, n in enumerate(names)}})
    df.to_csv(path, index=False, float_format="%.17g", na_rep="")


def twin_observations(cfgs, base, truth, f_dev, quantity, kw):
    """``[T, C]``: ``quantity`` of one cell per catchment that runs with the truth's parameters, after every step.

    The truth cells run the kernel the candidates run (forcing map, per-cell parameters, an objective bound) and are
    read after every step instead of recorded: the float32 unit lets the compiler fuse multiply-adds, so a recording
    kernel may round some products differently from a non-recording one.  Stepping one step at a time gives the same
    state as one launch over all steps."""
    import torch

    from topoflow_glacier_b200.engine import MeltEngine

    C, T = len(cfgs), f_dev.shape[0]
    adjust = {k: np.array([t[k] for t in truth]) for k in FORCING_DRAW if k in truth[0]}
    eng = MeltEngine({k: np.array([float(getattr(c, k)) for c in cfgs]) for k in STATIC_KEYS}, base, cfgs[0].start_time,
                     forcing_index=np.arange(C, dtype=np.int32), n_forcing_cols=C,
                     cell_params={k: np.array([t[k] for t in truth]) for k in CELL_PARAM_KEYS},
                     forcing_adjust=adjust or None, **kw)
    eng.set_objective(quantity, np.full((T, C), np.nan))   # selects the candidates' kernel; nothing is scored
    obs = torch.empty(T, C, dtype=torch.float64, device=f_dev.device)
    for t in range(T):
        eng.inputs[:5].copy_(f_dev[t])
        eng.step()
        obs[t] = eng.row(quantity).double()
    out = obs.cpu().numpy()
    eng.close()
    return out


def run(sets: int = 256, mode: str = "f64_fast", quantity: str = "M_total", daily: bool = False, obs_csv=None,
        write_obs=None, seed: int = 0, verbose: bool = True, forcing_params: bool = False) -> dict:
    import torch

    from topoflow_glacier_b200.engine import MeltEngine

    cats = catchments()
    names = [n for n, _ in cats]
    cfgs = [c for _, c in cats]
    C, K = len(cats), int(sets)
    base = default_constants()
    for k in KERNEL_CONSTANTS:
        vals = {float(getattr(c, k)) for c in cfgs}
        if len(vals) != 1 and k not in CELL_PARAM_KEYS:
            raise ValueError(f"catchments differ in {k}: one engine runs one set of constants")
        base[k] = float(getattr(cfgs[0], k))
    start = parse_start(cfgs[0].start_time)
    zone = cfgs[0].utc_offset_hours if cfgs[0].utc_offset_hours is not None else (cfgs[0].tz_name or "America/Los_Angeles")
    series = [convert_on_host(read_forcing_csv(ROOT / c.forcing_file, parse_start(c.start_time),
                                               parse_start(c.end_time))[:, :, None])[:, :, 0] for c in cfgs]
    T = min(s.shape[0] for s in series)
    forcing = np.ascontiguousarray(np.stack([s[:T] for s in series], axis=2))      # [T, 5, C]
    dtype = torch.float32 if mode == "f32" else torch.float64
    dev = torch.device("cuda", 0)
    f_dev = torch.as_tensor(forcing).to(dev, dtype).contiguous()
    kw = dict(zones=[zone], mode=mode, horizon_steps=T + 1)

    # candidates: cell c * K + k is candidate k of catchment c.  They depend on the seed alone, whatever the source of
    # the observations: one of them, at a seeded index, is the twin experiment's truth (with real observations just
    # one more uniform draw), so a run from a CSV of the twin's observations scores the same candidates.
    rng = np.random.default_rng(seed)
    cand = [draw(rng, K, forcing_params) for _ in range(C)]
    truth = [{k: float(v[0]) for k, v in draw(rng, 1, forcing_params).items()} for _ in range(C)]
    truth_idx = rng.integers(0, K, C)
    keys = tuple(cand[0])
    for c in range(C):
        for k in keys:
            cand[c][k][truth_idx[c]] = truth[c][k]
    cells = {k: np.repeat([float(getattr(c, k)) for c in cfgs], K) for k in STATIC_KEYS}
    params = {k: np.concatenate([cand[c][k] for c in range(C)]) for k in CELL_PARAM_KEYS}
    adjust = {k: np.concatenate([cand[c][k] for c in range(C)]) for k in FORCING_DRAW if k in keys}
    col = np.repeat(np.arange(C, dtype=np.int32), K)

    # observations [T, C]
    if obs_csv is not None:
        obs = read_obs_csv(obs_csv, names, start, T)
    else:
        obs = twin_observations(cfgs, base, truth, f_dev, quantity, kw)
        if daily:
            obs[(np.arange(T) % 24) != 12] = np.nan
    if write_obs:
        write_obs_csv(write_obs, obs, names, start)

    eng = MeltEngine(cells, base, cfgs[0].start_time, forcing_index=col, n_forcing_cols=C, cell_params=params,
                     forcing_adjust=adjust or None, **kw)
    eng.set_objective(quantity, obs)                      # obs_index: the forcing map (one column per catchment)
    eng.run(f_dev)
    sc = {k: v.cpu().numpy() for k, v in eng.scores().items()}
    column_terms = eng.column_term_launches > 0
    eng.close()

    best = []
    for c in range(C):
        nse = sc["nse"][c * K:(c + 1) * K]
        i = int(np.argmax(np.where(np.isnan(nse), -np.inf, nse)))
        best.append({"catchment": names[c], "index": i, "params": {k: float(cand[c][k][i]) for k in keys},
                     **{s: float(sc[s][c * K + i]) for s in ("n", "nse", "kge", "rmse", "bias")}})
    if verbose:
        print(f"{C} catchments x {K} candidates, {T} steps, mode {mode}, objective {quantity}"
              f"{' (daily observations)' if daily else ''}{', forcing parameters' if forcing_params else ''}"
              f"{', column terms' if column_terms else ''}")
        for c, b in enumerate(best):
            tag = "" if obs_csv is not None else f"  truth at {int(truth_idx[c])}"
            print(f"{b['catchment']}: best {b['index']:4d}  NSE {b['nse']:.6f}  KGE {b['kge']:.6f}  RMSE {b['rmse']:.3e}"
                  f"  bias {b['bias']:+.3e}  n {int(b['n'])}{tag}  " + " ".join(f"{k}={v:.4g}" for k, v in b["params"].items()))
    twin = obs_csv is None
    return {"best": best, "scores": sc, "obs": obs, "names": names, "sets": K, "truth": truth if twin else None,
            "truth_index": [int(i) for i in truth_idx] if twin else None, "column_terms": column_terms}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sets", type=int, default=256)
    ap.add_argument("--mode", default="f64_fast", choices=("f64", "f64_fast", "f32"))
    ap.add_argument("--quantity", default="M_total")
    ap.add_argument("--daily", action="store_true")
    ap.add_argument("--obs", default=None)
    ap.add_argument("--write-obs", default=None)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--forcing-params", action="store_true")
    a = ap.parse_args(argv)
    run(a.sets, a.mode, a.quantity, a.daily, a.obs, a.write_obs, a.seed, forcing_params=a.forcing_params)


if __name__ == "__main__":
    main()
