"""Ensemble of the shipped catchments under stochastic forcing perturbations, generated on the device.

    python examples/ensemble_topoflow_glacier.py [--members 32] [--T-sd 1.0] [--P-sd 0.3] [--rho 0.9]
                                                 [--mode f64|f64_fast|f32] [--seed 0]

Every catchment of ``config/`` (``cat-*.yaml`` except the ``-const`` variant) runs ``--members`` perturbed members.  All
(catchment, member) pairs are the cells of ONE engine: the forcing map lets the members of a catchment share its
forcing series, and ``MeltEngine(forcing_noise=...)`` gives each member its own stream of noise -- an additive AR(1)
air-temperature error of standard deviation ``--T-sd`` K and a mean-preserving log-normal precipitation factor whose
logarithm has standard deviation ``--P-sd``, both with lag-1 correlation ``--rho`` per hourly step.  Stream ids are
``catchment * members + member``.  A second engine runs the unperturbed catchments for reference.

Per catchment the example prints the ensemble mean and the 5-95 % range of the end-of-run snow water equivalent
``h_swe`` [m] and of the melt summed over the run (``M_total`` times the timestep) [m], and the unperturbed values:

    cat-3062784 swe_end mean=... p05=... p95=... ref=... melt_sum mean=... p05=... p95=... ref=...

Values are printed with 17 significant digits.  ``run()`` returns the same numbers as a dict.
"""

import argparse
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from topoflow_glacier_b200.config import KERNEL_CONSTANTS, TopoflowGlacierConfig, default_constants  # noqa: E402
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


def _swe_and_melt(eng, f_dev, dt_hours):
    """End-of-run h_swe and the summed melt M_total * dt of every cell, float64 on the host."""
    rec = eng.run(f_dev, record=("M_total",))
    melt = (rec["M_total"].double() * (3600.0 * dt_hours)).sum(dim=0)
    return eng.row("h_swe").double().cpu().numpy(), melt.cpu().numpy()


def run(members: int = 32, T_sd: float = 1.0, P_sd: float = 0.3, rho: float = 0.9, mode: str = "f64_fast",
        seed: int = 0, verbose: bool = True) -> dict:
    import torch

    from topoflow_glacier_b200.engine import MeltEngine

    cats = catchments()
    names = [n for n, _ in cats]
    cfgs = [c for _, c in cats]
    C, M = len(cats), int(members)
    if M < 1:
        raise ValueError("--members must be at least 1")
    base = default_constants()
    for k in KERNEL_CONSTANTS:
        if len({float(getattr(c, k)) for c in cfgs}) != 1:
            raise ValueError(f"catchments differ in {k}: one engine runs one set of constants")
        base[k] = float(getattr(cfgs[0], k))
    zone = cfgs[0].utc_offset_hours if cfgs[0].utc_offset_hours is not None else (cfgs[0].tz_name or "America/Los_Angeles")
    series = [convert_on_host(read_forcing_csv(ROOT / c.forcing_file, parse_start(c.start_time),
                                               parse_start(c.end_time))[:, :, None])[:, :, 0] for c in cfgs]
    T = min(s.shape[0] for s in series)
    forcing = np.ascontiguousarray(np.stack([s[:T] for s in series], axis=2))      # [T, 5, C]
    dtype = torch.float32 if mode == "f32" else torch.float64
    f_dev = torch.as_tensor(forcing).to(torch.device("cuda", 0), dtype).contiguous()
    dt = int(cfgs[0].dt)
    kw = dict(zones=[zone], mode=mode, horizon_steps=T + 1, dt_hours=dt)

    # the unperturbed catchments, one cell each
    ref = MeltEngine({k: np.array([float(getattr(c, k)) for c in cfgs]) for k in STATIC_KEYS}, base, cfgs[0].start_time,
                     forcing_index=np.arange(C, dtype=np.int32), n_forcing_cols=C, **kw)
    ref_swe, ref_melt = _swe_and_melt(ref, f_dev, dt)
    ref.close()

    # cell c * M + m is member m of catchment c, with its own stream
    cells = {k: np.repeat([float(getattr(c, k)) for c in cfgs], M) for k in STATIC_KEYS}
    col = np.repeat(np.arange(C, dtype=np.int32), M)
    noise = {"T_air_sd": T_sd, "T_air_rho": rho, "P_sd": P_sd, "P_rho": rho, "seed": int(seed),
             "stream": np.arange(C * M, dtype=np.int64)}
    eng = MeltEngine(cells, base, cfgs[0].start_time, forcing_index=col, n_forcing_cols=C, forcing_noise=noise, **kw)
    swe, melt = _swe_and_melt(eng, f_dev, dt)
    eng.close()

    out = {}
    for c, name in enumerate(names):
        row = {}
        for q, ens, r in (("swe_end", swe, ref_swe), ("melt_sum", melt, ref_melt)):
            v = ens[c * M:(c + 1) * M]
            lo, hi = np.percentile(v, [5.0, 95.0])
            row[q] = {"mean": float(v.mean()), "p05": float(lo), "p95": float(hi), "ref": float(r[c])}
        out[name] = row
    if verbose:
        print(f"{C} catchments x {M} members, {T} steps, mode {mode}, T_sd {T_sd} K, P_sd {P_sd}, rho {rho}, seed {seed}")
        for name, row in out.items():
            print(name + "".join(f" {q} " + " ".join(f"{k}={v:.17g}" for k, v in s.items()) for q, s in row.items()))
    return {"catchments": out, "members": M, "steps": T}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--members", type=int, default=32)
    ap.add_argument("--T-sd", type=float, default=1.0, dest="T_sd")
    ap.add_argument("--P-sd", type=float, default=0.3, dest="P_sd")
    ap.add_argument("--rho", type=float, default=0.9)
    ap.add_argument("--mode", default="f64_fast", choices=("f64", "f64_fast", "f32"))
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args(argv)
    run(a.members, a.T_sd, a.P_sd, a.rho, a.mode, a.seed)


if __name__ == "__main__":
    main()
