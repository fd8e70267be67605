"""Cost of stochastic forcing perturbations, arms alternated in one process on the same GPU.
Bench raster: 16 777 216 cells of per-cell synthetic forcing, f64_fast, 128 steps per run, exact basin aggregates.

  A  nothing bound
  B  forcing adjustments only (seeded T_air_offset in [-3, 3] K, P_multiplier in [0.5, 2])
  C  adjustments + noise with 4096 streams (4096 consecutive cells per stream: an ensemble member spread over cells)
  D  adjustments + noise with one stream per cell: the [steps][2][n_streams] scratch is capped at 2 GB, so tfg_run
     splits each 128-step run into launches of 8 steps
  P  the noise pre-pass alone (forcing_noise_series, the same kernel), for C's 4096 streams x 128 steps and for D's
     16 777 216 streams x 8 steps

    python scripts/forcing_noise_ab.py [--rounds 3] [--out profiles/forcing_noise_ab.jsonl]

CUDA events around every run (one ``MeltEngine.run`` of 128 steps, pre-pass included).  One JSON line per arm (mean ms
over rounds x runs, per-round means, G cell-steps/s), the ratios, and the card's name, power limit and SM clock read in
the same process before and after.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import bench  # noqa: E402
from topoflow_glacier_b200.config import default_constants  # noqa: E402
from topoflow_glacier_b200.engine import MeltEngine  # noqa: E402
from topoflow_glacier_b200.sharding import BasinAggregates  # noqa: E402
from topoflow_glacier_b200.synthetic import synthetic_cells  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--cells", type=int, default=1 << 24)
ap.add_argument("--streams", type=int, default=4096)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--launches", type=int, default=3, help="timed runs of 128 steps per round and arm")
ap.add_argument("--start", type=int, default=2400)
ap.add_argument("--out", default=None)
a = ap.parse_args()

dev = torch.device("cuda:0")
T, NB = 128, 4096
RANGES = {"T_air_offset": (-3.0, 3.0), "P_multiplier": (0.5, 2.0)}
NOISE = {"T_air_sd": 1.0, "T_air_rho": 0.9, "P_sd": 0.3, "P_rho": 0.9, "seed": 7}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(q.split(","), [x.strip() for x in r.stdout.splitlines()[0].split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(dev), "error": str(e)}


def time_series(e, n_steps, reps=5):
    """Mean ms of forcing_noise_series(start, n_steps): the pre-pass kernel over n_steps steps of every stream."""
    e.forcing_noise_series(a.start, n_steps)          # warm-up
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        e.forcing_noise_series(a.start, n_steps)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


lines = [{"gpu": gpu_info(), "torch": torch.__version__}]
print(json.dumps(lines[0]), flush=True)
tabs = synthetic_cells(a.cells, 4096, dev)
elev = tabs.pop("raw")["elev"]
cell = torch.arange(a.cells, device=dev, dtype=torch.int64)
basin = (cell // (-(-a.cells // NB))).to(torch.int32)
kw = dict(dt_hours=1, zones=[-8.0], basin_id=basin, n_basin=NB, mode="f64_fast", device_statics=tabs,
          horizon_steps=a.start + (a.launches + 2) * T + 64)
gen = torch.Generator(device=dev)
gen.manual_seed(11)
adj = {k: lo + (hi - lo) * torch.rand(a.cells, generator=gen, dtype=torch.float64, device=dev) for k, (lo, hi) in RANGES.items()}
noise = {"C": dict(NOISE, step0=a.start, stream=cell // (a.cells // a.streams)), "D": dict(NOISE, step0=a.start)}
arms = {}
for arm in ("A", "B", "C", "D"):
    arms[arm] = MeltEngine(None, default_constants(), "2012100100", forcing_adjust=adj if arm != "A" else None,
                           forcing_noise=noise.get(arm), **kw)
f = torch.empty(T, 5, a.cells, dtype=torch.float64, device=dev)
arms["A"].synth_forcing(f, a.start, T, elev, seed=20121001)
agg = BasinAggregates(T, NB, device=dev, exponents=arms["A"].agg_exponents())
for arm, e in arms.items():     # warm-up, every shape the timed window uses
    e.step_index = a.start
    e.run(f, T, basin_agg=agg.zero())
ms = {arm: [] for arm in arms}
for _ in range(a.rounds):
    for arm, e in arms.items():
        e.step_index = a.start
        k, _ = bench.time_launches(e, f, T, agg.zero, agg.reduce, a.launches, 1, dev)
        ms[arm].append(k)
out = []
for arm, e in arms.items():
    m = sum(ms[arm]) / len(ms[arm])
    nz = e.forcing_noise
    out.append({"workload": "raster", "mode": "f64_fast", "arm": arm, "forcing_adjust": arm != "A",
                "noise_streams": int(nz["stream_id"].numel()) if nz else 0, "cells": a.cells, "steps_per_run": T,
                "run_ms_mean": round(m, 3), "run_ms_rounds": [round(x, 3) for x in ms[arm]],
                "run_ms_spread": round(max(ms[arm]) - min(ms[arm]), 3), "G_cell_steps_per_s": round(a.cells * T / m / 1e6, 2)})
r = {o["arm"]: o["run_ms_mean"] for o in out}
out.append({"ratios": {"B_over_A": round(r["B"] / r["A"], 4), "C_over_B": round(r["C"] / r["B"], 4),
                       "D_over_B": round(r["D"] / r["B"], 4)}})
split = max(1, min(T, (1 << 31) // (a.cells * 2 * 8)))
out.append({"arm": "P", "pre_pass_ms": {f"{a.streams}_streams_x_{T}_steps": round(time_series(arms["C"], T), 3),
                                         f"{a.cells}_streams_x_{split}_steps": round(time_series(arms["D"], split), 3)}})
for rec in out:
    print(json.dumps(rec), flush=True)
    lines.append(rec)
for e in arms.values():
    e.close()
lines.append({"gpu_after": gpu_info()})
print(json.dumps(lines[-1]))
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text("".join(json.dumps(x) + "\n" for x in lines))
