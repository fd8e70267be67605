"""A/B of per-cell surface parameters: A = no parameters bound, B = per-cell parameters (seeded uniform draws in the
schema ranges), alternated in one process on the same GPU.  Two workloads, 16 777 216 cells, 128 steps per launch,
exact basin aggregates:

  raster  per-cell synthetic forcing (the bench raster), f64_fast
  sweep   a calibration sweep: 4096 forcing columns x 4096 parameter sets, forcing map + column-term pass, in
          f64_fast and f64

    python scripts/cell_params_ab.py [--rounds 3] [--out profiles/cell_params_ab.jsonl]

One JSON line per workload and arm (mean kernel ms over the rounds, spread, G cell-steps/s), preceded by the card's
name, power limit and SM clock read in the same process.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import bench  # noqa: E402
from topoflow_glacier_b200.config import CELL_PARAM_RANGES, default_constants  # noqa: E402
from topoflow_glacier_b200.engine import MeltEngine  # noqa: E402
from topoflow_glacier_b200.sharding import BasinAggregates  # noqa: E402
from topoflow_glacier_b200.synthetic import synthetic_cells  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--cells", type=int, default=1 << 24)
ap.add_argument("--cols", type=int, default=4096, help="forcing columns of the sweep (cells / cols parameter sets each)")
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--launches", type=int, default=3, help="timed launches per round and arm")
ap.add_argument("--start", type=int, default=2400)
ap.add_argument("--workloads", default="raster,sweep_f64_fast,sweep_f64")
ap.add_argument("--out", default=None)
a = ap.parse_args()

dev = torch.device("cuda:0")
T, NB = 128, 4096


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(q.split(","), [x.strip() for x in r.stdout.splitlines()[0].split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(dev), "error": str(e)}


def draws(n_sets, seed):
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    return {k: lo + (hi - lo) * torch.rand(n_sets, generator=gen, dtype=torch.float64, device=dev)
            for k, (lo, hi) in CELL_PARAM_RANGES.items()}


def workload(name):
    mode = "f64" if name == "sweep_f64" else "f64_fast"
    sweep = name.startswith("sweep")
    tabs = synthetic_cells(a.cells, 4096, dev)
    elev = tabs.pop("raw")["elev"]
    cell = torch.arange(a.cells, device=dev, dtype=torch.int64)
    basin = (cell // (-(-a.cells // NB))).to(torch.int32)
    kw = dict(dt_hours=1, zones=[-8.0], basin_id=basin, n_basin=NB, mode=mode, device_statics=tabs,
              horizon_steps=a.start + (a.launches + 2) * T + 64)
    if sweep:   # cell i: catchment i // sets (its forcing column), parameter set i % sets
        sets = a.cells // a.cols
        col = (cell // sets).to(torch.int32)
        params = {k: v[cell % sets] for k, v in draws(sets, 7).items()}
    else:
        col, params = None, draws(a.cells, 7)
    arms = {}
    for arm in ("A", "B"):
        e = MeltEngine(None, default_constants(), "2012100100", cell_params=params if arm == "B" else None, **kw)
        arms[arm] = e
    f = torch.empty(T, 5, a.cells, dtype=torch.float64, device=dev)
    arms["A"].synth_forcing(f, a.start, T, elev, seed=20121001)
    if sweep:
        f = f[:, :, :a.cols].contiguous()
        for e in arms.values():
            e.set_forcing_map(col, a.cols)
    agg = BasinAggregates(T, NB, device=dev, exponents=arms["A"].agg_exponents())
    for e in arms.values():     # warm-up
        e.step_index = a.start
        e.run(f, T, basin_agg=agg.zero())
    ms = {"A": [], "B": []}
    for _ in range(a.rounds):
        for arm, e in arms.items():
            e.step_index = a.start
            k, _ = bench.time_launches(e, f, T, agg.zero, agg.reduce, a.launches, 1, dev)
            ms[arm].append(k)
    out = []
    for arm, e in arms.items():
        m = sum(ms[arm]) / len(ms[arm])
        out.append({"workload": name, "mode": mode, "arm": arm, "cell_params": arm == "B", "cells": a.cells,
                    "steps_per_launch": T, "forcing_cols": a.cols if sweep else a.cells,
                    "column_terms": e.column_term_launches > 0, "kernel_ms_mean": round(m, 3),
                    "kernel_ms_rounds": [round(x, 3) for x in ms[arm]], "G_cell_steps_per_s": round(a.cells * T / m / 1e6, 2)})
        e.close()
    out.append({"workload": name, "B_over_A": round(out[1]["kernel_ms_mean"] / out[0]["kernel_ms_mean"], 4)})
    del f, arms
    torch.cuda.empty_cache()
    return out


lines = [{"gpu": gpu_info(), "torch": torch.__version__}]
print(json.dumps(lines[0]), flush=True)
for w in a.workloads.split(","):
    for rec in workload(w):
        print(json.dumps(rec), flush=True)
        lines.append(rec)
lines.append({"gpu_after": gpu_info()})
print(json.dumps(lines[-1]))
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text("".join(json.dumps(x) + "\n" for x in lines))
