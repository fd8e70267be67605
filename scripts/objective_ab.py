"""A/B of the in-kernel objective: A = no objective, B = objective on h_swe (hourly observations, and daily ones with 23
rows in 24 NaN), C = today's alternative, `record=("h_swe",)` plus a torch reduction of the recorded series against the
observations.  Arms alternate in one process on one engine, so they run the same cells and forcing.  Workloads,
16 777 216 cells, 128 steps per launch, exact basin aggregates:

  raster          per-cell synthetic forcing (the bench raster), f64_fast; cell i reads observation column i // 4096
  sweep_f64_fast  a calibration sweep: 4096 forcing columns x 4096 parameter sets, per-cell parameters, forcing map +
                  column-term pass; each cell reads its catchment's observation column
  sweep_f64       the same sweep in the strict mode

    python scripts/objective_ab.py [--rounds 3] [--out profiles/objective_ab.jsonl]

One JSON line per workload and arm (mean kernel ms over the rounds, spread, G cell-steps/s), preceded by the card's name,
power limit and SM clock read in the same process.  Arms A and B time the launch (CUDA events around `run`); arm C
times the launch and its reduction, and reports the bytes of its recorded series.
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
ap.add_argument("--cols", type=int, default=4096, help="forcing / observation columns")
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--launches", type=int, default=3, help="timed launches per round and arm")
ap.add_argument("--start", type=int, default=2400)
ap.add_argument("--workloads", default="raster,sweep_f64_fast,sweep_f64")
ap.add_argument("--arms", default="A,B_hourly,B_daily,C")
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


def time_record_and_reduce(e, f, agg, obs, obs_col):
    """Arm C: record h_swe for every cell-step, then reduce it against the observations with torch (per step)."""
    times = []
    for _ in range(a.launches):
        e.step_index = a.start
        tgt = agg.zero()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        rec = e.run(f, T, record=("h_swe",), basin_agg=tgt)["h_swe"]
        sums = torch.zeros(4, e.N, dtype=torch.float64, device=dev)
        for t in range(T):
            o = obs[t][obs_col]
            m = torch.isfinite(o)
            s = rec[t]
            d = s - o
            for row, v in enumerate((s, s * s, s * o, d * d)):
                sums[row] = torch.where(m, sums[row] + v, sums[row])
        ev1.record()
        agg.reduce()
        torch.cuda.synchronize()
        times.append(ev0.elapsed_time(ev1))
        del rec
    return sum(times) / len(times), int(T * e.N * 8)


def workload(name):
    mode = "f64" if name == "sweep_f64" else "f64_fast"
    sweep = name.startswith("sweep")
    tabs = synthetic_cells(a.cells, 4096, dev)
    elev = tabs.pop("raw")["elev"]
    cell = torch.arange(a.cells, device=dev, dtype=torch.int64)
    basin = (cell // (-(-a.cells // NB))).to(torch.int32)
    sets = a.cells // a.cols
    obs_col = (cell // sets).to(torch.int32)          # sweep: the catchment; raster: blocks of cells / cols cells
    kw = dict(dt_hours=1, zones=[-8.0], basin_id=basin, n_basin=NB, mode=mode, device_statics=tabs,
              horizon_steps=a.start + (a.launches + 2) * T + 64)
    params = {k: v[cell % sets] for k, v in draws(sets, 7).items()} if sweep else None
    e = MeltEngine(None, default_constants(), "2012100100", cell_params=params, **kw)
    f = torch.empty(T, 5, a.cells, dtype=torch.float64, device=dev)
    e.synth_forcing(f, a.start, T, elev, seed=20121001)
    if sweep:
        f = f[:, :, :a.cols].contiguous()
        e.set_forcing_map(obs_col, a.cols)
    agg = BasinAggregates(T, NB, device=dev, exponents=e.agg_exponents())
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    hourly = torch.rand(T, a.cols, generator=gen, dtype=torch.float64, device=dev)
    daily = hourly.clone()
    daily[(torch.arange(T, device=dev) + a.start) % 24 != 23] = float("nan")
    obs_of = {"B_hourly": hourly, "B_daily": daily}

    def bind(arm):
        if arm in obs_of:
            e.set_objective("h_swe", obs_of[arm], obs_step0=a.start, obs_index=obs_col)
        else:
            e.set_objective(None)

    arms = a.arms.split(",")
    for arm in arms:            # warm-up
        if arm == "C":
            continue
        bind(arm)
        e.step_index = a.start
        e.run(f, T, basin_agg=agg.zero())
    ms = {arm: [] for arm in arms}
    c_bytes = 0
    for _ in range(a.rounds):
        for arm in arms:
            bind(arm)
            if arm == "C":
                k, c_bytes = time_record_and_reduce(e, f, agg, hourly, obs_col)
            else:
                e.step_index = a.start
                k, _ = bench.time_launches(e, f, T, agg.zero, agg.reduce, a.launches, 1, dev)
            ms[arm].append(k)
    out = []
    base = sum(ms[arms[0]]) / len(ms[arms[0]])
    for arm in arms:
        m = sum(ms[arm]) / len(ms[arm])
        rec = {"workload": name, "mode": mode, "arm": arm, "objective": arm.startswith("B"), "cells": a.cells,
               "steps_per_launch": T, "forcing_cols": a.cols if sweep else a.cells, "cell_params": sweep,
               "column_terms": e.column_term_launches > 0, "kernel_ms_mean": round(m, 3),
               "kernel_ms_rounds": [round(x, 3) for x in ms[arm]], "G_cell_steps_per_s": round(a.cells * T / m / 1e6, 2),
               "over_A": round(m / base, 4)}
        if arm == "C":
            rec["recorded_bytes_per_launch"] = c_bytes
            rec["timed"] = "launch with record=('h_swe',) + torch reduction against the observations"
        out.append(rec)
    e.close()
    del f, e
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
