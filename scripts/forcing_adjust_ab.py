"""A/B of per-cell forcing adjustments (T_air_offset, P_multiplier), alternated in one process on the same GPU.
16 777 216 cells, 128 steps per launch, exact basin aggregates.  Adjustments are seeded uniform draws, T_air_offset in
[-3, 3] K and P_multiplier in [0.5, 2] (the ranges of examples/calibrate_topoflow_glacier.py --forcing-params).

  raster  per-cell synthetic forcing (the bench raster), f64_fast:  A = nothing bound,  B = adjustments bound
  sweep   4096 forcing columns x 4096 cells each, in f64_fast and f64:
            A = forcing map + column-term pass, nothing bound
            B = forcing map, adjustments bound (the column-term pass is then not taken)
            C = what a user does without the feature: every launch, a torch pass replicates the columns into per-cell
                forcing and adjusts it (index_select, add_, mul_), then the launch reads the per-cell block.  Timed over
                the pass and the launch (``total_ms_mean``); ``kernel_ms_mean`` is the launch alone.

    python scripts/forcing_adjust_ab.py [--rounds 3] [--out profiles/forcing_adjust_ab.jsonl]

One JSON line per workload and arm (mean ms over rounds x launches, the per-round means, G cell-steps/s), the ratios,
and the card's name, power limit and SM clock read in the same process before and after.
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
ap.add_argument("--cols", type=int, default=4096, help="forcing columns of the sweep")
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--launches", type=int, default=3, help="timed launches per round and arm")
ap.add_argument("--start", type=int, default=2400)
ap.add_argument("--workloads", default="raster,sweep_f64_fast,sweep_f64")
ap.add_argument("--out", default=None)
a = ap.parse_args()

dev = torch.device("cuda:0")
T, NB = 128, 4096
RANGES = {"T_air_offset": (-3.0, 3.0), "P_multiplier": (0.5, 2.0)}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(q.split(","), [x.strip() for x in r.stdout.splitlines()[0].split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(dev), "error": str(e)}


def draws(n, seed):
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    return {k: lo + (hi - lo) * torch.rand(n, generator=gen, dtype=torch.float64, device=dev) for k, (lo, hi) in RANGES.items()}


def time_pass_and_launch(e, f_cols, f_cell, idx, adj, agg):
    """Arm C: `launches` x (replicate + adjust + launch); events around each whole iteration and around the launch."""
    tot, ker = [], []
    torch.cuda.synchronize()
    for _ in range(a.launches):
        tgt = agg.zero()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        torch.index_select(f_cols, 2, idx, out=f_cell)
        f_cell[:, 1].add_(adj["T_air_offset"])
        f_cell[:, 0].mul_(adj["P_multiplier"])
        e1.record()
        e.run(f_cell, T, basin_agg=tgt)
        e2.record()
        agg.reduce()
        tot.append((e0, e2))
        ker.append((e1, e2))
    torch.cuda.synchronize()
    return (sum(x.elapsed_time(y) for x, y in ker) / len(ker), sum(x.elapsed_time(y) for x, y in tot) / len(tot))


def workload(name):
    mode = "f64" if name == "sweep_f64" else "f64_fast"
    sweep = name.startswith("sweep")
    tabs = synthetic_cells(a.cells, 4096, dev)
    elev = tabs.pop("raw")["elev"]
    cell = torch.arange(a.cells, device=dev, dtype=torch.int64)
    basin = (cell // (-(-a.cells // NB))).to(torch.int32)
    kw = dict(dt_hours=1, zones=[-8.0], basin_id=basin, n_basin=NB, mode=mode, device_statics=tabs,
              horizon_steps=a.start + (a.launches + 2) * T + 64)
    adj = draws(a.cells, 11)
    arms = {}
    if sweep:    # cell i reads column i // (cells / cols)
        col = (cell // (a.cells // a.cols)).to(torch.int32)
        f = torch.empty(T, 5, a.cols, dtype=torch.float64, device=dev)
        for arm in ("A", "B", "C"):
            fmap = dict(forcing_index=col, n_forcing_cols=a.cols) if arm != "C" else {}
            arms[arm] = MeltEngine(None, default_constants(), "2012100100", forcing_adjust=adj if arm == "B" else None,
                                   **fmap, **kw)
        arms["A"].synth_forcing(f, a.start, T, elev[:a.cols].contiguous(), seed=20121001)
        f_cell = torch.empty(T, 5, a.cells, dtype=torch.float64, device=dev)
        idx = col.to(torch.int64)
    else:
        f = torch.empty(T, 5, a.cells, dtype=torch.float64, device=dev)
        for arm in ("A", "B"):
            arms[arm] = MeltEngine(None, default_constants(), "2012100100", forcing_adjust=adj if arm == "B" else None, **kw)
        arms["A"].synth_forcing(f, a.start, T, elev, seed=20121001)
    agg = BasinAggregates(T, NB, device=dev, exponents=arms["A"].agg_exponents())
    for arm, e in arms.items():     # warm-up, every shape the timed window uses
        e.step_index = a.start
        if arm == "C":
            time_pass_and_launch(e, f, f_cell, idx, adj, agg)
        else:
            e.run(f, T, basin_agg=agg.zero())
    ms = {arm: [] for arm in arms}
    tot = {arm: [] for arm in arms}
    for _ in range(a.rounds):
        for arm, e in arms.items():
            e.step_index = a.start
            if arm == "C":
                k, t = time_pass_and_launch(e, f, f_cell, idx, adj, agg)
            else:
                k, _ = bench.time_launches(e, f, T, agg.zero, agg.reduce, a.launches, 1, dev)
                t = k
            ms[arm].append(k)
            tot[arm].append(t)
    out = []
    for arm, e in arms.items():
        m, mt = sum(ms[arm]) / len(ms[arm]), sum(tot[arm]) / len(tot[arm])
        out.append({"workload": name, "mode": mode, "arm": arm, "forcing_adjust": arm == "B", "torch_pass": arm == "C",
                    "cells": a.cells, "steps_per_launch": T, "forcing_cols": a.cols if sweep and arm != "C" else a.cells,
                    "column_terms": e.column_term_launches > 0, "kernel_ms_mean": round(m, 3),
                    "kernel_ms_rounds": [round(x, 3) for x in ms[arm]], "kernel_ms_spread": round(max(ms[arm]) - min(ms[arm]), 3),
                    "total_ms_mean": round(mt, 3), "total_ms_rounds": [round(x, 3) for x in tot[arm]],
                    "G_cell_steps_per_s": round(a.cells * T / mt / 1e6, 2)})
        e.close()
    r = {o["arm"]: o["total_ms_mean"] for o in out}
    ratios = {"workload": name, "B_over_A": round(r["B"] / r["A"], 4)}
    if "C" in r:
        ratios["C_over_B"] = round(r["C"] / r["B"], 4)
    out.append(ratios)
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
