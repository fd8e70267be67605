#!/usr/bin/env python
"""bench.py -- cell-timesteps/sec of the fused energy-balance + melt kernel on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mode f64_fast|f64|f32] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[3], SURVEY.md 8d cfg 4): a synthetic 4096 x 4096 glacierised raster
(16 777 216 cells) PER GPU, hourly forcing, advanced in chunks of ``--chunk`` (default 128) timesteps.
One bench "step" = one launch of the fused kernel over one forcing chunk for every cell of the rank
(+ the all-reduce of the per-basin aggregates when N > 1).  Weak scaling: per-GPU work is fixed.

* ``value``      whole-job cell-steps/s with the forcing chunk resident in HBM (86 GB in float64: far larger than
                 L2, so no flush is needed between launches);
* ``roofline``   the melt kernel alone, CUDA events on the launching stream; algorithmic bytes = 5 live forcings x
                 element size per cell-step (40 B float64 / 20 B float32), peak = MEASURED_PEAKS.json hbm_gbs;
* ``e2e``        the same metric through the public API with HOST buffers: pinned raw met columns ->
                 ForcingStreamer (cudaMemcpyAsync on a side stream + unit-conversion kernel) -> tfg_run ->
                 device->host copy of the eight BMI outputs and the basin aggregates, all inside the timed region;
* ``cpu_baseline``  the NumPy oracle (a port of the reference: kind "port") on all host cores, on a bounded
                 sample of the same cells and forcing; the sample is also used to check the GPU result.

``--impl reference`` times that CPU port alone (the reference itself is a pure-Python package whose build
backend is not installable offline, see DESIGN.md) and prints the line with "impl": "reference".

``--dump-outputs DIR`` writes, after the timed launches, what the last of them handed its caller (``dump_outputs``).
Cells and forcing are seeded, so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "cell_timesteps_per_sec"
UNIT = "cell-steps/s"
GRID_CELLS = 4096 * 4096
REGIONAL_CELLS = 100_000_000
N_BASIN = 4096
BMI_OUTPUTS = ("h_snow", "h_swe", "SM", "h_ice", "h_iwe", "IM", "M_total", "RH")
DUMP_CELLS = 1 << 18          # cells sampled per state row: 2 MB each in float64
DUMP_AGG_BYTES = 32 << 20     # basin aggregates: as many of the launch's last timesteps as fit


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.mark = index, [], None, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            # nvidia-smi needs a few hundred ms to come up (longer on an 8-GPU box): wait for its first line so that
            # a timed region of a few hundred ms is sampled from its first millisecond; only later rows are counted
            t0 = time.monotonic()
            while not self.rows and time.monotonic() - t0 < 8.0 and self.proc.poll() is None:
                time.sleep(0.02)
            self.mark = len(self.rows)
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in (self.rows[self.mark:] or self.rows[-1:]):   # the rows of the timed region (else the one just before it)
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------- CPU arm
def _oracle_worker(args):
    import numpy as np

    from oracle.np_ref import CellStatics, Constants, OracleModel

    statics, forcing, start, reps = args
    cells = CellStatics(**statics, tz=[-8.0])
    model = OracleModel(cells, Constants(), start, strict_pow=False)
    t0 = time.perf_counter()
    out = None
    for _ in range(reps):
        for t in range(forcing.shape[0]):
            out = model.step(*forcing[t])
    dt = time.perf_counter() - t0
    return dt, {k: np.array(out[k]) for k in ("M_total", "h_swe", "h_iwe", "RH")}


def cpu_port_throughput(statics: dict, forcing, start: str, cores: int, reps: int = 1):
    """All host cores, one oracle instance per core on its slice of the sample cells."""
    import multiprocessing as mp

    import numpy as np

    n = statics["lat"].size
    bounds = np.linspace(0, n, cores + 1).astype(int)
    jobs = []
    for i in range(cores):
        lo, hi = bounds[i], bounds[i + 1]
        if hi > lo:
            jobs.append(({k: v[lo:hi] for k, v in statics.items()}, np.ascontiguousarray(forcing[:, :, lo:hi]), start, reps))
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        res = pool.map(_oracle_worker, jobs)
    wall = time.perf_counter() - t0
    busy = max(r[0] for r in res)
    last = {k: np.concatenate([r[1][k] for r in res]) for k in res[0][1]}
    return n * forcing.shape[0] * reps / busy, wall, last


# ---- the UNMODIFIED reference (baseline/_ref, scripts/install_reference.py): one BMI instance per cell ------------------
REF_DIR = ROOT / "baseline" / "_ref"
SAMPLE_CONFIG = {  # the reference's own test configuration (tests/integration_test.py:18-38)
    "site_prefix": "cat-3062920", "forcing_file": "data/sample-cat-3062920.csv", "dt": 1, "start_time": "2013032000",
    "end_time": "2013033100", "da": 11.418749923500716, "slope": 88.582729, "aspect": 242.8644693769529,
    "lon": -121.81418, "lat": 46.81953220, "elev": 2446.3922737596167, "h_active_layer": 0.125, "h0_snow": 5.0,
    "h0_ice": 2.0, "h0_swe": 0.25, "h0_iwe": 1.834, "T_rain_snow": 0.0,
}


def reference_available() -> bool:
    return (REF_DIR / "topoflow_glacier" / "bmi" / "bmi_topoflow_glacier.py").exists()


def _reference_worker(args):
    """`n_inst` reference instances, each driven through the reference's own per-step loop (7 x set_value, update(),
    get_value; examples/run_topoflow_glacier.py:64-109) over the sample forcing."""
    n_inst, n_steps, seed = args
    import tempfile

    import numpy as np
    import pandas as pd
    import yaml

    os.environ["NGEN_EWTS_LOGGING"] = "DISABLED"
    devnull = os.open(os.devnull, os.O_WRONLY)   # the reference prints its logging banner on every construct: this
    os.dup2(devnull, 1)                          # worker's stdout must not reach the ONE JSON line of the parent
    for m in [m for m in sys.modules if m == "topoflow_glacier" or m.startswith("topoflow_glacier.")]:
        del sys.modules[m]   # never the drop-in package of the same name
    sys.path[:] = [str(REF_DIR)] + [q for q in sys.path if Path(q or ".").resolve() != ROOT]
    import topoflow_glacier

    assert str(REF_DIR) in topoflow_glacier.__file__, topoflow_glacier.__file__
    df = pd.read_csv(REF_DIR / "data" / "sample-cat-3062920.csv").iloc[:n_steps]
    P = df["RAINRATE"].values * 10 ** (-3)
    T = -273.15 + df["T2D"].values
    ws = (((df["U2D"]) ** 2 + (df["V2D"]) ** 2) ** 0.5).values
    cols = (P, T, df["LWDOWN"].values, df["SWDOWN"].values, df["PSFC"].values, df["Q2D"].values, ws)
    names = ("atmosphere_water__liquid_equivalent_precipitation_rate", "land_surface_air__temperature",
             "land_surface_radiation~incoming~longwave__energy_flux", "land_surface_radiation~incoming~shortwave__energy_flux",
             "land_surface_air__pressure", "atmosphere_air_water~vapor__relative_saturation", "wind_speed_UV")
    rng = np.random.default_rng(seed)
    busy, last = 0.0, 0.0
    with tempfile.TemporaryDirectory() as d:
        for i in range(n_inst):
            cfg = dict(SAMPLE_CONFIG, elev=float(rng.uniform(1200, 4300)), h0_swe=float(rng.uniform(0, 1.5)))
            cfg["h0_snow"] = cfg["h0_swe"] * 20.0
            path = Path(d) / f"c{i}.yaml"
            path.write_text(yaml.dump(cfg))
            model = topoflow_glacier.BmiTopoflowGlacier()
            model.initialize(str(path))
            dest = np.zeros(1)
            t0 = time.perf_counter()
            for t in range(len(P)):
                for name, col in zip(names, cols):
                    model.set_value(name, col[t])
                model.update()
                model.get_value("land_surface_water__runoff_volume_flux", dest)
            busy += time.perf_counter() - t0
            last = float(dest[0])
    return busy, n_inst * len(P), last


def reference_throughput(cores: int, inst_per_core: int = 2, n_steps: int = 288):
    """cell-steps/s of the real reference on `cores` host cores (one process each, slowest worker's busy time)."""
    import multiprocessing as mp

    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_reference_worker, [(inst_per_core, n_steps, 100 + i) for i in range(cores)])
    busy = max(r[0] for r in res)
    return sum(r[1] for r in res) / busy, busy, {"instances": cores * inst_per_core, "steps": n_steps}


def synthetic_host_sample(n_cells: int, n_steps: int, seed: int = 4096):
    """Host-only synthetic cells + forcing with the cfg-4 distributions (used when no GPU is involved)."""
    import numpy as np

    rng = np.random.Generator(np.random.PCG64(seed))
    U = lambda lo, hi: rng.uniform(lo, hi, n_cells)  # noqa: E731
    swe = U(0, 1.5)
    iwe = U(0, 60) * (rng.uniform(size=n_cells) < 0.4)
    statics = {"da": np.full(n_cells, 9e-4), "slope": U(0, 120), "aspect": U(0, 360), "lon": U(-122.1, -121.4),
               "lat": U(46.5, 47.1), "elev": U(1200, 4300), "h0_snow": swe * 20.0, "h0_ice": iwe * (1000.0 / 917.0),
               "h0_swe": swe, "h0_iwe": iwe, "T_rain_snow": np.zeros(n_cells)}
    hours = np.arange(n_steps)[:, None]
    T2D = (275.15 + 9 * np.sin(2 * np.pi * ((274 + hours // 24) % 365 - 105) / 365)
           + 4 * np.sin(2 * np.pi * (hours % 24 - 15) / 24) + rng.normal(0, 2, (n_steps, n_cells))
           - 6.5e-3 * (statics["elev"][None, :] - 2400.0))
    PSFC = 88900 + rng.normal(0, 400, (n_steps, n_cells))
    Tc = T2D - 273.15
    esat = 611.0 * np.exp(17.3 * Tc / (Tc + 237.3))
    q = np.clip(0.8 * (0.622 * esat / (PSFC - 0.378 * esat)) * rng.uniform(0.5, 1, (n_steps, n_cells)), 5e-4, 0.012)
    rain = np.where(rng.uniform(size=(n_steps, n_cells)) < 0.12, rng.exponential(0.5, (n_steps, n_cells)), 0.0)
    uz = 3.0 * np.hypot(rng.normal(size=(n_steps, n_cells)), rng.normal(size=(n_steps, n_cells)))
    forcing = np.stack([rain * 1e-3, T2D - 273.15, PSFC, q, uz], axis=1)
    return statics, np.ascontiguousarray(forcing)


def run_reference_arm(args):
    """The reference's own CPU implementation of the path on all host cores, a bounded sample per step.

    When `baseline/_ref` holds the unmodified reference (scripts/install_reference.py) THAT is what is timed: one BMI
    instance per cell, the reference's per-step driver loop, one process per core (kind "reference").  The vectorised
    NumPy port (oracle/np_ref.py, ~1000x faster per core, proven bit-equal to the reference) is timed beside it and
    reported as `cpu_baseline_port`; it is the headline only if the reference copy is absent.
    """
    rank, _, world = env_rank()
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    n_cells = min(args.cpu_cells or 131072 * cores, 1 << 21)
    n_steps = args.cpu_steps
    statics, forcing = synthetic_host_sample(n_cells, n_steps)
    times = []
    for i in range(args.warmup + args.steps):
        thr, wall, _ = cpu_port_throughput(statics, forcing, "2012100100", cores)
        if i >= args.warmup:
            times.append((thr, wall))
    cs = n_cells * n_steps
    # like the GPU arm (device time, max over ranks): the slowest worker's compute time per step, not the wall
    # clock around fork + pickling of the sample
    busy = sum(cs / thr for thr, _ in times)
    port_value = cs * len(times) / busy
    port = {"value": port_value, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_cells} cells x {n_steps} timesteps per step, oracle/np_ref.py, one process per core; "
                      "timed as the slowest worker's compute time (pool start-up and pickling excluded)"}
    if reference_available():
        inst, steps_ref = args.ref_instances_per_core, 288
        # --warmup untimed runs, then exactly --steps timed ones (--ref-instances-per-core bounds the cost of each)
        runs = [reference_throughput(cores, inst, steps_ref) for _ in range(args.warmup + args.steps)][args.warmup:]
        value = sum(r[0] for r in runs) / len(runs)
        ms = 1e3 * sum(r[1] for r in runs) / len(runs)
        base = {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                "sample": f"{cores * inst} reference instances (one cell each, baseline/_ref: unmodified NGWPC/topoflow-glacier "
                          f"+ stub bmipy/timezonefinder/pyprojroot) x {steps_ref} hourly steps of the sample forcing, the "
                          "reference's own set_value x7 / update() / get_value loop, one process per core"}
        cfg = {"workload": "one reference BMI instance per cell, sample forcing (the reference cannot run a grid)",
               "cells": cores * inst, "timesteps_per_step": steps_ref}
    else:
        value, ms, base = port_value, 1e3 * busy / len(times), port
        cfg = {"workload": "synthetic glacierised raster (cfg-4 distributions), CPU sample", "cells": n_cells,
               "timesteps_per_step": n_steps}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg, "cpu_baseline": base,
        "cpu_baseline_port": port,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------- GPU arm
def knife_edge_report(got: dict, want: dict) -> dict:
    """GPU result against the CPU port on the sample cells, final state after `cpu_steps` steps.

    A cell counts as "within tolerance" when every compared quantity meets the parity bound of tests/helpers.py
    (|gpu - cpu| <= 1e-12 |cpu| + atol).  Cells outside it are classified with the test suite's own detectors instead of
    a blanket relative threshold: `knife_edge` = one side holds an exactly melted-out pack where the other keeps a
    rounding residue (helpers.knife_edge_mask on the final step); `log_law` = the snow surface is within a few ulp-
    amplifications of the wind height (kappa / ln((z - h_snow)/z0) is singular at h_snow = z - z0)."""
    import numpy as np

    sys.path.insert(0, str(ROOT / "tests"))
    from helpers import ATOL, RTOL, knife_edge_mask

    bad = np.zeros(want["RH"].shape, dtype=bool)
    for k in got:
        bad |= np.abs(got[k] - want[k]) > RTOL * np.abs(want[k]) + ATOL[k]
    g2 = {k: got[k][None, :] for k in ("h_swe", "h_iwe")}
    w2 = {k: want[k][None, :] for k in ("h_swe", "h_iwe")}
    knife = knife_edge_mask(g2, w2)[0]
    hs = want["h_swe"] * 20.0
    cond = 1e-16 * np.maximum(hs, 1.0) / np.maximum(np.abs(9.99 - hs) * np.abs(np.log(np.maximum((10.0 - hs) / 0.01, 1.0001))), 1e-300)
    log_law = cond > 1e-13          # relative amplification of one ulp of h_snow in the drag coefficient
    rel = np.zeros(want["RH"].shape)
    for k in got:
        rel = np.maximum(rel, np.abs(got[k] - want[k]) / (np.abs(want[k]) + 1e-12))
    return {"cells": int(bad.size), "within_tolerance": int((~bad).sum()),
            "outside_at_melt_out_knife_edge": int((bad & knife).sum()),
            "outside_at_log_law_singularity": int((bad & ~knife & log_law).sum()),
            "outside_downstream_of_an_earlier_knife_edge": int((bad & ~knife & ~log_law).sum()),
            "median_rel_err": float(np.median(rel)), "tolerance": "1e-12*|ref| + atol (tests/helpers.py)"}


def time_launches(eng, forcing, Tc, zero_agg, reduce_agg, steps, world, dev):
    """`steps` launches of the fused kernel + aggregate reduction; CUDA events around every launch (launching stream)
    and around the whole region.  Returns (mean kernel ms, device ms of the region = max over ranks)."""
    import torch
    import torch.distributed as dist

    evs = []
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a_all, b_all = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a_all.record()
    for _ in range(steps):
        tgt = zero_agg()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.run(forcing, Tc, basin_agg=tgt)
        b.record()
        reduce_agg()
        evs.append((a, b))
    b_all.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t = torch.tensor([a_all.elapsed_time(b_all)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return sum(a.elapsed_time(b) for a, b in evs) / len(evs), float(t.item())


def dump_outputs(out_dir, eng, agg) -> None:
    """Write what the last timed launch handed its caller to ``out_dir/<name>.npy``: the BMI output rows of the state
    (``BMI_OUTPUTS``, engine dtype, ``[cells]``) and the launch's per-basin aggregates (float64 ``[timesteps, n_basin]``,
    one file per ``sharding.AGG_NAMES`` entry, prefixed ``basin_``).

    A row longer than ``DUMP_CELLS`` is cut to a fixed sample of that many cells (seed 0, ascending cell order), the
    aggregates to the last timesteps that fit in ``DUMP_AGG_BYTES``: at most 48 MB in all, the same cells and
    timesteps on every run with the same arguments.  With several ranks this is rank 0's shard of cells."""
    import numpy as np
    import torch

    from topoflow_glacier_b200.sharding import AGG_NAMES

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    torch.cuda.synchronize()
    cells = None
    if eng.N > DUMP_CELLS:
        pick = np.sort(np.random.default_rng(0).choice(eng.N, DUMP_CELLS, replace=False))
        cells = torch.as_tensor(pick, device=eng.device)
    for name in BMI_OUTPUTS:
        row = eng.row(name)
        np.save(out / f"{name}.npy", (row if cells is None else row[cells]).cpu().numpy())
    n_t = max(1, min(agg.buffer.shape[0], DUMP_AGG_BYTES // (agg.buffer[0].numel() * 8)))
    tail = agg.buffer[-n_t:].cpu().numpy()
    for j, name in enumerate(AGG_NAMES):
        np.save(out / f"basin_{name}.npy", np.ascontiguousarray(tail[..., j]))


def run_gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.config import default_constants
    from topoflow_glacier_b200.engine import MeltEngine
    from topoflow_glacier_b200.forcing import DEFAULT_PACKING, ForcingStreamer, bind_host_to_gpu, pinned_block
    from topoflow_glacier_b200.sharding import BasinAggregates, ShardedMeltEngine
    from topoflow_glacier_b200.synthetic import synthetic_cells

    rank, local_rank, world = env_rank()
    # ---- CPU baselines first (rank 0, N == 1), before CUDA is initialised so that fork() is safe ------------
    cpu = cpu_ref = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        ns = min(args.cpu_cells or 131072 * cores, 1 << 21)
        statics_h, forcing_h = synthetic_host_sample(ns, args.cpu_steps)
        thr, wall_cpu, last = cpu_port_throughput(statics_h, forcing_h, "2012100100", cores)
        cpu = {"value": thr, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{ns} cells (cfg-4 distributions) x {args.cpu_steps} timesteps, oracle/np_ref.py, one process "
                         f"per core ({wall_cpu:.1f} s wall)", "_sample": (statics_h, forcing_h, last)}
        if reference_available():  # the unmodified reference beside it (one BMI instance per cell, baseline/_ref)
            rthr, rbusy, rinfo = reference_throughput(cores, args.ref_instances_per_core, 288)
            cpu_ref = {"value": rthr, "unit": UNIT, "cores": cores, "kind": "reference",
                       "sample": f"{rinfo['instances']} reference instances x {rinfo['steps']} steps of the sample forcing, "
                                 f"set_value x7 / update() / get_value per step, one process per core ({rbusy:.1f} s)"}
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the melt path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    numa = bind_host_to_gpu(local_rank)   # pinned staging buffers are first-touched next to this rank's GPU
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    consts = default_constants()
    peak, peak_src = measured_peak()

    def clocked(fn):
        smp = ClockSampler(local_rank)
        smp.start()
        out = fn()
        return out, smp.stop()

    def roofline_of(mode, cell_steps, kern_ms, traffic=None):
        es = 4 if mode == "f32" else 8
        achieved = es * _lib.N_FORCING * cell_steps / (kern_ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "kernel": "tfg::run_kernel", "kernel_ms": kern_ms,
                "algorithmic_bytes_per_cell_step": es * _lib.N_FORCING,
                "note": "FP64-pipe / issue bound, not HBM bound: see compute_roofline, profiles/ and DESIGN.md"}

    # =================================================================================================================
    # headline: one synthetic 4096 x 4096 raster per GPU (weak scaling), or the regional grid when --workload regional
    # =================================================================================================================
    Tc, mode = args.chunk, args.mode
    regional = args.workload == "regional"
    es = 4 if mode == "f32" else 8
    horizon = (args.warmup + args.steps + 4) * Tc + (2 * args.e2e_steps + args.warmup + 24) * max(args.e2e_chunk, Tc) + 64

    def make_engine(mode, n_total_or_cells, sharded, seed_base, chunk, horizon):
        """(engine, elevation, basin ids, zero_agg, reduce_agg, total cells, first cell): a raster per rank, or this
        rank's shard of the regional grid through the product API (sharding.ShardedMeltEngine)."""
        if sharded:
            total = n_total_or_cells
            per_basin = -(-total // N_BASIN)
            keep = {}

            def factory(lo, hi):
                tabs = synthetic_cells(hi - lo, seed=seed_base + rank, device=dev)
                keep["elev"] = tabs.pop("raw")["elev"]
                return tabs

            sh = ShardedMeltEngine(factory, consts, "2012100100", n_total=total, n_basin=N_BASIN, zones=[-8.0], mode=mode,
                                   basin_id=lambda lo, hi: (torch.arange(lo, hi, device=dev, dtype=torch.int64) // per_basin).to(torch.int32),
                                   exact=(args.agg == "exact"), device=local_rank, horizon_steps=horizon, dt_hours=1)
            agg = sh.aggregates(chunk)
            return sh.engine, keep["elev"], sh.engine.basin_id, agg.zero, agg.reduce, total, sh.bounds[0], agg
        n_cells = n_total_or_cells
        total, first = n_cells * world, rank * n_cells
        tabs = synthetic_cells(n_cells, seed=seed_base + rank, device=dev)
        elev = tabs.pop("raw")["elev"]
        per_basin = -(-total // N_BASIN)
        basin_id = ((torch.arange(n_cells, device=dev, dtype=torch.int64) + first) // per_basin).to(torch.int32)
        eng = MeltEngine(None, consts, "2012100100", dt_hours=1, zones=[-8.0], basin_id=basin_id, n_basin=N_BASIN, mode=mode,
                         device=local_rank, horizon_steps=horizon, device_statics=tabs)
        agg = BasinAggregates(chunk, N_BASIN, device=dev, exponents=eng.agg_exponents() if args.agg == "exact" else None)
        return eng, elev, basin_id, agg.zero, agg.reduce, total, first, agg

    eng, elev, basin_id, zero_agg, reduce_agg, total_cells, first_cell, agg = make_engine(
        mode, args.cells, regional, 100 if regional else 4096, Tc, horizon)
    n_cells = eng.N
    elev = elev.to(eng.dtype)
    forcing = torch.empty(Tc, 5, n_cells, dtype=eng.dtype, device=dev)
    eng.synth_forcing(forcing, 0, Tc, elev, seed=20121001 + rank)
    agg_exps = eng.agg_exponents() if args.agg == "exact" else None
    fp64_peak = eng.measure_fp64_peak()  # DFMA microbenchmark, before the timed region
    torch.cuda.synchronize()

    # ---- GPU result on the CPU sample (same host-generated cells and forcing): the correctness check -----
    if cpu is not None:
        statics_h, forcing_h, last = cpu.pop("_sample")
        nt = forcing_h.shape[0]
        chk = MeltEngine(statics_h, consts, "2012100100", zones=[-8.0], mode=mode, device=local_rank, horizon_steps=nt + 1)
        chk.run(torch.as_tensor(forcing_h).to(dev, chk.dtype).contiguous(), nt)
        torch.cuda.synchronize()
        g = {k: chk.row(k).to(torch.float64).cpu().numpy() for k in ("M_total", "h_swe", "h_iwe", "RH")}
        if mode != "f32":
            cpu["gpu_vs_cpu_on_sample"] = knife_edge_report(g, last)
        chk.close()
        del chk

    for _ in range(args.warmup):
        eng.run(forcing, Tc, basin_agg=zero_agg())
        reduce_agg()
    t0 = time.perf_counter()
    (kern_ms, dev_ms), clocks = clocked(lambda: time_launches(eng, forcing, Tc, zero_agg, reduce_agg, args.steps, world, dev))
    wall = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:   # before the legs below advance the same engine further
        dump_outputs(args.dump_outputs, eng, agg)
    cell_steps = n_cells * Tc  # this rank's launch
    value = total_cells * Tc * args.steps / (dev_ms * 1e-3)

    # ---- same launch on spatially coherent weather (precipitation shared by 4096 consecutive cells) --------------
    coherent = None
    if not args.no_coherent:
        eng.synth_forcing(forcing, 0, Tc, elev, seed=20121001 + rank, storm_cells=4096)
        eng.run(forcing, Tc, basin_agg=zero_agg())
        ms2, _ = time_launches(eng, forcing, Tc, zero_agg, lambda: None, max(2, args.steps // 2), 1, dev)
        coherent = {"cell_steps_per_s_per_gpu": cell_steps / (ms2 * 1e-3), "kernel_ms": ms2,
                    "forcing": "as above, precipitation occurrence shared by 4096 consecutive cells"}
        eng.synth_forcing(forcing, 0, Tc, elev, seed=20121001 + rank)

    # =================================================================================================================
    # end to end through the public API with host buffers
    # =================================================================================================================
    Te = args.e2e_chunk
    if regional:  # keep only the block the e2e leg streams; the kernel-leg chunk goes back to the allocator
        forcing = forcing[:Te].clone()
        torch.cuda.empty_cache()
    raw_name = args.e2e_raw
    raw_dtype = {"int16": torch.int16, "float32": torch.float32, "float64": torch.float64}[raw_name]
    blk = forcing[:Te].to(torch.float64)
    raw_f = torch.stack([blk[:, 0] * 1e3, blk[:, 1] + 273.15, blk[:, 2], blk[:, 3], blk[:, 4] * 0.6, blk[:, 4] * 0.8], dim=1)
    if raw_name == "int16":  # NetCDF-style packed columns (forcing.pack_forcing, on the device here: 16.7 M cells)
        sc = torch.as_tensor(DEFAULT_PACKING[0], device=dev).view(1, 6, 1)
        of = torch.as_tensor(DEFAULT_PACKING[1], device=dev).view(1, 6, 1)
        raw_dev = torch.clamp(torch.round((raw_f - of) / sc), -32768, 32767).to(torch.int16)
    else:
        raw_dev = raw_f.to(raw_dtype)
    # the host only fills this block: write-combined pages (device reads over PCIe need no cache snoop)
    raw_host = (pinned_block((Te, 6, n_cells), raw_dtype, write_combined=True) if args.e2e_wc
                else torch.empty(Te, 6, n_cells, dtype=raw_dtype).pin_memory())
    raw_host.copy_(raw_dev)
    del raw_dev, raw_f, blk
    out_names = BMI_OUTPUTS
    out_dtype = torch.float32 if args.e2e_out == "float32" else eng.dtype
    out_host = [torch.empty(len(out_names), n_cells, dtype=out_dtype).pin_memory() for _ in range(2)]
    drain = torch.cuda.Stream(device=dev)
    drained = [torch.cuda.Event() for _ in range(2)]

    def e2e_loop(streamer, host_block, aggs, agg_hosts, k_steps):
        """k_steps host blocks streamed back to back: H2D of block i+1, the kernel of block i and the D2H of the
        results of block i-1 overlap (PCIe is full duplex); every block's outputs reach pinned host memory."""
        cur = torch.cuda.current_stream()
        for i, chunk in enumerate(streamer.chunks([host_block] * k_steps)):
            j = i % 2
            cur.wait_event(drained[j])  # result buffers of two blocks ago have left the device
            eng.run(chunk, chunk.shape[0], basin_agg=aggs[j].zero())
            aggs[j].reduce()
            snap = eng.snapshot_outputs(out_names, out_dtype)
            done = torch.cuda.Event()
            done.record(cur)
            with torch.cuda.stream(drain):
                drain.wait_event(done)
                out_host[j].copy_(snap, non_blocking=True)
                agg_hosts[j].copy_(aggs[j].buffer, non_blocking=True)
                snap.record_stream(drain)
                drained[j].record(drain)
        drain.synchronize()
        cur.synchronize()

    def timed_e2e(fn, k_steps):
        fn(2)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        fn(k_steps)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    streamer = ForcingStreamer(eng, Te, raw_dtype=raw_name)
    agg_e = [BasinAggregates(Te, N_BASIN, device=dev, exponents=agg_exps) for _ in range(2)]
    agg_host = [torch.empty(Te, N_BASIN, 3, dtype=torch.float64).pin_memory() for _ in range(2)]
    e2e_s = timed_e2e(lambda k: e2e_loop(streamer, raw_host, agg_e, agg_host, k), args.e2e_steps)
    e2e_value = total_cells * Te * args.e2e_steps / e2e_s
    h2d = raw_host.numel() * raw_host.element_size()
    d2h = out_host[0].numel() * out_host[0].element_size() + agg_host[0].numel() * 8

    # ---- what binds the end-to-end leg: each of its three stages alone, per block ------------------------------------
    def stage_ms(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        t = torch.tensor([(time.perf_counter() - t0) / reps * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    d_raw_probe = streamer.d_raw[0]
    snap_probe = eng.snapshot_outputs(out_names, out_dtype)
    ms_h2d = stage_ms(lambda: d_raw_probe.copy_(raw_host, non_blocking=True))            # all ranks at once
    ms_d2h = stage_ms(lambda: out_host[0].copy_(snap_probe, non_blocking=True))
    ms_kernel = kern_ms * Te / Tc
    solo_h2d = None
    if world > 1:  # the same copy with the other ranks idle: PCIe alone, without contention for the host's memory
        for r in range(world):
            if r == rank:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(3):
                    d_raw_probe.copy_(raw_host, non_blocking=True)
                torch.cuda.synchronize()
                solo_h2d = (time.perf_counter() - t0) / 3 * 1e3
            dist.barrier()
    stages = {"h2d_ms": ms_h2d, "kernel_ms": ms_kernel, "d2h_ms": ms_d2h}
    slowest = max(stages, key=stages.get)
    bound = {"h2d_ms": "pcie", "kernel_ms": "kernel", "d2h_ms": "d2h"}[slowest]
    if slowest == "h2d_ms" and solo_h2d is not None and ms_h2d > 1.25 * solo_h2d:
        bound = "host_dram"   # all ranks copying at once are slower than one alone: the host memory system binds, not PCIe
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "timesteps_per_step": Te, "steps": args.e2e_steps,
           "raw_dtype": raw_name, "host_block": "write-combined" if args.e2e_wc else "pinned", "out_dtype": args.e2e_out, "bound": bound,
           "stage_ms_per_block": {**stages, "h2d_alone_ms": solo_h2d, "h2d_GBps_per_gpu": h2d / ms_h2d / 1e6,
                                  "d2h_GBps_per_gpu": d2h / ms_d2h / 1e6},
           "host_numa_binding": numa,
           "path": f"pinned host {raw_name} met columns -> ForcingStreamer (tfg_ingest_async + tfg_convert_forcing"
                   f"{'_packed' if raw_name == 'int16' else ''}) -> tfg_run -> D2H of the 8 BMI outputs ({args.e2e_out}) + basin aggregates"}

    # ---- the same end-to-end path with CATCHMENT forcing (tfg_bind_forcing_map) --------------------------------
    # One forcing series per basin (4096 columns) instead of one per 30 m cell, as the reference's one-CSV-per-
    # catchment drivers supply it: the host block shrinks to ~0.003 B per cell-step and PCIe no longer binds.
    shared = None
    if not regional and not args.no_shared:
        del raw_host, streamer, d_raw_probe
        Ts = Tc
        eng.set_forcing_map(basin_id % N_BASIN, N_BASIN)
        raw_cols = torch.empty(Ts, 6, N_BASIN, dtype=torch.float32).pin_memory()
        blk = forcing[:Ts, :, :N_BASIN].to(torch.float64)
        raw_cols.copy_(torch.stack([blk[:, 0] * 1e3, blk[:, 1] + 273.15, blk[:, 2], blk[:, 3], blk[:, 4] * 0.6,
                                    blk[:, 4] * 0.8], dim=1).to(torch.float32))
        del blk   # a view: it would keep the whole forcing chunk alive
        streamer2 = ForcingStreamer(eng, Ts, raw_dtype="float32")
        agg_s = [BasinAggregates(Ts, N_BASIN, device=dev, exponents=agg_exps) for _ in range(2)]
        agg_sh = [torch.empty(Ts, N_BASIN, 3, dtype=torch.float64).pin_memory() for _ in range(2)]
        n_sh = max(8, args.e2e_steps)   # the last block's D2H is not overlapped: amortise it over a few blocks
        t_sh = timed_e2e(lambda k: e2e_loop(streamer2, raw_cols, agg_s, agg_sh, k), n_sh)
        shared = {"value": total_cells * Ts * n_sh / t_sh, "unit": UNIT, "steps": n_sh,
                  "h2d_bytes_per_step": raw_cols.numel() * raw_cols.element_size(),
                  "d2h_bytes_per_step": out_host[0].numel() * out_host[0].element_size() + agg_sh[0].numel() * 8,
                  "timesteps_per_step": Ts, "forcing_columns": N_BASIN, "out_dtype": args.e2e_out,
                  "path": "as e2e, one float32 forcing series per basin (tfg_bind_forcing_map) instead of one per cell"}
        # the launch alone on device-resident columns (column-term pass + melt kernel), CUDA events around each launch
        fcol = forcing[:Ts, :, :N_BASIN].contiguous()
        for _ in range(2):
            eng.run(fcol, Ts, basin_agg=zero_agg())
        k_sh, _ = time_launches(eng, fcol, Ts, zero_agg, reduce_agg, 3, world, dev)
        shared["launch_ms"] = k_sh
        shared["launch_cell_steps_per_s_per_gpu"] = n_cells * Ts / (k_sh * 1e-3)
        shared["column_terms"] = bool(eng.column_term_launches > 0)   # TFG_OPT_COLUMN_TERMS (env TFG_COLUMN_TERMS=0 switches it off)
        del fcol
        eng.set_forcing_map(None)
        del streamer2, agg_s

    # =================================================================================================================
    # sub-records: the other arithmetic modes (N == 1) and the strong-scaling regional grid (every N)
    # =================================================================================================================
    def free_headline():
        nonlocal eng, forcing, agg, agg_e, out_host, elev, basin_id, zero_agg, reduce_agg, snap_probe
        eng.close()
        eng = forcing = agg = agg_e = out_host = elev = basin_id = zero_agg = reduce_agg = snap_probe = None
        import gc

        gc.collect()
        torch.cuda.empty_cache()

    modes = {}
    strong = None
    headline_cfg = (mode, n_cells, Tc)
    if not regional and (not args.no_modes or not args.no_strong):
        free_headline()
    if not regional and world == 1 and not args.no_modes:
        for m in ("f64", "f32"):
            if m == mode:
                continue
            e2, el2, _, z2, r2, tot2, _, a2 = make_engine(m, args.cells, False, 4096, Tc, (args.warmup + 30) * Tc + 64)
            f2 = torch.empty(Tc, 5, e2.N, dtype=e2.dtype, device=dev)
            e2.synth_forcing(f2, 0, Tc, el2.to(e2.dtype), seed=20121001 + rank)
            nrep = 2 if m == "f64" else max(3, args.steps // 2, 20)   # f32: >= 0.7 s of timed region for the clock sampler
            for _ in range(2):
                e2.run(f2, Tc, basin_agg=z2())
            (kms, dms), clk = clocked(lambda: time_launches(e2, f2, Tc, z2, r2, nrep, 1, dev))
            modes[m] = {"value": tot2 * Tc * nrep / (dms * 1e-3), "unit": UNIT, "dtype": "f32" if m == "f32" else "f64",
                        "arithmetic_mode": m, "steps": nrep, "ms_per_step": dms / nrep, "clocks": clk,
                        "roofline": roofline_of(m, e2.N * Tc, kms)}
            e2.close()
            del e2, f2, a2, el2
            torch.cuda.empty_cache()
    if not regional and not args.no_strong:
        # BASELINE configs[4]: ONE 100 M-cell grid sharded over the GPUs (strong scaling) through ShardedMeltEngine;
        # timesteps per launch grow with the GPU count (the shard shrinks): 16 on one GPU ... 128 on eight
        Tr = min(128, 16 * world)
        e3, el3, _, z3, r3, tot3, _, a3 = make_engine(mode, REGIONAL_CELLS, True, 100, Tr, (args.warmup + args.steps + 64) * Tr + 64)
        f3 = torch.empty(Tr, 5, e3.N, dtype=e3.dtype, device=dev)
        e3.synth_forcing(f3, 0, Tr, el3.to(e3.dtype), seed=20121001 + rank)
        for _ in range(3):
            e3.run(f3, Tr, basin_agg=z3())
            r3()
        k_est, _ = time_launches(e3, f3, Tr, z3, r3, 1, world, dev)
        nrep = max(3, args.steps // 2, int(-(-800.0 // k_est)))   # >= 0.8 s of timed region: the clock sampler ticks every 100 ms
        (kms, dms), clk = clocked(lambda: time_launches(e3, f3, Tr, z3, r3, nrep, world, dev))
        strong = {"value": tot3 * Tr * nrep / (dms * 1e-3), "unit": UNIT, "scaling": "strong", "n_gpus": world,
                  "cells_total": tot3, "cells_per_gpu": e3.N, "timesteps_per_step": Tr, "steps": nrep,
                  "ms_per_step": dms / nrep, "clocks": clk, "roofline": roofline_of(mode, e3.N * Tr, kms),
                  "workload": "synthetic 100M-cell regional grid sharded over the GPUs (BASELINE configs[4]) through "
                              "sharding.ShardedMeltEngine, basin aggregates all-reduced over NCCL"}
        e3.close()
        del e3, f3, a3

    if rank == 0:
        mode, n_cells, Tc = headline_cfg
        traffic = None
        tp = ROOT / "profiles" / "traffic.json"
        if tp.exists():
            try:
                traffic = json.loads(tp.read_text()).get(f"{mode}:{n_cells}x{Tc}")
            except Exception:  # noqa: BLE001
                traffic = None
        # the unit that actually binds (DESIGN.md section 4): FP64 pipe at 1 warp-instruction / 2 cycles / scheduler
        compute = None
        mp = ROOT / "profiles" / "kernel_mix.json"
        if mp.exists() and mode != "f32":
            try:
                mix = json.loads(mp.read_text())[mode]
                # ceiling = measured DFMA thread-ops/s / FP64 instructions per cell-step (a warp-instruction is 32 of them)
                ceiling = fp64_peak / mix["fp64_warp_inst_per_warp_step"]
                # issue ceiling: one warp-instruction per cycle and scheduler (4 per SM)
                sms = torch.cuda.get_device_properties(dev).multi_processor_count
                mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
                issue_ceiling = sms * 4 * mhz * 1e6 * 32 / mix["warp_inst_per_warp_step"]
                compute = {"bound": "fp64_pipe", "fp64_warp_inst_per_warp_step": mix["fp64_warp_inst_per_warp_step"],
                           "warp_inst_per_warp_step": mix["warp_inst_per_warp_step"],
                           "issue_ceiling_cell_steps_per_s": issue_ceiling,
                           "frac_of_issue_ceiling": (cell_steps / (kern_ms * 1e-3)) / issue_ceiling,
                           "fp64_peak_tflops_measured": 2 * fp64_peak / 1e12,
                           "ceiling_cell_steps_per_s": ceiling, "frac_of_ceiling": (cell_steps / (kern_ms * 1e-3)) / ceiling,
                           "ncu_fp64_pipe_active_pct": mix["fp64_pipe_active_pct"],
                           "ncu_issue_active_pct": mix["issue_active_pct"], "source": mix["source"]}
            except Exception:  # noqa: BLE001
                compute = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong" if regional else "weak",
            "vs_baseline": None,
            "dtype": "f32" if mode == "f32" else "f64", "data": "synthetic",
            "config": {"workload": ("synthetic 100M-cell regional grid sharded over the GPUs (BASELINE configs[4]), hourly forcing"
                                    if regional else
                                    "synthetic 4096x4096 glacierised raster per GPU (BASELINE configs[3]), hourly forcing"),
                       "cells_total": total_cells, "cells_per_gpu": n_cells, "timesteps_per_step": Tc, "arithmetic_mode": mode,
                       "basin_aggregates": N_BASIN, "aggregate_sums": args.agg, "forcing": "device-resident chunk, Philox synthetic, reused each step",
                       "l2": f"inputs {es * 5 * cell_steps / 1e9:.1f} GB per launch >> 126 MB L2 (no flush needed)",
                       "parallelism": f"cells sharded x{world}, all_reduce of basin aggregates"},
            "roofline": roofline_of(mode, cell_steps, kern_ms, traffic),
            "compute_roofline": compute,
            "e2e": e2e,
            "e2e_catchment_forcing": shared,
            "gpu_launches": args.steps, "clocks": clocks, "wall_s": wall, "coherent_weather": coherent,
            "modes": modes or None, "strong_regional": strong,
        }
        if cpu is not None:   # the real reference when its copy travelled (kind "reference"), the NumPy port beside it
            line["cpu_baseline"] = cpu_ref if cpu_ref is not None else cpu
            line["cpu_baseline_port"] = cpu
        print(json.dumps(line))
    if eng is not None:
        eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="f64_fast", choices=["f64", "f64_fast", "f32"])
    ap.add_argument("--workload", default="raster", choices=["raster", "regional"],
                    help="raster: 4096x4096 cells PER GPU (BASELINE configs[3], weak scaling); regional: 100 M cells in "
                         "total, sharded over the GPUs (configs[4], strong scaling, 16 timesteps per launch)")
    ap.add_argument("--cells", type=int, default=0, help="cells per GPU (raster) / in total (regional)")
    ap.add_argument("--chunk", type=int, default=0, help="timesteps per launch (default 128 raster, 16 regional)")
    ap.add_argument("--e2e-chunk", type=int, default=16)
    ap.add_argument("--e2e-steps", type=int, default=8,
                    help="host blocks streamed in the end-to-end leg (the pipeline's fill and drain -- first H2D, last kernel + D2H -- are inside the timed region and amortise over them)")
    ap.add_argument("--e2e-wc", type=int, default=0, help="1: the pinned forcing block is write-combined (forcing.pinned_block)")
    ap.add_argument("--e2e-raw", default="int16", choices=["int16", "float32", "float64"],
                    help="host met columns: int16 = NetCDF-style packed (scale_factor / add_offset), 12 B per cell-step")
    ap.add_argument("--e2e-out", default="float32", choices=["float32", "native"],
                    help="element type of the BMI outputs copied back to the host every block")
    ap.add_argument("--no-modes", action="store_true", help="skip the f64 / f32 sub-records (N = 1)")
    ap.add_argument("--no-strong", action="store_true", help="skip the 100 M-cell strong-scaling sub-record")
    ap.add_argument("--cpu-cells", type=int, default=0)
    ap.add_argument("--cpu-steps", type=int, default=24)
    ap.add_argument("--ref-instances-per-core", type=int, default=2,
                    help="reference BMI instances each host core runs through 288 steps (baseline/_ref)")
    ap.add_argument("--agg", default="float", choices=["float", "exact"],
                    help="basin sums: float64 atomics, or order-independent fixed-point accumulators (TFG_OPT_EXACT_AGG)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-coherent", action="store_true")
    ap.add_argument("--no-shared", action="store_true", help="skip the catchment-forcing end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed launches, write the outputs of the last one to DIR/<name>.npy (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm; --impl reference has none")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    regional = args.workload == "regional"
    args.cells = args.cells or (REGIONAL_CELLS if regional else GRID_CELLS)
    args.chunk = args.chunk or (16 if regional else 128)
    if regional:  # 100 M cells fill the HBM of one GPU: no second forcing realisation, one-timestep e2e blocks
        args.no_coherent, args.no_cpu, args.e2e_chunk = True, True, 1
        args.no_modes = args.no_strong = True
    return run_reference_arm(args) if args.impl == "reference" else run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
