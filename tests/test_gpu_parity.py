"""GPU: the CUDA path (through the C ABI, via MeltEngine.run -> tfg_run) against the oracle.

Every case of tests/golden is run on the device with all intermediates recorded and compared with
(a) the oracle run here on the same inputs and (b) the committed reference vectors.
float64 modes: |gpu - ref| <= 1e-12*|ref| + atol(quantity)  (helpers.ATOL).
"""

import json
import os
from pathlib import Path

import numpy as np
import pytest

from helpers import ATOL, CASES, RTOL, err_report, f32_bound_report, load_case, make_engine, make_oracle

pytestmark = pytest.mark.gpu
REPORT = Path(os.environ.get("GRAFT_REPO_ROOT", Path(__file__).resolve().parent.parent)) / "gpurun_out"

REC = ["h_snow", "h_swe", "SM", "h_ice", "h_iwe", "IM", "M_total", "RH", "p0", "e_sat_air", "e_air", "T_dew", "T_surf",
       "e_sat_surf", "Ri", "Dn", "Dh", "Qh", "W_p", "e_surf", "Qe", "TSN_offset", "albedo", "n", "Qn_SW", "em_air",
       "Qn_LW", "Q_sum", "Eccs", "Ecci", "snow3day", "P_rain", "P_snow"]
VOLS = ["vol_P", "vol_PR", "vol_PS", "vol_SM", "vol_IM", "P_max"]


def _oracle_series(case):
    ora = make_oracle(case, strict_pow=case["N"] <= 4)
    T = case["forcing"].shape[0]
    out = {k: np.empty((T, case["N"])) for k in REC}
    for t in range(T):
        d = ora.step(*case["forcing"][t])
        for k in REC:
            out[k][t] = d[k]
    out.update({k: getattr(ora, k) for k in VOLS})
    return out


_ORACLE = {}


def oracle_series(name):
    if name not in _ORACLE:
        _ORACLE[name] = (load_case(name), None)
        _ORACLE[name] = (_ORACLE[name][0], _oracle_series(_ORACLE[name][0]))
    return _ORACLE[name]


def _dump(tag, rep):
    REPORT.mkdir(exist_ok=True)
    p = REPORT / "parity_report.json"
    cur = json.loads(p.read_text()) if p.exists() else {}
    cur[tag] = rep
    p.write_text(json.dumps(cur, indent=1, sort_keys=True))


@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
@pytest.mark.parametrize("name", CASES)
def test_fused_run_matches_oracle(name, mode, cuda_device):
    import torch

    case, want = oracle_series(name)
    eng = make_engine(case, mode=mode)
    forcing = torch.as_tensor(case["forcing"]).to(cuda_device)
    got = eng.run(forcing, record=REC)
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy() for k, v in got.items()}
    got.update({k: eng.row(k).cpu().numpy() for k in VOLS})
    rep, bad = {}, []
    for k in REC + VOLS:
        ok, ratio, dabs, drel = err_report(got[k], want[k], ATOL[k])
        rep[k] = {"ok": ok, "err_over_tol": ratio, "max_abs": dabs, "max_rel": drel}
        if not ok:
            t = int(np.argmax(np.abs(got[k] - want[k]).reshape(len(got[k]), -1).max(axis=1))) if got[k].ndim == 2 else -1
            bad.append((k, ratio, dabs, drel, t))
    # and against the committed reference vectors (made on the build machine)
    rows = case["rows"] if case["rows"] is not None else slice(None)
    for k, ref in case["ref"].items():
        g = got[k][rows] if k in REC else got[k]
        r = ref if k in REC else ref[-1]
        ok, ratio, dabs, drel = err_report(g, r, ATOL[k])
        rep["golden:" + k] = {"ok": ok, "err_over_tol": ratio, "max_abs": dabs, "max_rel": drel}
        if not ok:
            bad.append(("golden:" + k, ratio, dabs, drel, -1))
    _dump(f"{name}/{mode}", rep)
    eng.close()
    assert not bad, bad


@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_single_steps_equal_fused_run(mode, cuda_device):
    """n_steps=1 launches (exact window re-sum, state through HBM every step) == one fused launch, bit for bit."""
    import torch

    case = load_case("rand64")
    T = case["forcing"].shape[0]
    a, b = make_engine(case, mode=mode), make_engine(case, mode=mode)
    forcing = torch.as_tensor(case["forcing"]).to(cuda_device, a.dtype)
    a.run(forcing)
    for t in range(T):
        b.run(forcing[t:t + 1].contiguous(), 1)
    # and a split into uneven chunks (window seeded from HBM at each launch)
    c = make_engine(case, mode=mode)
    done = 0
    for k in (5, 1, 17, T - 23):
        c.run(forcing[done:done + k].contiguous(), k)
        done += k
    torch.cuda.synchronize()
    assert torch.equal(a.state, b.state) and torch.equal(a.ring, b.ring)
    assert torch.equal(a.state, c.state) and torch.equal(a.ring, c.ring)
    for e in (a, b, c):
        e.close()


@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_kernel_instantiations_agree_bit_for_bit(mode, cuda_device):
    """Recording, basin aggregates and the diagnostic integrals select different template instantiations of the
    kernel.  None of them may change the state: the strict mode uses single-rounding intrinsics throughout, the fast
    float64 unit is compiled with -fmad=false and spells out every fused multiply-add (tfg_num.cuh fmadd)."""
    import torch

    case = load_case("rand64")
    f = torch.as_tensor(case["forcing"]).to(cuda_device)
    T, N = f.shape[0], case["N"]
    basin = (np.arange(N) // 8).astype(np.int32)
    plain = make_engine(case, mode=mode)
    plain.run(f)
    rec = make_engine(case, mode=mode)
    rec.run(f, record=REC)
    agg = make_engine(case, mode=mode, basin_id=basin, n_basin=int(basin.max()) + 1)
    agg.run(f, basin_agg=torch.zeros(T, int(basin.max()) + 1, 3, dtype=torch.float64, device=cuda_device))
    novol = make_engine(case, mode=mode, diag_integrals=False)
    novol.run(f)
    torch.cuda.synchronize()
    for other in (rec, agg):
        assert torch.equal(plain.state, other.state) and torch.equal(plain.ring, other.ring)
    assert torch.equal(plain.state[:12], novol.state[:12]) and torch.equal(plain.ring, novol.ring)
    for e in (plain, rec, agg, novol):
        e.close()


@pytest.mark.parametrize("name", CASES)
def test_f32_mode_tolerance(name, cuda_device):
    """fp32 mode has its own, looser, stated tolerance (DESIGN.md "fp32 mode"), checked on every golden case: both
    formulations of SATTERLUND (evaluated in float32, there is no strict fallback), dt = 2 / 3 / 24 h (36, 24, 3 window
    slots), polar day and night, a year outside the perihelion table, the snow-to-ice handover and a water year.

    The water-equivalent balances run in float64 inside the float32 kernel (tfg_bind_mass_residual), so depths do not
    drift with float32 accumulation: their error is the flux error (2e-3) times the melt so far.  The bound is
    helpers.f32_bound_report: every cell-step of cells without a shifted melt-out, fluxes and rates outside +-3 steps of
    a shifted melt-out and depths within 1 % at the end for the others, whose number is bounded by the melt-out events."""
    import torch

    case, want = oracle_series(name)
    eng = make_engine(case, mode="f32")
    forcing = torch.as_tensor(case["forcing"]).to(cuda_device, torch.float32)
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in eng.run(forcing, record=REC).items()}
    eng.close()
    rep, bad = f32_bound_report(got, want, case["statics"]["h0_snow"], case.get("consts", {}).get("z0_air", 0.01))
    _dump(f"{name}/f32", rep)
    assert not bad, (bad, rep)


@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_large_random_sample_with_knife_edges(mode, cuda_device):
    """16 384 random cells x 36 steps (bench distributions): everything within tolerance except cells that
    crossed a melt-out knife edge, which must be rare and are reported."""
    import torch

    import bench

    N, T = 16384, 36
    statics, forcing = bench.synthetic_host_sample(N, T, seed=11)
    statics["h0_swe"][::7] *= 1e-3  # plenty of thin snowpacks that melt out inside the window
    statics["h0_snow"][::7] *= 1e-3
    case = {"statics": statics, "N": N, "forcing": forcing, "start_time": "2013040100"}
    from oracle.np_ref import CellStatics, Constants, OracleModel

    ora = OracleModel(CellStatics(**statics, tz=[-8.0]), Constants(), case["start_time"], strict_pow=False)
    keys = ["h_swe", "h_iwe", "h_snow", "h_ice", "SM", "IM", "M_total", "RH", "Q_sum", "Qn_SW", "Qn_LW", "Qh", "Qe",
            "albedo", "Eccs", "Ecci", "T_surf"]
    want = {k: np.empty((T, N)) for k in keys}
    for t in range(T):
        d = ora.step(*forcing[t])
        for k in keys:
            want[k][t] = d[k]
    from topoflow_glacier_b200.engine import MeltEngine
    from helpers import default_constants, knife_edge_mask

    eng = MeltEngine(statics, default_constants(), case["start_time"], zones=[-8.0], mode=mode, horizon_steps=T + 1)
    got = {k: v.cpu().numpy() for k, v in eng.run(torch.as_tensor(forcing).to(cuda_device), record=keys).items()}
    eng.close()
    mask = knife_edge_mask(got, want)
    # The log-law drag coefficient kappa/ln((z - h_snow)/z0) (reference :670) is singular at h_snow = z - z0 = 9.99 m.
    # Condition number of Dn with respect to h_snow: |d ln Dn / d ln h| = 2 h / ((z - h) |ln((z - h)/z0)|) (0 once the
    # argument is clamped at 0.01).  h_snow carries a few ulp (~5e-16 relative) of legitimate difference between two
    # libms, so a 1e-12 bound on the fluxes is only meaningful where cond * 5e-16 < 1e-12 / 4, i.e. cond < 500: such a
    # cell is masked from the step it enters that zone (its state is contaminated afterwards), and counted.
    hs = np.vstack([statics["h0_snow"][None, :], want["h_snow"][:-1]])      # depth the step STARTS from
    arg = (10.0 - hs) / 0.01
    with np.errstate(divide="ignore", invalid="ignore"):
        cond = np.where(arg > 0.01, 2.0 * hs / (np.abs(10.0 - hs) * np.abs(np.log(np.maximum(arg, 1e-300)))), 0.0)
    singular = np.maximum.accumulate(np.nan_to_num(cond, posinf=np.inf) > 500.0, axis=0)
    mask |= singular
    singular = singular[-1]
    melted = int(((want["h_swe"][0] > 0) & (want["h_swe"][-1] == 0)).sum())
    rep = {"cells": N, "steps": T, "cells_melted_out": melted, "knife_edge_cells": int(mask[-1].sum() - singular.sum()),
           "log_law_singular_cells": int(singular.sum())}
    bad = []
    for k in keys:
        ok, ratio, dabs, drel = err_report(got[k][~mask], want[k][~mask], ATOL[k])
        rep[k] = {"ok": ok, "err_over_tol": ratio, "max_abs": dabs, "max_rel": drel}
        if not ok:
            bad.append((k, ratio, dabs, drel))
    _dump(f"random16k/{mode}", rep)
    assert melted > 100
    assert rep["knife_edge_cells"] <= max(5, 0.15 * melted) and singular.sum() <= 0.02 * N, rep
    assert not bad, bad


@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_time_zones_and_dst_per_cell(mode, cuda_device):
    """Cells in different zones (IANA names with DST, fixed offsets) across the March 2013 DST switch: the per-cell
    UTC-offset table (tz_idx) reproduces the oracle's per-instance gmt_offset_hours (solar_funcs.py:1616-1637)."""
    import torch

    from helpers import default_constants
    from oracle.np_ref import CellStatics, Constants, OracleModel
    from topoflow_glacier_b200.engine import MeltEngine

    case = load_case("cats288")
    s = {k: np.tile(v, 2) for k, v in case["statics"].items()}
    s["lon"] = s["lon"] + np.array([0, 0, 0, 0, 15.0, 15.0, -30.0, 0.5])
    zones = ["America/Los_Angeles", "America/Denver", -8.0, "Pacific/Honolulu"]
    tz_idx = np.array([0, 0, 2, 0, 1, 1, 3, 2], dtype=np.uint8)
    T = 120
    forcing = np.tile(case["forcing"][:T], (1, 1, 2))
    start = "2013030800"  # DST begins 2013-03-10 10:00 UTC in the two US zones
    ora = OracleModel(CellStatics(**s, tz=[zones[i] for i in tz_idx]), Constants(), start, strict_pow=True)
    keys = ("TSN_offset", "Qn_SW", "Q_sum", "M_total", "h_swe", "albedo")
    want = ora.run(forcing, record=keys)
    eng = MeltEngine(s, default_constants(), start, zones=zones, tz_idx=tz_idx, mode=mode, horizon_steps=T + 1)
    got = {k: v.cpu().numpy() for k, v in eng.run(torch.as_tensor(forcing).cuda(), record=keys).items()}
    eng.close()
    # solar time normally advances 1 h per step (-23 h at the daily wrap); it stalls for one step when DST begins
    jumps = np.abs(np.diff(want["TSN_offset"], axis=0)) < 0.5
    assert jumps[:, [0, 1, 3, 4, 5]].any(axis=0).all() and not jumps[:, [2, 7]].any()
    for k in keys:
        ok, ratio, dabs, drel = err_report(got[k], want[k], ATOL[k])
        assert ok, (k, ratio, dabs, drel)


@pytest.mark.parametrize("chunk", [0, 7])
@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_snowfall_window_threshold_knife_edge(mode, chunk, cuda_device):
    """The 3-day snowfall total is steered to within ~1e-13 of the 0.03 m threshold (:1040).  The fused kernel keeps
    an incremental sum and must fall back to the exact reference-order re-sum inside its guard band, so the
    'days since snowfall' counter n must equal the oracle's at every step, exactly."""
    import torch

    case = load_case("cats288")
    T, N = 400, case["N"]
    rng = np.random.default_rng(5)
    forcing = np.repeat(case["forcing"][:1], T, axis=0).copy()
    forcing[:, 1] = -5.0                                    # all precipitation falls as snow
    base = 0.03 / 72 / 20.0                                 # 72 identical entries sum to the threshold
    forcing[:, 0] = base * (1.0 + rng.choice([-1, 1], (T, N)) * rng.uniform(0, 3e-13, (T, N)))
    forcing[200:230, 0] = 0.0                               # a dry spell: the total drops below, then recovers
    c2 = dict(case, forcing=forcing)
    ora = make_oracle(c2, strict_pow=True)
    want = ora.run(forcing, record=("n", "snow3day", "albedo"))
    eng = make_engine(c2, mode=mode)
    f_dev = torch.as_tensor(forcing).cuda()
    if chunk:   # short launches: the running window sum is carried from launch to launch (tfg_bind_window_carry)
        parts = []
        for t0 in range(0, T, chunk):
            parts.append(eng.run(f_dev[t0:t0 + chunk].contiguous(), record=("n", "snow3day", "albedo")))
            if t0 == chunk:
                assert torch.isfinite(eng.window_carry[2]).all()    # ... and is in use
        got = {k: torch.cat([pp[k] for pp in parts]).cpu().numpy() for k in parts[0]}
    else:
        got = {k: v.cpu().numpy() for k, v in eng.run(f_dev, record=("n", "snow3day", "albedo")).items()}
    eng.close()
    near = np.abs(want["snow3day"] - 0.03) < 1e-12
    assert near.sum() > 100, near.sum()                     # the test really sits on the knife edge
    flips = np.diff((want["snow3day"] >= 0.03).astype(int), axis=0) != 0
    assert flips.sum() > 20
    assert np.array_equal(got["n"], want["n"])
    # the decisions above are exact; the recorded total is the exact re-sum inside the kernel's drift band
    # (~336 roundings of 0.03 in the strict mode, 1e-9 in the fast mode) and the incremental sum outside it
    np.testing.assert_allclose(got["snow3day"][near], want["snow3day"][near], rtol=0, atol=2e-15)
    tight = np.abs(want["snow3day"] - 0.03) < 1e-16
    assert np.array_equal(got["snow3day"][tight], want["snow3day"][tight])


@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_tma_staged_forcing_is_bit_identical(mode, cuda_device):
    """Forcing tiles through cp.async.bulk + mbarrier (4 stages) == per-thread prefetching loads, bit for bit;
    cell counts that are not a multiple of the block size fall back to the load path transparently."""
    import torch

    import bench
    from helpers import default_constants
    from topoflow_glacier_b200.engine import MeltEngine

    for N, T in ((128 * 37, 29), (128 * 3, 2), (1000, 9)):
        statics, forcing = bench.synthetic_host_sample(N, T, seed=3)
        f = torch.as_tensor(forcing).to(cuda_device, torch.float32 if mode == "f32" else torch.float64)
        basin = (np.arange(N) // 200).astype(np.int32)
        out = []
        for tma in (False, True):
            eng = MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode=mode, horizon_steps=T + 1,
                             basin_id=basin, n_basin=int(basin.max()) + 1, tma_staging=tma)
            agg = torch.zeros(T, int(basin.max()) + 1, 3, dtype=torch.float64, device=cuda_device)
            eng.run(f, basin_agg=agg)
            torch.cuda.synchronize()
            out.append((eng.state.clone(), eng.ring.clone(), agg))
            eng.close()
        assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])
        assert torch.allclose(out[0][2], out[1][2], rtol=1e-12, atol=0)


@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_extreme_and_missing_forcing(mode, cuda_device):
    """Edge inputs: calm air (uz = 0), no precipitation, polar cold / desert heat, vanishing humidity (outside the
    fast mode's sanity window -> its libdevice fallback), and NaN forcing (missing data) in single cells.  Finite
    cells match the oracle; NaN appears in exactly the cells and quantities where the oracle has it."""
    import torch

    case = load_case("rand64")
    T, N = 24, case["N"]
    f = case["forcing"][:T].copy()
    f[:, 4, 0] = 0.0                       # uz == 0: Richardson denominator 0 -> 0.01 (:642-643)
    f[:, 0, 1] = 0.0                       # never any precipitation
    f[:, 1, 2] = -88.0                     # extreme cold
    f[:, 1, 3] = 58.0                      # extreme heat
    f[:, 3, 4] = 3e-9                      # q below the fast path's sanity window
    f[:, 4, 5] = 1e-120                    # denormal-ish wind
    f[:, 2, 6] = 30000.0                   # very low surface pressure
    f[5:, 1, 7] = np.nan                   # temperature missing from step 5 on
    f[9, 0, 8] = np.nan                    # one missing precipitation value
    c2 = dict(case, forcing=f)
    keys = ("RH", "Q_sum", "M_total", "SM", "IM", "h_swe", "h_iwe", "Eccs", "albedo", "Qh")
    want = make_oracle(c2, strict_pow=False).run(f, record=keys)
    eng = make_engine(c2, mode=mode)
    got = {k: v.cpu().numpy() for k, v in eng.run(torch.as_tensor(f).cuda(), record=keys).items()}
    eng.close()
    mask = knife = None
    from helpers import knife_edge_mask
    knife = knife_edge_mask({k: np.nan_to_num(got[k]) for k in ("h_swe", "h_iwe")},
                            {k: np.nan_to_num(want[k]) for k in ("h_swe", "h_iwe")})
    for k in keys:
        assert np.array_equal(np.isnan(got[k]), np.isnan(want[k])), k
        ok, ratio, dabs, drel = err_report(got[k][~knife], want[k][~knife], ATOL[k])
        assert ok, (k, ratio, dabs, drel)
    assert np.isnan(want["Q_sum"][5:, 7]).all() and not np.isnan(want["Q_sum"][:5, 7]).any()
    assert knife[-1].sum() <= 3


def test_engine_argument_errors(cuda_device):
    """Loud failures at the boundary: wrong dtype / shape / device, unknown record names, bad step counts."""
    import torch

    case = load_case("cats288")
    eng = make_engine(case, mode="f64")
    good = torch.as_tensor(case["forcing"][:4]).cuda()
    with pytest.raises(ValueError):
        eng.run(good.float())
    with pytest.raises(ValueError):
        eng.run(good.cpu())
    with pytest.raises(ValueError):
        eng.run(good[:, :4].contiguous(), 4)
    with pytest.raises(ValueError):
        eng.run(good.transpose(1, 2), 4)
    with pytest.raises(KeyError):
        eng.run(good, record=("no_such_quantity",))
    with pytest.raises(RuntimeError):
        eng.run(good, 0)
    with pytest.raises(RuntimeError):  # aggregates requested without basin ids
        eng.run(good, basin_agg=torch.zeros(4, 0, 3, dtype=torch.float64, device="cuda"))
    assert eng.step_index == 0
    eng.run(good)
    assert eng.step_index == 4
    eng.close()


@pytest.mark.parametrize("chunk", [0, 16])
@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_window_sum_recovers_from_missing_precipitation(mode, chunk, cuda_device):
    """A missing (NaN) or absurd (inf) precipitation value poisons the 3-day snowfall total only while it is inside the
    72-slot window -- the reference re-sums the window every step (:1035-1037), so `n` resumes counting 72 steps
    later.  The fused kernel keeps a running sum: it must fall back to the exact re-sum while the sum is not finite
    (ADVICE r1, tfg_run.cuh:334), for one launch and for launches that carry the running sum between them."""
    import torch

    case = load_case("cats288")
    T = 120
    f = case["forcing"][:T].copy()
    f[:, 1] = -4.0                       # snowfall
    f[:, 0] = 2e-5
    f[7, 0, 0] = np.nan                  # cell 0: one missing value
    f[9, 0, 1] = np.inf                  # cell 1: +inf enters, inf - inf = NaN when it leaves the window
    c2 = dict(case, forcing=f)
    want = make_oracle(c2, strict_pow=True).run(f, record=("n", "snow3day"))
    eng = make_engine(c2, mode=mode)
    f_dev = torch.as_tensor(f).cuda()
    if chunk:
        parts = [eng.run(f_dev[t0:t0 + chunk].contiguous(), record=("n", "snow3day")) for t0 in range(0, T, chunk)]
        got = {k: torch.cat([p[k] for p in parts]).cpu().numpy() for k in parts[0]}
    else:
        got = {k: v.cpu().numpy() for k, v in eng.run(f_dev, record=("n", "snow3day")).items()}
    eng.close()
    assert np.isnan(want["snow3day"][7:79, 0]).all() and np.isfinite(want["snow3day"][79:, 0]).all()
    assert np.isfinite(want["snow3day"][81:, 1]).all()
    for k in ("n", "snow3day"):
        assert np.array_equal(np.isnan(got[k]), np.isnan(want[k])), k
        assert np.array_equal(np.isinf(got[k]), np.isinf(want[k])), k
    ok = np.isfinite(want["snow3day"])
    np.testing.assert_allclose(got["snow3day"][ok], want["snow3day"][ok], rtol=1e-12, atol=1e-13)
    assert np.array_equal(got["n"][:, 2:], want["n"][:, 2:])                      # untouched cells: exact
    np.testing.assert_array_equal(got["n"][ok[:, 0], 0], want["n"][ok[:, 0], 0])  # poisoned cells: exact once clean
    np.testing.assert_array_equal(got["n"][ok[:, 1], 1], want["n"][ok[:, 1], 1])


@pytest.mark.parametrize("name,mode", [("cats288", "f64_fast"), ("cfgspace", "f64_fast"), ("south_dt3", "f64_fast"),
                                       ("cats288", "f64"), ("cfgspace", "f64"), ("satterlund", "f64")])
def test_column_term_path_matches_oracle(name, mode, cuda_device):
    """The oracle, through the column-term pass (TFG_OPT_COLUMN_TERMS): every golden cell is replicated `rep` times behind
    a forcing map, so that the forcing-only part of update() is evaluated once per column by column_terms_kernel and the
    melt kernel runs its `PRE` instantiation.  All recorded quantities and integrals of every replica must meet the same
    tolerances as the per-cell path (SURVEY.md section 8a table in helpers.ATOL)."""
    import torch

    from helpers import default_constants
    from topoflow_glacier_b200.engine import MeltEngine

    case, want = oracle_series(name)
    n, T = case["N"], case["forcing"].shape[0]
    rep = max(8, -(-65536 // (min(T, 128) * n)))          # >= 65 536 cell-steps per launch, >= 8 cells per column
    statics = {k: np.repeat(np.asarray(v), rep) for k, v in case["statics"].items()}
    col = np.repeat(np.arange(n, dtype=np.int32), rep)
    consts = default_constants()
    consts.update(case.get("consts", {}))
    eng = MeltEngine(statics, consts, case["start_time"], dt_hours=case.get("dt", 1), zones=[case.get("tz", "America/Los_Angeles")],
                     mode=mode, horizon_steps=T + 1, forcing_index=col, n_forcing_cols=n)
    got = eng.run(torch.as_tensor(case["forcing"]).to(cuda_device), record=REC)
    torch.cuda.synchronize()
    assert eng.column_term_launches >= 1
    got = {k: v.cpu().numpy() for k, v in got.items()}
    got.update({k: eng.row(k).cpu().numpy() for k in VOLS})
    bad = []
    for k in REC + VOLS:
        g = got[k].reshape(*got[k].shape[:-1], n, rep)
        assert (g == g[..., :1]).all() or np.isnan(g).any(), k          # replicas of a cell agree bit for bit
        ok, ratio, dabs, drel = err_report(g[..., 0], want[k], ATOL[k])
        if not ok:
            bad.append((k, ratio, dabs, drel))
    eng.close()
    assert not bad, bad
