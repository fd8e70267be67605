"""The float32 mode (`mode="f32"`) against the oracle beyond the golden cases, and its missing-data semantics.

The float32 kernel has no strict fallback: forcing that is missing (NaN) or extreme runs through its own arithmetic.
These tests hold it to the stated float32 bound (helpers.f32_bound_report, DESIGN.md section 6) on a large random
sample, across a DST switch and on extreme forcing, require NaN in exactly the oracle's cells, steps and quantities, and
check the days-since-snowfall counter bit for bit against a float32 replica of the kernel's snowfall window.
The oracle is fed the float32-rounded forcing widened to float64, so that both sides see the same inputs.
"""

from fractions import Fraction

import numpy as np
import pytest

from helpers import default_constants, err_report, f32_bound_report, load_case, make_engine, make_oracle

THR32 = np.float32(0.03)   # the 0.03 m threshold of :1040 as the float32 kernel compares it


def f32_forcing(f):
    """(float32 forcing for the kernel, the same values widened to float64 for the oracle)."""
    f32 = np.ascontiguousarray(f, dtype=np.float32)
    return f32, f32.astype(np.float64)


def window_sum(ring):
    """The kernel's exact window sum (tfg_run.cuh window_sum_exact, NumPy's pairwise order) of ``ring`` [N, slots],
    oldest entry first, in the dtype of ``ring``: eight interleaved accumulators, then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)),
    then the remainder."""
    slots = ring.shape[1]
    if slots < 8:
        res = np.zeros(ring.shape[0], dtype=ring.dtype)
        for i in range(slots):
            res = res + ring[:, i]
        return res
    r = [ring[:, j].copy() for j in range(8)]
    i = 8
    while i < slots - slots % 8:
        for j in range(8):
            r[j] = r[j] + ring[:, i + j]
        i += 8
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for i in range(slots - slots % 8, slots):
        res = res + ring[:, i]
    return res


def snow_window_replica(P, T_air, T_rs, consts=None, dt=1):
    """Float32 replica of :1027-1041 as the float32 kernel evaluates it: ``(n, total)``, each [T, N] float32.

    Each ring entry is RN32(RN32(P_snow * dt) * ws_ratio) with the constants the library passes, cast to float
    (tfg_abi.cu derive()); the total is window_sum in float32; n is reset where total >= 0.03f and advances by
    (float)days_per_dt where total < 0.03f -- neither for a NaN total."""
    c = default_constants()
    c.update(consts or {})
    dt32, ws32 = np.float32(dt), np.float32(c["rho_H2O"] / c["rho_snow"])
    dpd32 = np.float32(dt / 86400.0)
    P, T_air = np.asarray(P, dtype=np.float32), np.asarray(T_air, dtype=np.float32)
    T_rs = np.asarray(T_rs, dtype=np.float32)
    steps, N = P.shape
    ring = np.zeros((N, int(72 // dt)), dtype=np.float32)
    n = np.zeros(N, dtype=np.float32)
    n_out, tot_out = np.empty((steps, N), np.float32), np.empty((steps, N), np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for t in range(steps):
            P_snow = P[t] * (T_air[t] <= T_rs).astype(np.float32)       # :604, P * bool
            ring = np.roll(ring, -1, axis=1)
            ring[:, -1] = (P_snow * dt32) * ws32
            tot = window_sum(ring)
            n = np.where(tot >= THR32, np.float32(0), n)
            n = np.where(tot < THR32, n + dpd32, n).astype(np.float32)
            n_out[t], tot_out[t] = n, tot
    return n_out, tot_out


def knife_edge_forcing(case, T=400, K=32, seed=5):
    """cats288's first forcing row held for T steps, all snow, with the 72 window entries steered to within a few
    float32 ulps of 0.03 m: P = p0 + k ulp(p0), k uniform in [-K, K], where 72 entries of p0 sum closest to 0.03f;
    a dry spell at steps 200-229 drops the total below the threshold and lets it recover."""
    rng = np.random.default_rng(seed)
    f = np.repeat(case["forcing"][:1], T, axis=0).astype(np.float32)
    f[:, 1] = -5.0
    base = np.float32(0.03 / 72 / 20.0)
    ulp = np.spacing(base)
    ws = np.float32(default_constants()["rho_H2O"] / default_constants()["rho_snow"])
    cands = [np.float32(base + c * ulp) for c in range(-64, 65)]
    p0 = min(cands, key=lambda p: abs(float(window_sum(np.full((1, 72), np.float32(p * ws), np.float32))[0]) - float(THR32)))
    k = rng.integers(-K, K + 1, (T, case["N"]))
    f[:, 0] = (p0 + k.astype(np.float32) * ulp).astype(np.float32)
    f[200:230, 0] = 0.0
    return f


def test_snow_window_replica_self_check():
    """CPU: the replica sums in the reference's order (bit for bit with the oracle's float64 window sum), and in float32
    it decides on the same side of 0.03 as the exact rational sum of its entries wherever that sum is farther from the
    threshold than the float32 summation error (16 roundings of the sum of |entries|).  The steered forcing of
    test_snowfall_threshold_knife_edge_exact really sits on the edge."""
    from oracle.np_ref import _pairwise72

    rng = np.random.default_rng(0)
    ring = rng.uniform(0, 1e-3, (257, 72)) * rng.choice([1.0, 1e-9], (257, 72))
    assert np.array_equal(window_sum(ring), _pairwise72(ring))

    case = load_case("cats288")
    f = knife_edge_forcing(case)
    n, tot = snow_window_replica(f[:, 0], f[:, 1], case["statics"]["T_rain_snow"])
    ws = np.float32(default_constants()["rho_H2O"] / default_constants()["rho_snow"])
    entries = (f[:, 0] * np.float32(1.0)) * ws
    thr = Fraction(float(THR32))
    checked = 0
    for t in range(f.shape[0]):
        for c in range(case["N"]):
            win = entries[max(0, t - 71):t + 1, c]
            exact = sum((Fraction(float(e)) for e in win), Fraction(0))
            if abs(exact - thr) > 16 * 2.0 ** -24 * float(np.abs(win).sum()):
                assert (tot[t, c] < THR32) == (exact < thr), (t, c)
                checked += 1
    assert checked > 200
    near = np.abs(tot.astype(np.float64) - float(THR32)) <= 4 * float(np.spacing(THR32))
    assert near.sum() > 100
    assert (np.diff((tot >= THR32).astype(int), axis=0) != 0).sum() > 20


@pytest.mark.gpu
def test_f32_large_random_sample(cuda_device):
    """16 379 random cells x 36 steps (bench distributions, every 7th pack thinned to melt out inside the window).  N is
    not a multiple of 32: the tail warp runs replica lanes, and the float32 kernel's window slot pointer walks past
    them.  Everything within the float32 bound, with at least 100 melt-outs to move."""
    import torch

    import bench
    from oracle.np_ref import CellStatics, Constants, OracleModel
    from topoflow_glacier_b200.engine import MeltEngine

    N, T = 16379, 36
    statics, forcing = bench.synthetic_host_sample(N, T, seed=11)
    statics["h0_swe"][::7] *= 1e-3
    statics["h0_snow"][::7] *= 1e-3
    f32, f64 = f32_forcing(forcing)
    keys = ("h_swe", "h_iwe", "h_snow", "h_ice", "SM", "IM", "M_total", "RH", "Q_sum", "Qn_SW", "Qn_LW", "Qh", "Qe",
            "albedo", "T_surf")
    ora = OracleModel(CellStatics(**statics, tz=[-8.0]), Constants(), "2013040100", strict_pow=False)
    want = ora.run(f64, record=keys)
    eng = MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f32", horizon_steps=T + 1)
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in eng.run(torch.as_tensor(f32).to(cuda_device), record=keys).items()}
    eng.close()
    rep, bad = f32_bound_report(got, want, statics["h0_snow"])
    assert rep["melt_out_events"] >= 100, rep
    assert not bad, (bad, rep)


@pytest.mark.gpu
def test_f32_time_zones_and_dst_per_cell(cuda_device):
    """Per-cell zones (IANA names with DST, fixed offsets) across the March 2013 DST switch in float32: the solar-time
    stall falls at the oracle's steps, and fluxes and depths meet the float32 bound."""
    import torch

    from oracle.np_ref import CellStatics, Constants, OracleModel
    from topoflow_glacier_b200.engine import MeltEngine

    case = load_case("cats288")
    s = {k: np.tile(v, 2) for k, v in case["statics"].items()}
    s["lon"] = s["lon"] + np.array([0, 0, 0, 0, 15.0, 15.0, -30.0, 0.5])
    zones = ["America/Los_Angeles", "America/Denver", -8.0, "Pacific/Honolulu"]
    tz_idx = np.array([0, 0, 2, 0, 1, 1, 3, 2], dtype=np.uint8)
    T = 120
    f32, f64 = f32_forcing(np.tile(case["forcing"][:T], (1, 1, 2)))
    start = "2013030800"  # DST begins 2013-03-10 10:00 UTC in the two US zones
    ora = OracleModel(CellStatics(**s, tz=[zones[i] for i in tz_idx]), Constants(), start, strict_pow=True)
    keys = ("TSN_offset", "Qn_SW", "Q_sum", "M_total", "h_swe", "h_snow", "h_iwe", "albedo")
    want = ora.run(f64, record=keys)
    eng = MeltEngine(s, default_constants(), start, zones=zones, tz_idx=tz_idx, mode="f32", horizon_steps=T + 1)
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in eng.run(torch.as_tensor(f32).to(cuda_device), record=keys).items()}
    eng.close()
    stall_want = np.abs(np.diff(want["TSN_offset"], axis=0)) < 0.5
    stall_got = np.abs(np.diff(got["TSN_offset"], axis=0)) < 0.5
    assert stall_want[:, [0, 1, 3, 4, 5]].any(axis=0).all() and not stall_want[:, [2, 7]].any()
    assert np.array_equal(stall_got, stall_want)
    ok, ratio, dabs, drel = err_report(got["TSN_offset"], want["TSN_offset"], 1e-4, 0)   # hours
    assert ok, ("TSN_offset", ratio, dabs, drel)
    rep, bad = f32_bound_report(got, want, s["h0_snow"])
    assert not bad, (bad, rep)


NAN_KEYS = ("h_swe", "h_iwe", "SM", "IM", "M_total", "Eccs", "Ecci", "Q_sum", "T_surf", "P_rain", "P_snow", "n", "snow3day",
            "albedo")


@pytest.mark.gpu
def test_f32_extreme_and_missing_forcing(cuda_device):
    """The edits of test_extreme_and_missing_forcing, plus a NaN precipitation value while it snows and a NaN T_air for
    one step and from a step on.  NaN appears in exactly the oracle's cells, steps and quantities (a missing value
    poisons the cell's pack as in the reference); finite values meet the float32 bound."""
    import torch

    case = load_case("rand64")
    T, N = 24, case["N"]
    f = case["forcing"][:T].copy()
    f[:, 4, 0] = 0.0                       # uz == 0: Richardson denominator 0 -> 0.01 (:642-643)
    f[:, 0, 1] = 0.0                       # never any precipitation
    f[:, 1, 2] = -88.0                     # extreme cold
    f[:, 1, 3] = 58.0                      # extreme heat
    f[:, 3, 4] = 3e-9                      # vanishing humidity
    f[:, 4, 5] = 1e-120                    # denormal-ish wind: 0 in float32 (and so for the oracle here)
    f[:, 2, 6] = 30000.0                   # very low surface pressure
    f[5:, 1, 7] = np.nan                   # temperature missing from step 5 on
    f[9, 0, 8] = np.nan                    # one missing precipitation value
    f[:, 1, 9] = -6.0                      # snowing ...
    f[:, 0, 9] = 5e-4
    f[12, 0, 9] = np.nan                   # ... when one precipitation value is missing
    f[10, 0, 10] = 3e-4
    f[10, 1, 10] = np.nan                  # temperature missing for one step (while it precipitates)
    f[15:, 1, 11] = np.nan                 # temperature missing from step 15 on
    f32, f64 = f32_forcing(f)
    c2 = dict(case, forcing=f64)
    keys = NAN_KEYS + ("h_snow", "h_ice", "Qn_SW", "Qn_LW", "Qh", "Qe", "RH")
    ora = make_oracle(c2, strict_pow=False)
    want = ora.run(f64, record=keys)
    eng = make_engine(c2, mode="f32")
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in eng.run(torch.as_tensor(f32).to(cuda_device), record=keys).items()}
    vols = {k: eng.row(k).cpu().numpy().astype(np.float64) for k in ("vol_PR", "vol_PS")}
    eng.close()
    # the oracle side of each edit: the pack of the snowing cell and both temperature cells is poisoned for good, the
    # single missing temperature gives no precipitation and a NaN energy sum for one step
    assert np.isnan(want["h_swe"][12:, 9]).all() and not np.isnan(want["h_swe"][:12, 9]).any()
    assert np.isnan(want["Q_sum"][10:, 10]).all() and not np.isnan(want["Q_sum"][:10, 10]).any()
    assert want["P_rain"][10, 10] == 0 and want["P_snow"][10, 10] == 0 and f[10, 0, 10] > 0
    assert np.isnan(want["Q_sum"][15:, 11]).all() and np.isnan(want["Q_sum"][5:, 7]).all()
    for k in keys:
        bad = np.argwhere(np.isnan(got[k]) != np.isnan(want[k]))
        assert len(bad) == 0, (k, "NaN pattern differs at (step, cell)", bad[:8].tolist())
    for k in ("P_rain", "P_snow"):   # P * bool of the same float32 values: exact
        assert np.array_equal(got[k], want[k], equal_nan=True), k
    for k, v in vols.items():
        w = getattr(ora, k)
        assert np.array_equal(np.isnan(v), np.isnan(w)), k
        ok, ratio, dabs, drel = err_report(v, w, 1e-9, 1e-5)
        assert ok, (k, ratio, dabs, drel)
    ok, ratio, dabs, drel = err_report(got["n"], want["n"], 0, 1e-5)
    assert ok and np.array_equal(got["n"] == 0, want["n"] == 0), ("n", ratio, dabs, drel)
    rep, bad = f32_bound_report(got, want, case["statics"]["h0_snow"])
    assert not bad, (bad, rep)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 16])
def test_f32_window_sum_recovers_from_missing_precipitation(chunk, cuda_device):
    """Float32 twin of test_window_sum_recovers_from_missing_precipitation.  A NaN or +inf precipitation value poisons
    the 3-day snowfall total only while it is inside the 72-slot window, and NaN holds `n` where the reference holds
    it: the NaN and inf patterns of `n` and `snow3day` are the oracle's.  `n` accumulates float32 days, so it is
    compared bit for bit with the float32 replica (and its resets with the oracle's); the total is within the running
    sum's drift bound of the oracle's."""
    import torch

    case = load_case("cats288")
    T = 120
    f = case["forcing"][:T].copy()
    f[:, 1] = -4.0                       # snowfall
    f[:, 0] = 2e-5
    f[7, 0, 0] = np.nan                  # cell 0: one missing value
    f[9, 0, 1] = np.inf                  # cell 1: +inf enters, inf - inf = NaN when it leaves the window
    f32, f64 = f32_forcing(f)
    c2 = dict(case, forcing=f64)
    want = make_oracle(c2, strict_pow=True).run(f64, record=("n", "snow3day"))
    n_rep, _ = snow_window_replica(f32[:, 0], f32[:, 1], case["statics"]["T_rain_snow"])
    eng = make_engine(c2, mode="f32")
    f_dev = torch.as_tensor(f32).to(cuda_device)
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
    assert np.array_equal(got["n"], n_rep)
    assert np.array_equal(got["n"] == 0, want["n"] == 0)
    ok = np.isfinite(want["snow3day"])
    # the running sum drifts by at most its guard band: 1.2e-7 per rounding, (72 seed + 2 per step) roundings
    np.testing.assert_allclose(got["snow3day"][ok], want["snow3day"][ok], rtol=1.2e-7 * (72 + 2 * T), atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 7])
def test_snowfall_threshold_knife_edge_exact(chunk, cuda_device):
    """The float32 kernel's incremental window sum must fall back to the exact re-sum inside its guard band
    (1.2e-7 x rounding count, tfg_run.cuh): with the 72 entries steered to within a few float32 ulps of 0.03 m, `n` equals
    the float32 replica bit for bit at every step, fused and in 7-step launches that carry the running sum; near the
    threshold the recorded total is the exact re-sum."""
    import torch

    case = load_case("cats288")
    f = knife_edge_forcing(case)
    T = f.shape[0]
    n_rep, tot_rep = snow_window_replica(f[:, 0], f[:, 1], case["statics"]["T_rain_snow"])
    near = np.abs(tot_rep.astype(np.float64) - float(THR32)) <= 4 * float(np.spacing(THR32))
    assert near.sum() > 100, near.sum()                     # the test really sits on the knife edge
    assert (np.diff((tot_rep >= THR32).astype(int), axis=0) != 0).sum() > 20
    eng = make_engine(dict(case, forcing=f), mode="f32")
    f_dev = torch.as_tensor(f).to(cuda_device)
    if chunk:   # short launches: the running window sum is carried from launch to launch (tfg_bind_window_carry)
        parts = []
        for t0 in range(0, T, chunk):
            parts.append(eng.run(f_dev[t0:t0 + chunk].contiguous(), record=("n", "snow3day")))
            if t0 == chunk:
                assert torch.isfinite(eng.window_carry[2]).all()    # ... and is in use
        got = {k: torch.cat([pp[k] for pp in parts]).cpu().numpy() for k in parts[0]}
    else:
        got = {k: v.cpu().numpy() for k, v in eng.run(f_dev, record=("n", "snow3day")).items()}
    eng.close()
    bad = np.argwhere(got["n"] != n_rep)
    assert len(bad) == 0, ("n differs at (step, cell)", bad[:8].tolist(), int(len(bad)))
    assert np.array_equal(got["snow3day"][near], tot_rep[near])
