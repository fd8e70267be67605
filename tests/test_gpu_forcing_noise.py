"""Stochastic forcing perturbations (tfg_bind_forcing_noise): the device series equals a NumPy replica of its definition
within a derived bound and has the statistics it claims; a perturbed forcing map equals per-cell forcing perturbed with
torch from that series, bit for bit, in every mode; results do not depend on the launch split, the per-step paths, a
checkpoint rewind or sharding; without noise nothing moves; errors name the field."""

import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from helpers import default_constants

ROOT = Path(__file__).resolve().parent.parent
COUNTER_TAG = 0x4E4F4953


def _bits(x):
    import torch

    x = x.contiguous()
    return x.view(torch.int32 if x.element_size() == 4 else torch.int64)


def _same(a, b):
    """Bit for bit (NaN patterns included)."""
    import torch

    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


# ---------------------------------------------------------------------------------------------------- host replica
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint64 arrays holding 32-bit words (the round function of tfg_abi.cu's philox4x32_10)."""
    c = [np.asarray(v, dtype=np.uint64) & _M32 for v in (c0, c1, c2, c3)]
    k0, k1 = np.asarray(k0, dtype=np.uint64) & _M32, np.asarray(k1, dtype=np.uint64) & _M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _M32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _M32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return c


def host_normals(seed, ids, s):
    """(e_T, e_P, r) of every stream id at absolute step s, float64, as include/tfglacier.h defines them."""
    ids = np.asarray(ids, dtype=np.int64).astype(np.uint64)
    w = philox4x32_10(ids & _M32, ids >> np.uint64(32), np.full(ids.shape, s, np.uint64), np.full(ids.shape, COUNTER_TAG,
                      np.uint64), np.uint64(seed) & _M32, np.uint64(seed) >> np.uint64(32))
    a = (w[0] << np.uint64(21)) | (w[1] >> np.uint64(11))
    b = (w[2] << np.uint64(21)) | (w[3] >> np.uint64(11))
    ua = (a + np.uint64(1)).astype(np.float64) * 2.0**-53
    ub = b.astype(np.float64) * 2.0**-53
    r = np.sqrt(-2.0 * np.log(ua))
    x = 2.0 * ub
    return r * np.cos(np.pi * x), r * np.sin(np.pi * x), r


# Error bounds of one step of the replica against the device (libdevice), from the functions' documented accuracy:
# log and sincospi within 1 ulp on the device, glibc's log within 1 ulp, and cos(pi * x) on the host off by the rounding
# of pi * x (|pi x| < 2 pi, so < 2 pi * 2^-53 absolute) plus 1 ulp.  Then |r' - r| / r <= 2^-51 (half the log's relative
# error, plus the two square roots' roundings), |trig' - trig| <= 8 * 2^-52, and each product adds half an ulp per side.
EPS = 2.0**-52


def replica_with_bound(seed, ids, s0, step0, n, sd_T, rho_T, sd_P, rho_P):
    """Host series dT, fP [n, n_streams] for steps [step0, step0 + n) and elementwise bounds on |device - host|.

    The per-step error delta of e is carried through z(s) = rho z(s-1) + c e(s) as B(s) = rho B(s-1) + c delta(s) + the
    three roundings of the step (at most an ulp each of |rho z|, |c e| and |z| when the inputs differ): a per-step error
    amplified at most 1 / (1 - rho) times."""
    out = {}
    for q, sd, rho in (("T", sd_T, rho_T), ("P", sd_P, rho_P)):
        out[q] = (sd, rho, np.sqrt(1.0 - rho * rho))
    z = {"T": None, "P": None}
    B = {"T": 0.0, "P": 0.0}
    dT, fP, bT, bP = [], [], [], []
    for s in range(s0, step0 + n):
        eT, eP, r = host_normals(seed, ids, s)
        delta = r * (11 * EPS)
        for q, e in (("T", eT), ("P", eP)):
            sd, rho, c = out[q]
            if s == s0:
                z[q], B[q] = e, delta
            else:
                prev = z[q]
                z[q] = rho * prev + c * e
                B[q] = rho * B[q] + c * delta + EPS * (np.abs(rho * prev) + np.abs(c * e) + np.abs(z[q]))
        if s >= step0:
            dT.append(sd_T * z["T"])
            bT.append(sd_T * B["T"] + EPS * np.abs(sd_T * z["T"]))       # + the product's rounding on both sides
            half = 0.5 * (sd_P * sd_P)
            f = np.exp(sd_P * z["P"] - half)
            fP.append(f)
            # the exponent's error (B carried, plus its two roundings on both sides), through exp: f * expm1(da); then
            # the two exponentials' 1 ulp each
            da = sd_P * B["P"] + 2 * EPS * (np.abs(sd_P * z["P"]) + half)
            bP.append(f * np.expm1(da) + 2 * EPS * f)
    return np.array(dT), np.array(fP), np.array(bT), np.array(bP)


# ---------------------------------------------------------------------------------------------------- host only
def test_philox_replica_reproduces_the_random123_known_answers():
    for ctr, key, want in (((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
                           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
                           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
                            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))):
        got = philox4x32_10(*ctr, *key)
        assert tuple(int(w) for w in got) == want


def test_header_declares_the_binding_and_ctypes_matches_it():
    from topoflow_glacier_b200 import _lib

    header = (ROOT / "include" / "tfglacier.h").read_text()
    assert ("TFG_API int tfg_bind_forcing_noise(tfg_ctx* ctx, const tfg_forcing_noise* n, void* stream);" in header)
    assert ("TFG_API int tfg_forcing_noise_series(tfg_ctx* ctx, int64_t step0, int32_t n_steps, void* dT, void* fP, "
            "void* stream);" in header)
    body = re.search(r"typedef struct tfg_forcing_noise \{(.*?)\} tfg_forcing_noise;", header, re.S).group(1)
    decls = re.findall(r"^\s*(const \w+\*|\w+)\s+([\w, ]+);", body, re.M)
    ctype = {"uint64_t": C.c_uint64, "int64_t": C.c_int64, "double": C.c_double, "const int64_t*": C.c_void_p,
             "const int32_t*": C.c_void_p}
    fields = [(n.strip(), ctype[t]) for t, names in decls for n in names.split(",")]
    assert [n for n, _ in fields] == ["seed", "step0", "T_air_sd", "T_air_rho", "P_sd", "P_rho", "n_streams",
                                      "stream_id", "cell_stream"]
    assert [(n, t) for n, t in _lib.ForcingNoise._fields_] == fields
    assert C.sizeof(_lib.ForcingNoise) == 9 * 8
    assert _lib.PROTOTYPES["tfg_bind_forcing_noise"] == (C.c_int, [C.c_void_p, C.POINTER(_lib.ForcingNoise), C.c_void_p])
    assert _lib.PROTOTYPES["tfg_forcing_noise_series"] == (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                                                     C.c_void_p, C.c_void_p])


def test_check_forcing_noise_ranges():
    import torch

    from topoflow_glacier_b200.config import FORCING_NOISE_RANGES, check_forcing_noise

    assert FORCING_NOISE_RANGES == {"T_air_sd": (0.0, 5.0), "T_air_rho": (0.0, 1.0), "P_sd": (0.0, 1.5),
                                    "P_rho": (0.0, 1.0)}
    for ends in ((0, 0), (1, 1)):
        ok = {k: r[e] for (k, r), e in zip(FORCING_NOISE_RANGES.items(), ends * 2)}
        got = check_forcing_noise(dict(ok, seed=2**64 - 1, step0=2**32 - 1, stream=torch.tensor([0, 2**40])))
        assert got["seed"] == 2**64 - 1 and got["step0"] == 2**32 - 1
    check_forcing_noise({"seed": 0, "stream": np.array([0, 5])})
    for k, (lo, hi) in FORCING_NOISE_RANGES.items():
        for bad in (np.nan, np.inf, -np.inf, np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)):
            with pytest.raises(ValueError, match=k):
                check_forcing_noise({"seed": 1, k: bad})
    for bad in (-1, 2**64, 1.5, True):
        with pytest.raises(ValueError, match="seed"):
            check_forcing_noise({"seed": bad})
    with pytest.raises(ValueError, match="seed"):
        check_forcing_noise({"T_air_sd": 1.0})
    for bad in (-1, 2**32, 0.5):
        with pytest.raises(ValueError, match="step0"):
            check_forcing_noise({"seed": 1, "step0": bad})
    with pytest.raises(ValueError, match="stream"):
        check_forcing_noise({"seed": 1, "stream": np.array([3, -1])})
    with pytest.raises(ValueError, match="T_sd"):
        check_forcing_noise({"seed": 1, "T_sd": 1.0})


# ---------------------------------------------------------------------------------------------------- GPU helpers
def _engine(statics, mode, T, **kw):
    from topoflow_glacier_b200.engine import MeltEngine

    N = statics["lat"].size
    basin = kw.pop("basin_id", (np.arange(N) // 384).astype(np.int32))
    return MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode=mode, horizon_steps=T + 1,
                      basin_id=basin, n_basin=int(basin.max()) + 1, **kw)


def _setup(n_per_col=256, M=6, T=300, seed=91, n_streams=64, odd=True):
    """M catchment columns of n_per_col cells on a forcing map; n_streams global stream ids (some above 2^32) spread
    across the catchments; adjustments at their range ends; with ``odd``, NaN rows and forcings the noise pushes out
    of the fast mode's lean ranges (T_air near 90 degC, P near 10 m/h)."""
    import bench
    from topoflow_glacier_b200.config import CELL_PARAM_RANGES

    N = n_per_col * M
    statics, _ = bench.synthetic_host_sample(N, 1, seed=seed)
    _, fcols = bench.synthetic_host_sample(M, T, seed=seed + 1)
    fcols = fcols.copy()
    if odd and T >= 100:
        fcols[40, :, 1 % M] = np.nan
        fcols[41, 1, 2 % M] = np.nan
        fcols[60:64, 1, 3 % M] = 80.0
        fcols[80:84, 0, 4 % M] = 2.0
        fcols[90, 1, 0] = -85.0
    col = np.repeat(np.arange(M, dtype=np.int32), n_per_col)
    rng = np.random.default_rng(seed + 2)
    ids = rng.choice(np.concatenate([np.arange(1000, 1000 + n_streams), 2**33 + np.arange(n_streams)]), n_streams,
                     replace=False).astype(np.int64)
    stream = ids[rng.integers(0, n_streams, N)]
    stream[:n_streams] = ids                                   # every id is read
    off, mul = rng.uniform(-30.0, 30.0, N), rng.uniform(0.0, 10.0, N)
    off[0::7], off[3::7], mul[0::7], mul[3::7] = -30.0, 30.0, 0.0, 10.0
    adj = {"T_air_offset": off, "P_multiplier": mul}
    params = {k: rng.uniform(lo, hi, N) for k, (lo, hi) in CELL_PARAM_RANGES.items()}
    noise = {"T_air_sd": 5.0, "T_air_rho": 0.9, "P_sd": 1.5, "P_rho": 0.5, "seed": 2**63 + 12345, "stream": stream}
    return statics, np.ascontiguousarray(fcols), col, adj, params, noise


def _perturbed_per_cell(fc, col, adj, dT, fP, cell_stream, dtype):
    """Per-cell forcing replicated from the columns and perturbed with torch in the engine dtype:
    T_air' = (T_air + off) + dT[stream], P' = (P * mul) * fP[stream] (off = 0, mul = 1 without adjustments)."""
    import torch

    dev = fc.device
    f = fc[:, :, torch.as_tensor(col, dtype=torch.int64, device=dev)].clone()
    N = f.shape[2]
    off = torch.as_tensor(adj["T_air_offset"] if adj else np.zeros(N)).to(dev).to(dtype)
    mul = torch.as_tensor(adj["P_multiplier"] if adj else np.ones(N)).to(dev).to(dtype)
    cs = cell_stream.to(torch.int64)
    f[:, 1] = (f[:, 1] + off) + dT[:, cs]
    f[:, 0] = (f[:, 0] * mul) * fP[:, cs]
    return f.contiguous()


def _run_all(e, f, T, record=True):
    import torch

    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.sharding import BasinAggregates

    agg = BasinAggregates(T, e.n_basin, device=e.device, exponents=e.agg_exponents())
    rec = e.run(f, T, record=_lib.REC_NAMES if record else None, basin_agg=agg.accumulator)
    torch.cuda.synchronize()
    return rec, e.state.clone(), e.ring.clone(), e.window_carry.clone(), agg.accumulator.clone()


def _assert_same_run(a, b):
    from topoflow_glacier_b200 import _lib

    for name in _lib.REC_NAMES:
        if name in a[0] or name in b[0]:
            assert _same(a[0][name], b[0][name]), name
    for i, what in ((1, "state"), (2, "window"), (3, "running window sum"), (4, "exact basin words")):
        assert _same(a[i], b[i]), what


def _state(e):
    import torch

    torch.cuda.synchronize()
    return e.state.clone(), e.ring.clone()


def _assert_same_state(a, b):
    assert _same(a[0], b[0]), "state"
    assert _same(a[1], b[1]), "window"


# ---------------------------------------------------------------------------------------------------- 1. generator
@pytest.mark.gpu
@pytest.mark.parametrize("rho", [0.0, 0.9, 1.0])
def test_series_equals_the_host_replica_within_its_bound(rho, cuda_device):
    """float64 series against the NumPy replica, within the derived bound; both float64 modes give the same bits, and
    the float32 series is the float64 one rounded to float32."""
    import torch

    T, s0, step0 = 400, 5, 9
    statics, _, _, _, _, _ = _setup(n_per_col=64, M=2, T=2, odd=False)
    N = statics["lat"].size
    ids = np.arange(N, dtype=np.int64) * 977 + np.where(np.arange(N) % 2, 2**32 + 3, 0)
    noise = {"T_air_sd": 5.0, "T_air_rho": rho, "P_sd": 1.5, "P_rho": rho, "seed": 0xDEADBEEF12345678, "stream": ids,
             "step0": s0}
    got = {}
    for mode in ("f64", "f64_fast", "f32"):
        e = _engine(statics, mode, T + step0, forcing_noise=noise)
        dT, fP, sid = e.forcing_noise_series(step0, T)
        got[mode] = (dT.clone(), fP.clone(), sid.cpu().numpy())
        e.close()
    assert _same(got["f64"][0], got["f64_fast"][0]) and _same(got["f64"][1], got["f64_fast"][1])
    assert _same(got["f32"][0], got["f64"][0].float()) and _same(got["f32"][1], got["f64"][1].float())
    sid = got["f64"][2]
    assert np.array_equal(sid, np.unique(ids))
    hT, hP, bT, bP = replica_with_bound(noise["seed"], sid, s0, step0, T, 5.0, rho, 1.5, rho)
    dT, fP = got["f64"][0].cpu().numpy(), got["f64"][1].cpu().numpy()
    errT, errP = np.abs(dT - hT), np.abs(fP - hP)
    assert np.all(errT <= bT), (errT.max(), bT[errT > bT][:5])
    assert np.all(errP <= bP), (errP.max(), bP[errP > bP][:5])
    assert bT.max() < 1e-11 and np.max(bP / hP) < 1e-11        # the bound itself says something
    if rho == 1.0:                                               # a constant random bias per stream
        assert np.array_equal(dT, np.broadcast_to(dT[0], dT.shape))


@pytest.mark.gpu
def test_series_statistics(cuda_device):
    """4096 streams x 2000 steps: mean, variance and lag-1 autocorrelation of z, the T-P and stream-stream
    correlations and the mean of fP within 5 standard errors of 0, 1, rho, 0, 0 and 1 (standard errors of an AR(1)
    series)."""
    S, T, rho, sd_T, sd_P = 4096, 2000, 0.7, 2.0, 0.8
    statics, _, _, _, _, _ = _setup(n_per_col=S // 4, M=4, T=2, odd=False)
    e = _engine(statics, "f64", T, forcing_noise={"T_air_sd": sd_T, "T_air_rho": rho, "P_sd": sd_P, "P_rho": rho,
                                                   "seed": 42})
    dT, fP, _ = e.forcing_noise_series(0, T)
    dT, fP = dT.cpu().numpy(), fP.cpu().numpy()
    e.close()
    zT = dT / sd_T
    zP = (np.log(fP) + 0.5 * sd_P**2) / sd_P
    n = S * T
    sum_r2 = (1 + rho**2) / (1 - rho**2)                         # sum over all lags of rho^(2|k|)
    for z in (zT, zP):
        assert abs(z.mean()) <= 5 * np.sqrt((1 + rho) / (1 - rho) / n)
        assert abs(z.var() - 1.0) <= 5 * np.sqrt(2.0 * sum_r2 / n)
        r1 = np.sum(z[1:] * z[:-1]) / np.sum(z * z)
        assert abs(r1 - rho) <= 5 * np.sqrt((1 - rho**2) / n) + 1.0 / T   # plus the estimator's O(1/T) bias
    assert abs(np.mean(zT * zP)) <= 5 * np.sqrt(sum_r2 / n)
    pair = np.mean(zT[:, 0::2] * zT[:, 1::2], axis=0)               # 2048 independent pairs of streams
    assert abs(pair.mean()) <= 5 * np.sqrt(sum_r2 / T / pair.size)
    v = np.exp(sd_P**2) - 1.0
    k = np.arange(1, 400)
    var_mean = (v + 2.0 * np.sum(np.exp(sd_P**2 * rho**k) - 1.0)) / n
    assert abs(fP.mean() - 1.0) <= 5 * np.sqrt(var_mean)


# ---------------------------------------------------------------------------------------------------- 2. equivalence
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
@pytest.mark.parametrize("with_adj,with_params,with_obj", [(False, False, False), (True, False, False),
                                                            (False, True, True), (True, True, True)])
def test_perturbed_map_equals_perturbed_per_cell_forcing(mode, with_adj, with_params, with_obj, cuda_device):
    """300 steps (three launches) on a forcing map with noise bound against per-cell forcing perturbed in advance
    from forcing_noise_series, bit for bit; with an objective, its sums also equal the host loop."""
    import torch

    from topoflow_glacier_b200.objective import series_sums

    T = 300
    statics, fcols, col, adj, params, noise = _setup(T=T)
    N, M = col.size, fcols.shape[2]
    dtype = torch.float32 if mode == "f32" else torch.float64
    fc = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    obs = np.random.default_rng(7).uniform(0.0, 1.0, (250, M))
    obs[::9] = np.nan
    kw = dict(cell_params=params if with_params else None)
    mapped = _engine(statics, mode, T, forcing_index=col, n_forcing_cols=M, forcing_noise=noise,
                     forcing_adjust=adj if with_adj else None, **kw)
    assert mapped.forcing_noise is not None and mapped.forcing_noise["stream_id"].numel() == 64
    dT, fP, _ = mapped.forcing_noise_series(0, T)
    fcell = _perturbed_per_cell(fc, col, adj if with_adj else None, dT, fP, mapped.forcing_noise["cell_stream"], dtype)
    assert bool(torch.isnan(fcell).any())
    if mode == "f64_fast":                                       # the strict fallback runs on perturbed values
        assert bool((fcell[:, 1].abs() >= 90.0).any()) and bool((fcell[:, 0] >= 10.0).any())
    out = []
    for e, f in ((mapped, fc), (_engine(statics, mode, T, **kw), fcell)):
        if with_obj:
            e.set_objective("h_swe", obs, obs_step0=20, obs_index=col)
        got = _run_all(e, f, T)
        assert e.column_term_launches == 0
        out.append((got, torch.stack(e.objective_sums()).clone() if with_obj else None))
        e.close()
    _assert_same_run(out[0][0], out[1][0])
    if with_obj:
        assert _same(out[0][1], out[1][1])
        o_cell = np.full((T, N), np.nan)
        o_cell[20:270] = obs[:, col]
        want, _ = series_sums(out[0][0][0]["h_swe"].double().cpu(), o_cell)
        assert _same(out[0][1].cpu(), want)


# ---------------------------------------------------------------------------------------------------- 3. reproducibility
BMI_CONFIG = {"site_prefix": "cat-x", "forcing_file": "-", "dt": 1, "start_time": "2013040100",
              "end_time": "2013043000", "da": 11.4, "slope": 88.6, "aspect": 242.9, "lon": -121.8, "lat": 46.8,
              "elev": 2446.4, "h0_snow": 5.0, "h0_ice": 2.0, "h0_swe": 0.25, "h0_iwe": 1.834, "T_rain_snow": 0.0,
              "utc_offset_hours": -8.0}
BMI_INPUTS = ("atmosphere_water__liquid_equivalent_precipitation_rate", "land_surface_air__temperature",
              "land_surface_air__pressure", "atmosphere_air_water~vapor__relative_saturation", "wind_speed_UV")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_launch_split_per_step_paths_and_rewind_equal_the_straight_run(mode, cuda_device):
    """One 300-step run equals 300 step() calls, launches of 7 + 121 + 172 steps, BMI update() after set_value (whose
    input variables keep what the caller set), and a rewind to step 50 followed by a rerun."""
    import torch

    from topoflow_glacier_b200 import BmiTopoflowGlacier

    T = 300
    statics, fcols, col, adj, _, noise = _setup(n_per_col=64, M=3, T=T, seed=23, n_streams=16)
    M = fcols.shape[2]
    dtype = torch.float32 if mode == "f32" else torch.float64
    fc = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    kw = dict(forcing_index=col, n_forcing_cols=M, forcing_noise=noise, forcing_adjust=adj)
    straight = _engine(statics, mode, T, **kw)
    straight.run(fc)
    want = _state(straight)
    straight.close()

    steps = _engine(statics, mode, T, **kw)
    for t in range(T):
        steps.inputs[:5].copy_(fc[t])
        steps.step()
    _assert_same_state(_state(steps), want)
    steps.close()

    split = _engine(statics, mode, T, **kw)
    for a, b in ((0, 7), (7, 128), (128, 300)):
        split.run(fc[a:b].contiguous())
    _assert_same_state(_state(split), want)
    split.close()

    rew = _engine(statics, mode, T, **kw)
    rew.run(fc[:50].contiguous())
    sd = rew.state_dict()
    rew.run(fc[50:].contiguous())
    rew.load_state_dict(sd)
    assert rew.step_index == 50
    rew.run(fc[50:].contiguous())
    _assert_same_state(_state(rew), want)
    rew.close()

    bmi = BmiTopoflowGlacier()
    bmi.initialize_cells(dict(BMI_CONFIG, precision=mode), dict(statics, **adj), forcing_index=col, n_forcing_cols=M,
                         forcing_noise=noise)
    assert bmi._engine.forcing_noise is not None
    for t in range(T):
        for name, v in zip(BMI_INPUTS, fcols[t]):
            bmi.set_value(name, np.ascontiguousarray(v))
        bmi.update()
    _assert_same_state(_state(bmi._engine), want)
    got = bmi.get_value("land_surface_air__temperature", np.empty(M))
    assert np.array_equal(got, fcols[T - 1, 1].astype(np.float32 if mode == "f32" else np.float64), equal_nan=True)
    bmi.finalize()


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_sharded_engine_two_ranks_equal_one(tmp_path, cuda_device):
    """Two gloo ranks, each listing only the streams its cells read, equal one engine in state and exact words."""
    import os
    import subprocess
    import sys

    import torch

    from topoflow_glacier_b200.engine import MeltEngine
    from topoflow_glacier_b200.sharding import BasinAggregates

    T, NB = 150, 7
    statics, fcols, col, _, _, noise = _setup(n_per_col=640, M=8, T=T, seed=37)
    N, M = col.size, fcols.shape[2]
    basin = np.random.default_rng(4).integers(0, NB, N).astype(np.int32)
    np.savez(tmp_path / "in.npz", forcing=fcols, basin=basin, col=col, stream=noise["stream"],
             **{f"s_{k}": v for k, v in statics.items()})
    one = MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", basin_id=basin,
                     n_basin=NB, horizon_steps=T + 1, forcing_index=col, n_forcing_cols=M, forcing_noise=noise)
    agg = BasinAggregates(T, NB, device=cuda_device, exponents=one.agg_exponents())
    one.run(torch.as_tensor(fcols).cuda(), basin_agg=agg.zero())
    agg.reduce()
    torch.cuda.synchronize()
    scalars = {k: v for k, v in noise.items() if k != "stream"}
    script = tmp_path / "w.py"
    script.write_text(f'''
import os, sys
sys.path.insert(0, {str(ROOT)!r})
os.environ["NGEN_EWTS_LOGGING"] = "DISABLED"
import numpy as np, torch, torch.distributed as dist
from topoflow_glacier_b200.config import default_constants
from topoflow_glacier_b200.sharding import ShardedMeltEngine
dist.init_process_group("gloo")
rank = dist.get_rank()
z = np.load({str(tmp_path / "in.npz")!r})
statics = {{k[2:]: z[k] for k in z.files if k.startswith("s_")}}
f = torch.as_tensor(z["forcing"]).cuda()
T = f.shape[0]
sh = ShardedMeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", basin_id=z["basin"],
                       n_basin={NB}, horizon_steps=T + 1, device=0, forcing_index=z["col"], n_forcing_cols={M},
                       forcing_noise=dict({scalars!r}, stream=z["stream"]))
_, g = sh.run(f)
lo, hi = sh.bounds
np.savez({str(tmp_path)!r} + f"/out{{rank}}.npz", words=sh.aggregates(T).accumulator.cpu().numpy(),
         state=sh.state.cpu().numpy(), lo=lo, hi=hi, n_streams=sh.engine.forcing_noise["stream_id"].numel())
dist.destroy_process_group()
sys.stdout.write("rank %d ok\\n" % rank)
''')
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29637", str(script)],
                       capture_output=True, text=True, env=env, timeout=560)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    outs = [np.load(tmp_path / f"out{k}.npz") for k in range(2)]
    for o in outs:
        assert np.array_equal(o["words"], agg.accumulator.cpu().numpy())
        want = one.state[:, int(o["lo"]):int(o["hi"])].cpu().numpy()   # NaN-poisoned cells included: compare bits
        assert np.array_equal(o["state"].view(np.int64), want.view(np.int64))
        lo, hi = int(o["lo"]), int(o["hi"])
        assert int(o["n_streams"]) == np.unique(noise["stream"][lo:hi]).size
    one.close()


# ---------------------------------------------------------------------------------------------------- 4. nothing else moves
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_zero_noise_and_unbinding_give_the_unbound_bits(mode, cuda_device):
    """sd = 0 is not bound and gives the unbound bits; unbinding restores the adjustment kernels' and the plain
    kernels' bits."""
    import torch

    T = 140
    statics, fcols, col, adj, _, noise = _setup(n_per_col=128, M=4, T=T, seed=13, odd=False)
    M = fcols.shape[2]
    dtype = torch.float32 if mode == "f32" else torch.float64
    fc = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    kw = dict(forcing_index=col, n_forcing_cols=M, column_terms=False)
    for a in (None, adj):
        plain = _engine(statics, mode, T, forcing_adjust=a, **kw)
        want = _run_all(plain, fc, T)
        plain.close()
        zero = _engine(statics, mode, T, forcing_adjust=a, forcing_noise=dict(noise, T_air_sd=0.0, P_sd=0.0), **kw)
        assert zero.forcing_noise is None
        _assert_same_run(_run_all(zero, fc, T), want)
        zero.close()
        e = _engine(statics, mode, T, forcing_adjust=a, forcing_noise=noise, **kw)
        sd = e.state_dict()
        noisy = _run_all(e, fc, T)
        assert not _same(noisy[1], want[1])
        e.set_forcing_noise(None)
        assert e.forcing_noise is None
        e.load_state_dict(sd)
        _assert_same_run(_run_all(e, fc, T), want)
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_column_term_pass_is_not_taken_while_bound(mode, cuda_device):
    import torch

    T = 256                                                    # two launches of 128 steps, both large enough for the pass
    statics, fcols, col, _, _, noise = _setup(n_per_col=1024, M=4, T=T, seed=17)
    M = fcols.shape[2]
    f = torch.as_tensor(fcols).to(cuda_device, torch.float64).contiguous()
    e = _engine(statics, mode, T, forcing_index=col, n_forcing_cols=M, column_terms=True)
    fresh = _engine(statics, mode, T, forcing_index=col, n_forcing_cols=M, column_terms=True)
    sd = e.state_dict()
    e.run(f)
    n0 = e.column_term_launches
    assert n0 == 2
    e.load_state_dict(sd)
    e.set_forcing_noise(noise)
    e.run(f)
    assert e.column_term_launches == n0
    e.set_forcing_noise(None)
    e.load_state_dict(sd)
    got = _run_all(e, f, T)
    assert e.column_term_launches == n0 + 2
    _assert_same_run(got, _run_all(fresh, f, T))
    e.close()
    fresh.close()


# ---------------------------------------------------------------------------------------------------- 5. the example
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_ensemble_example(mode, capsys, cuda_device):
    """A one-member ensemble without noise prints the unperturbed run's numbers; a perturbed one spreads around it."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("ens", ROOT / "examples" / "ensemble_topoflow_glacier.py")
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    capsys.readouterr()
    ex.main(["--members", "1", "--T-sd", "0", "--P-sd", "0", "--mode", mode])
    lines = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("cat-")]
    assert len(lines) == len(ex.catchments())
    for ln in lines:
        for q in ("swe_end", "melt_sum"):
            m = re.search(q + r" mean=(\S+) p05=(\S+) p95=(\S+) ref=(\S+)", ln)
            assert m, ln
            mean, p05, p95, ref = (float(x) for x in m.groups())
            assert mean == p05 == p95 == ref, ln
    r = ex.run(members=16, mode=mode, verbose=False)
    spread = 0
    for row in r["catchments"].values():
        for s in row.values():
            assert s["p05"] <= s["mean"] <= s["p95"]
            spread += s["p95"] > s["p05"]
    assert spread > 0


# ---------------------------------------------------------------------------------------------------- 6. errors
@pytest.mark.gpu
def test_errors_name_the_field(cuda_device):
    import torch

    from topoflow_glacier_b200 import _lib

    statics, fcols, col, _, _, noise = _setup(n_per_col=64, M=2, T=40, seed=47, odd=False)
    N = col.size
    e = _engine(statics, "f64", 40)
    for k, v in (("T_air_sd", 5.5), ("T_air_rho", -0.1), ("P_sd", float("nan")), ("P_rho", float("inf"))):
        with pytest.raises(ValueError, match=k):
            e.set_forcing_noise(dict(noise, **{k: v}))
    with pytest.raises(ValueError, match="stream: one value per cell"):
        e.set_forcing_noise(dict(noise, stream=np.zeros(N + 1, np.int64)))
    with pytest.raises(ValueError, match="step0"):
        e.set_forcing_noise(dict(noise, step0=2**32))
    assert e.forcing_noise is None
    # the library checks too, and on error leaves nothing bound
    ids = torch.arange(4, dtype=torch.int64, device=cuda_device)
    good = torch.zeros(N, dtype=torch.int32, device=cuda_device)
    base = dict(seed=1, step0=0, T_air_sd=1.0, T_air_rho=0.5, P_sd=0.5, P_rho=0.5, n_streams=4)
    cases = [(dict(T_air_sd=float("nan")), "T_air_sd"), (dict(T_air_rho=1.0 + 2**-52), "T_air_rho"),
             (dict(P_sd=1.5000000000000002), "P_sd"), (dict(P_rho=-0.0 - 2**-1074), "P_rho"), (dict(step0=-1), "step0")]
    for over, field in cases:
        b = _lib.ForcingNoise(**dict(base, **over), stream_id=ids.data_ptr(), cell_stream=good.data_ptr())
        assert e.lib.tfg_bind_forcing_noise(e.ctx, C.byref(b), e.stream_ptr) != 0
        assert field.encode() in e.lib.tfg_last_error(), (field, e.lib.tfg_last_error())
    bad_cell = good.clone()
    bad_cell[N - 1] = 4                                          # outside [0, n_streams)
    b = _lib.ForcingNoise(**base, stream_id=ids.data_ptr(), cell_stream=bad_cell.data_ptr())
    assert e.lib.tfg_bind_forcing_noise(e.ctx, C.byref(b), e.stream_ptr) != 0
    assert b"cell_stream" in e.lib.tfg_last_error()
    neg = ids.clone()
    neg[2] = -5
    b = _lib.ForcingNoise(**base, stream_id=neg.data_ptr(), cell_stream=good.data_ptr())
    assert e.lib.tfg_bind_forcing_noise(e.ctx, C.byref(b), e.stream_ptr) != 0
    assert b"stream_id" in e.lib.tfg_last_error()
    b = _lib.ForcingNoise(**dict(base, n_streams=N - 1), stream_id=None, cell_stream=None)
    assert e.lib.tfg_bind_forcing_noise(e.ctx, C.byref(b), e.stream_ptr) != 0
    assert b"n_streams" in e.lib.tfg_last_error()
    f = torch.as_tensor(fcols[:, :, col]).to(cuda_device).contiguous()
    e.run(f[:2].contiguous())                                    # nothing bound after the failures: the plain kernel
    # a launch before step0, and steps at or past 2^32
    e.set_forcing_noise(dict(noise, step0=5))
    with pytest.raises(RuntimeError, match="step0"):
        e.run(f[2:4].contiguous())
    with pytest.raises(RuntimeError, match="step0"):
        e.forcing_noise_series(4, 2)
    with pytest.raises(RuntimeError, match=r"2\^32"):
        e.forcing_noise_series(2**32 - 1, 2)
    e.set_forcing_noise(dict(noise, step0=2**32 - 4))
    dT, _, _ = e.forcing_noise_series(2**32 - 2, 2)              # the last two steps there are
    assert bool(torch.isfinite(dT).all())
    # before statics
    ctx = C.c_void_p()
    _lib.check(e.lib.tfg_create(C.byref(ctx), 0, _lib.F64_STRICT), "tfg_create")
    b = _lib.ForcingNoise(**base, stream_id=None, cell_stream=None)
    assert e.lib.tfg_bind_forcing_noise(ctx, C.byref(b), None) != 0
    assert b"tfg_bind_static" in e.lib.tfg_last_error()
    e.lib.tfg_destroy(ctx)
    # binding statics again unbinds: the next run is the unbound one
    e.set_forcing_noise(noise)
    sd = e.state_dict()
    e._bind_static()
    e.run(f[2:].contiguous())
    plain = _engine(statics, "f64", 40)
    plain.load_state_dict(sd)
    plain.run(f[2:].contiguous())
    _assert_same_state(_state(e), _state(plain))
    e.close()
    plain.close()
