"""Per-cell forcing adjustments (T_air_offset, P_multiplier): a run with adjustments bound equals, bit for bit, a run
whose per-cell forcing was adjusted in advance with the same two IEEE operations -- in every mode, with and without
per-cell parameters and an objective, across launch splits, the per-step path, rebinding and sharding; identity values
give the unbound bits; the column-term pass is not taken while adjustments are bound."""

import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from helpers import default_constants

ROOT = Path(__file__).resolve().parent.parent
KEYS = ("T_air_offset", "P_multiplier")
BASE_CONFIG = {
    "site_prefix": "cat-x", "forcing_file": "-", "dt": 1, "start_time": "2013032000", "end_time": "2013033100",
    "da": 11.4, "slope": 88.6, "aspect": 242.9, "lon": -121.8, "lat": 46.8, "elev": 2446.4, "h0_snow": 5.0,
    "h0_ice": 2.0, "h0_swe": 0.25, "h0_iwe": 1.834, "T_rain_snow": 0.0, "utc_offset_hours": -8.0,
}


def _bits(x):
    import torch

    x = x.contiguous()
    return x.view(torch.int32 if x.element_size() == 4 else torch.int64)


def _same(a, b):
    """Bit for bit (NaN patterns included)."""
    import torch

    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


# ---------------------------------------------------------------------------------------------------- host only
def test_header_declares_the_binding_and_ctypes_matches_it():
    from topoflow_glacier_b200 import _lib

    header = (ROOT / "include" / "tfglacier.h").read_text()
    assert "TFG_API int tfg_bind_forcing_adjust(tfg_ctx* ctx, const tfg_forcing_adjust* a, void* stream);" in header
    body = re.search(r"typedef struct tfg_forcing_adjust \{(.*?)\} tfg_forcing_adjust;", header, re.S).group(1)
    fields = re.findall(r"const double\* (\w+);", body)
    assert fields == list(KEYS)
    assert [f for f, _ in _lib.ForcingAdjust._fields_] == fields
    assert C.sizeof(_lib.ForcingAdjust) == len(fields) * C.sizeof(C.c_void_p)
    res, args = _lib.PROTOTYPES["tfg_bind_forcing_adjust"]
    assert res is C.c_int and args == [C.c_void_p, C.POINTER(_lib.ForcingAdjust), C.c_void_p]


def test_check_forcing_adjust_ranges():
    import torch

    from topoflow_glacier_b200.config import (FORCING_ADJUST_IDENTITY, FORCING_ADJUST_KEYS, FORCING_ADJUST_RANGES,
                                              check_forcing_adjust)

    assert FORCING_ADJUST_KEYS == KEYS
    assert FORCING_ADJUST_RANGES == {"T_air_offset": (-30.0, 30.0), "P_multiplier": (0.0, 10.0)}
    assert FORCING_ADJUST_IDENTITY == {"T_air_offset": 0.0, "P_multiplier": 1.0}
    ends = {k: np.array([lo, hi, 0.5 * (lo + hi)]) for k, (lo, hi) in FORCING_ADJUST_RANGES.items()}
    assert set(check_forcing_adjust(ends)) == set(KEYS)
    check_forcing_adjust({k: torch.as_tensor(v) for k, v in ends.items()})
    for k, (lo, hi) in FORCING_ADJUST_RANGES.items():
        for bad in (np.nan, np.inf, -np.inf, np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)):
            with pytest.raises(ValueError, match=k):
                check_forcing_adjust({k: np.array([0.5 * (lo + hi), bad])})
    with pytest.raises(ValueError, match="P_factor"):
        check_forcing_adjust({"P_factor": np.array([1.0])})


def test_yaml_keys_parse_and_legacy_p_factor_stays_ignored():
    from pydantic import ValidationError

    from topoflow_glacier_b200.config import TopoflowGlacierConfig

    c = TopoflowGlacierConfig.model_validate(dict(BASE_CONFIG, T_air_offset=-9.75, P_multiplier=1.5))
    assert (c.T_air_offset, c.P_multiplier) == (-9.75, 1.5)
    d = TopoflowGlacierConfig.model_validate(BASE_CONFIG)
    assert (d.T_air_offset, d.P_multiplier) == (0.0, 1.0)
    legacy = TopoflowGlacierConfig.model_validate(dict(BASE_CONFIG, P_factor=3.0))
    assert legacy.P_factor == 3.0 and (legacy.T_air_offset, legacy.P_multiplier) == (0.0, 1.0)
    for bad in ({"T_air_offset": 30.5}, {"T_air_offset": float("nan")}, {"P_multiplier": -0.1}, {"P_multiplier": 11.0}):
        with pytest.raises(ValidationError):
            TopoflowGlacierConfig.model_validate(dict(BASE_CONFIG, **bad))


def test_ensemble_members_may_differ_in_the_adjustments():
    from topoflow_glacier_b200.bmi import ensemble_cell_params
    from topoflow_glacier_b200.config import TopoflowGlacierConfig

    cfgs = [TopoflowGlacierConfig.model_validate(dict(BASE_CONFIG, T_air_offset=o, P_multiplier=m))
            for o, m in ((0.0, 1.0), (-6.5, 2.0), (3.0, 0.0))]
    assert set(ensemble_cell_params(cfgs)) == {"dust_atten", "canopy_factor", "cloud_factor", "z0_air", "em_surf"}


# ---------------------------------------------------------------------------------------------------- GPU
def _setup(n_per_col=256, M=6, T=300, seed=91, odd=True):
    """M catchment columns, n_per_col cells each on a forcing map, per-cell adjustments that include both range ends;
    with ``odd`` (T >= 100), NaN rows and forcings that the adjustments push out of the fast mode's lean ranges."""
    import bench
    from topoflow_glacier_b200.config import CELL_PARAM_RANGES

    N = n_per_col * M
    statics, _ = bench.synthetic_host_sample(N, 1, seed=seed)
    _, fcols = bench.synthetic_host_sample(M, T, seed=seed + 1)
    fcols = fcols.copy()
    if odd and T >= 100:
        fcols[40, :, 1 % M] = np.nan                # a whole NaN row of one column
        fcols[41, 1, 2 % M] = np.nan                # a missing temperature
        fcols[60:64, 1, 3 % M] = 75.0               # T_air within the lean range, +30 K takes it past 90 degC
        fcols[80:84, 0, 4 % M] = 2.0                # P = 2 m/h, * 10 takes it past 10 m/h
        fcols[90, 1, 0] = -85.0                     # -30 K takes it past -90 degC
    col = np.repeat(np.arange(M, dtype=np.int32), n_per_col)
    rng = np.random.default_rng(seed + 2)
    off = rng.uniform(-30.0, 30.0, N)
    mul = rng.uniform(0.0, 10.0, N)
    for v, lo, hi in ((off, -30.0, 30.0), (mul, 0.0, 10.0)):
        v[0::7] = lo
        v[3::7] = hi
    off[5::11], mul[5::11] = 0.0, 1.0              # identity cells among the others
    params = {k: rng.uniform(lo, hi, N) for k, (lo, hi) in CELL_PARAM_RANGES.items()}
    return statics, np.ascontiguousarray(fcols), col, {"T_air_offset": off, "P_multiplier": mul}, params


def _adjusted_per_cell(f_cols, col, adj, dtype):
    """The per-cell forcing replicated from the columns and adjusted with torch in the engine's dtype."""
    import torch

    f = f_cols[:, :, torch.as_tensor(col, dtype=torch.int64, device=f_cols.device)].clone()
    off = torch.as_tensor(adj["T_air_offset"]).to(f.device).to(dtype)
    mul = torch.as_tensor(adj["P_multiplier"]).to(f.device).to(dtype)
    f[:, 1] = f[:, 1] + off
    f[:, 0] = f[:, 0] * mul
    return f.contiguous()


def _run_all(e, f, T, n_basin, record=True):
    import torch

    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.sharding import BasinAggregates

    agg = BasinAggregates(T, n_basin, device=e.device, exponents=e.agg_exponents())
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


def _engine(statics, mode, T, params=None, **kw):
    from topoflow_glacier_b200.engine import MeltEngine

    N = statics["lat"].size
    basin = kw.pop("basin_id", (np.arange(N) // 384).astype(np.int32))
    return MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode=mode, horizon_steps=T + 1,
                      basin_id=basin, n_basin=int(basin.max()) + 1, cell_params=params, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
@pytest.mark.parametrize("with_params,with_obj", [(False, False), (True, False), (False, True), (True, True)])
def test_adjusted_map_equals_adjusted_per_cell_forcing(mode, with_params, with_obj, cuda_device):
    """The central equivalence: 300 steps (three launches) on a forcing map with adjustments bound against per-cell
    forcing adjusted in advance, bit for bit; with an objective, its sums also equal the host loop."""
    import torch

    from topoflow_glacier_b200.objective import series_sums

    T = 300
    statics, fcols, col, adj, params = _setup(T=T)
    N, M = col.size, fcols.shape[2]
    dtype = torch.float32 if mode == "f32" else torch.float64
    fc = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    fcell = _adjusted_per_cell(fc, col, adj, dtype)
    obs = np.random.default_rng(7).uniform(0.0, 1.0, (250, M))
    obs[::9] = np.nan
    out = []
    for route in ("map", "cell"):
        kw = dict(forcing_index=col, n_forcing_cols=M, forcing_adjust=adj) if route == "map" else {}
        e = _engine(statics, mode, T, params if with_params else None, **kw)
        assert (e.forcing_adjust is not None) == (route == "map")
        if with_obj:
            e.set_objective("h_swe", obs, obs_step0=20, obs_index=col)
        got = _run_all(e, fc if route == "map" else fcell, T, e.n_basin)
        assert e.column_term_launches == 0
        sums = torch.stack(e.objective_sums()).clone() if with_obj else None
        out.append((got, sums))
        e.close()
    _assert_same_run(out[0][0], out[1][0])
    if with_obj:
        assert _same(out[0][1], out[1][1])
        o_cell = np.full((T, N), np.nan)
        o_cell[20:270] = obs[:, col]
        want, _ = series_sums(out[0][0][0]["h_swe"].double().cpu(), o_cell)
        assert _same(out[0][1].cpu(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_identity_adjustments_give_the_unbound_bits(mode, cuda_device):
    """Identity arrays are not bound; bound explicitly through the C ABI on some cells, those cells get the unbound bits."""
    import torch

    from topoflow_glacier_b200 import _lib

    T = 140
    statics, fcols, col, adj, _ = _setup(n_per_col=128, M=4, T=T, seed=13, odd=False)   # no NaN: payloads aside
    N, M = col.size, fcols.shape[2]
    dtype = torch.float32 if mode == "f32" else torch.float64
    fc = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    kw = dict(forcing_index=col, n_forcing_cols=M, column_terms=False)
    plain = _engine(statics, mode, T, **kw)
    want = _run_all(plain, fc, T, plain.n_basin)
    plain.close()
    ident = _engine(statics, mode, T, forcing_adjust={"T_air_offset": np.zeros(N), "P_multiplier": np.ones(N)}, **kw)
    assert ident.forcing_adjust is None
    _assert_same_run(_run_all(ident, fc, T, ident.n_basin), want)
    ident.close()
    e = _engine(statics, mode, T, **kw)
    some = np.zeros(N, dtype=bool)
    some[::3] = True                                           # cells that keep the identity, bound explicitly
    off = torch.as_tensor(np.where(some, 0.0, adj["T_air_offset"])).to(cuda_device)
    mul = torch.as_tensor(np.where(some, 1.0, adj["P_multiplier"])).to(cuda_device)
    a = _lib.ForcingAdjust(T_air_offset=off.data_ptr(), P_multiplier=mul.data_ptr())
    _lib.check(e.lib.tfg_bind_forcing_adjust(e.ctx, C.byref(a), e.stream_ptr), "tfg_bind_forcing_adjust")
    got = _run_all(e, fc, T, e.n_basin)
    e.close()
    idx = torch.as_tensor(np.flatnonzero(some), device=cuda_device)
    for name in want[0]:
        assert _same(got[0][name][:, idx], want[0][name][:, idx]), name
    for i in (1, 2, 3):
        assert _same(got[i][:, idx], want[i][:, idx]), i
    assert not _same(got[1], want[1])                           # the other cells did change


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_column_term_pass_is_not_taken_while_bound(mode, cuda_device):
    import torch

    T = 256                                                    # two launches of 128 steps, both large enough for the pass
    statics, fcols, col, adj, _ = _setup(n_per_col=1024, M=4, T=T, seed=17)
    M = fcols.shape[2]
    f = torch.as_tensor(fcols).to(cuda_device, torch.float64).contiguous()
    e = _engine(statics, mode, T, forcing_index=col, n_forcing_cols=M, column_terms=True)
    fresh = _engine(statics, mode, T, forcing_index=col, n_forcing_cols=M, column_terms=True)
    sd = e.state_dict()
    e.run(f)
    n0 = e.column_term_launches
    assert n0 == 2
    e.set_forcing_adjust(adj)
    e.load_state_dict(sd)
    e.run(f)
    assert e.column_term_launches == n0
    e.set_forcing_adjust(None)
    assert e.forcing_adjust is None
    e.load_state_dict(sd)
    got = _run_all(e, f, T, e.n_basin)
    assert e.column_term_launches == n0 + 2
    _assert_same_run(got, _run_all(fresh, f, T, fresh.n_basin))
    e.close()
    fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_per_step_paths_equal_the_fused_run(mode, cuda_device):
    """step() from the input block, and BMI update() after set_value, equal one fused run; the BMI inputs keep what the
    caller set."""
    import torch

    from topoflow_glacier_b200 import BmiTopoflowGlacier

    T = 30
    statics, fcols, col, adj, _ = _setup(n_per_col=64, M=3, T=T, seed=23)
    N, M = col.size, fcols.shape[2]
    dtype = torch.float32 if mode == "f32" else torch.float64
    fc = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    kw = dict(forcing_index=col, n_forcing_cols=M, forcing_adjust=adj)
    fused = _engine(statics, mode, T, basin_id=np.zeros(N, np.int32), **kw)
    fused.run(fc)
    steps = _engine(statics, mode, T, basin_id=np.zeros(N, np.int32), **kw)
    for t in range(T):
        steps.inputs[:5].copy_(fc[t])
        steps.step()
    torch.cuda.synchronize()
    assert _same(steps.state, fused.state) and _same(steps.ring, fused.ring)
    bmi = BmiTopoflowGlacier()
    cells = dict(statics, **adj)
    bmi.initialize_cells(dict(BASE_CONFIG, start_time="2013040100", utc_offset_hours=-8.0, precision=mode), cells,
                         forcing_index=col, n_forcing_cols=M)
    assert bmi._engine.forcing_adjust is not None
    names = ("atmosphere_water__liquid_equivalent_precipitation_rate", "land_surface_air__temperature",
             "land_surface_air__pressure", "atmosphere_air_water~vapor__relative_saturation", "wind_speed_UV")
    for t in range(T):
        for name, v in zip(names, fcols[t]):
            bmi.set_value(name, np.ascontiguousarray(v))
        bmi.update()
    torch.cuda.synchronize()
    assert _same(bmi._engine.state, fused.state) and _same(bmi._engine.ring, fused.ring)
    got = bmi.get_value("land_surface_air__temperature", np.empty(M))
    assert np.array_equal(got, fcols[T - 1, 1].astype(np.float32 if mode == "f32" else np.float64))
    bmi.finalize()
    fused.close()
    steps.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_rebinding_between_launches_equals_checkpoint_handover(mode, cuda_device):
    import torch

    T, t1 = 160, 70
    statics, fcols, col, adj, _ = _setup(n_per_col=128, M=4, T=T, seed=29)
    M = fcols.shape[2]
    adj2 = {"T_air_offset": -0.5 * adj["T_air_offset"], "P_multiplier": np.clip(10.0 - adj["P_multiplier"], 0, 10)}
    dtype = torch.float32 if mode == "f32" else torch.float64
    f = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    kw = dict(forcing_index=col, n_forcing_cols=M)
    e = _engine(statics, mode, T, forcing_adjust=adj, **kw)
    e.run(f[:t1].contiguous())
    e.set_forcing_adjust(adj2)
    e.run(f[t1:].contiguous())
    a = _engine(statics, mode, T, forcing_adjust=adj, **kw)
    a.run(f[:t1].contiguous())
    sd = a.state_dict()
    assert not any("adjust" in k for k in sd)                   # bindings, not state
    b = _engine(statics, mode, T, forcing_adjust=adj2, **kw)
    b.load_state_dict(sd)
    b.run(f[t1:].contiguous())
    torch.cuda.synchronize()
    assert _same(e.state, b.state) and _same(e.ring, b.ring)
    for x in (e, a, b):
        x.close()


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_sharded_engine_two_ranks_equal_one(tmp_path, cuda_device):
    import os
    import subprocess
    import sys

    import torch

    from topoflow_glacier_b200.engine import MeltEngine
    from topoflow_glacier_b200.sharding import BasinAggregates

    T, NB = 20, 7
    statics, fcols, col, adj, _ = _setup(n_per_col=640, M=8, T=T, seed=37)
    N, M = col.size, fcols.shape[2]
    basin = np.random.default_rng(4).integers(0, NB, N).astype(np.int32)
    np.savez(tmp_path / "in.npz", forcing=fcols, basin=basin, col=col, **{f"s_{k}": v for k, v in statics.items()},
             **{f"a_{k}": v for k, v in adj.items()})
    one = MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", basin_id=basin,
                     n_basin=NB, horizon_steps=T + 1, forcing_index=col, n_forcing_cols=M, forcing_adjust=adj)
    agg = BasinAggregates(T, NB, device=cuda_device, exponents=one.agg_exponents())
    one.run(torch.as_tensor(fcols).cuda(), basin_agg=agg.zero())
    agg.reduce()
    torch.cuda.synchronize()
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
adj = {{k[2:]: z[k] for k in z.files if k.startswith("a_")}}
f = torch.as_tensor(z["forcing"]).cuda()
T = f.shape[0]
sh = ShardedMeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", basin_id=z["basin"],
                       n_basin={NB}, horizon_steps=T + 1, device=0, forcing_index=z["col"], n_forcing_cols={M},
                       forcing_adjust=adj)
_, g = sh.run(f)
lo, hi = sh.bounds
np.savez({str(tmp_path)!r} + f"/out{{rank}}.npz", agg=g.cpu().numpy(), words=sh.aggregates(T).accumulator.cpu().numpy(),
         state=sh.state.cpu().numpy(), lo=lo, hi=hi)
dist.destroy_process_group()
sys.stdout.write("rank %d ok\\n" % rank)
''')
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29631", str(script)],
                       capture_output=True, text=True, env=env, timeout=560)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    outs = [np.load(tmp_path / f"out{k}.npz") for k in range(2)]
    for o in outs:
        assert np.array_equal(o["agg"], agg.buffer.cpu().numpy())
        assert np.array_equal(o["words"], agg.accumulator.cpu().numpy())
        assert np.array_equal(o["state"], one.state[:, int(o["lo"]):int(o["hi"])].cpu().numpy())
    one.close()


@pytest.mark.gpu
def test_bmi_yaml_ensemble_equals_initialize_cells(tmp_path, cuda_device):
    """Members carrying the two keys equal initialize_cells with the same arrays; P_factor: 3.0 changes nothing."""
    import torch
    import yaml

    from topoflow_glacier_b200 import BmiTopoflowGlacier
    from topoflow_glacier_b200.statics import CELL_KEYS

    T = 48
    members = [(0.0, 1.0), (-9.75, 2.5), (6.5, 0.0), (-30.0, 10.0), (30.0, 0.5)]
    K = len(members)
    statics, forcing = __import__("bench").synthetic_host_sample(K, T, seed=43)
    names = []
    for i, (o, m) in enumerate(members):
        c = dict(BASE_CONFIG, T_air_offset=o, P_multiplier=m, **{k: float(v[i]) for k, v in statics.items()})
        (tmp_path / f"m{i}.yaml").write_text(yaml.dump(c))
        names.append(f"m{i}.yaml")
    head = yaml.safe_load((tmp_path / names[0]).read_text())
    (tmp_path / "ens.yaml").write_text(yaml.dump(dict(head, ensemble=names[1:])))
    f = torch.as_tensor(forcing).cuda()
    ens = BmiTopoflowGlacier()
    ens.initialize(str(tmp_path / "ens.yaml"))
    assert ens._engine.forcing_adjust is not None
    ens.load_forcing(f)
    ens.update_until(T * 3600.0)
    cells = BmiTopoflowGlacier()
    arrays = {k: np.asarray(statics[k], dtype=np.float64) for k in CELL_KEYS}
    arrays.update(T_air_offset=np.array([o for o, _ in members]), P_multiplier=np.array([m for _, m in members]))
    cells.initialize_cells(tmp_path / names[0], arrays, zones=[-8.0])
    cells.load_forcing(f)
    cells.update_until(T * 3600.0)
    torch.cuda.synchronize()
    assert _same(ens._engine.state, cells._engine.state) and _same(ens._engine.ring, cells._engine.ring)
    out = []
    for extra in ({}, {"P_factor": 3.0}):
        (tmp_path / "one.yaml").write_text(yaml.dump(dict(BASE_CONFIG, **extra)))
        b = BmiTopoflowGlacier()
        b.initialize(str(tmp_path / "one.yaml"))
        assert b._engine.forcing_adjust is None
        b.load_forcing(f[:, :, :1].contiguous())
        b.update_until(T * 3600.0)
        torch.cuda.synchronize()
        out.append((b._engine.state.clone(), b._engine.ring.clone()))
        b.finalize()
    assert _same(out[0][0], out[1][0]) and _same(out[0][1], out[1][1])
    ens.finalize()
    cells.finalize()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_twin_experiment_with_forcing_params(mode, cuda_device):
    import importlib.util

    spec = importlib.util.spec_from_file_location("calib", ROOT / "examples" / "calibrate_topoflow_glacier.py")
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    r = ex.run(sets=96, mode=mode, quantity="M_total", seed=2, verbose=False, forcing_params=True)
    K = r["sets"]
    assert not r["column_terms"]
    for c, b in enumerate(r["best"]):
        ti = c * K + r["truth_index"][c]
        assert set(KEYS) <= set(b["params"]) and set(KEYS) <= set(r["truth"][c])
        assert -3.0 <= r["truth"][c]["T_air_offset"] <= 3.0 and 0.5 <= r["truth"][c]["P_multiplier"] <= 2.0
        assert r["scores"]["rmse"][ti] == 0.0 and r["scores"]["nse"][ti] == 1.0, (c, r["scores"]["nse"][ti])
        assert b["index"] == r["truth_index"][c], (c, b)


@pytest.mark.gpu
def test_bind_errors_name_the_field(cuda_device):
    import torch

    from topoflow_glacier_b200 import _lib

    statics, _, col, adj, _ = _setup(n_per_col=64, M=2, T=2, seed=47, odd=False)
    N = col.size
    e = _engine(statics, "f64", 2)
    with pytest.raises(ValueError, match="T_air_offset"):
        e.set_forcing_adjust({"T_air_offset": np.full(N, np.nan)})
    with pytest.raises(ValueError, match="P_multiplier"):
        e.set_forcing_adjust({"P_multiplier": np.full(N, 10.5)})
    with pytest.raises(ValueError, match="T_air_offset: one value per cell"):
        e.set_forcing_adjust({"T_air_offset": np.zeros(N + 1) + 1.0})
    # the library checks on the device too: values that reach it directly are refused and leave nothing bound
    for field, value in (("T_air_offset", float("nan")), ("T_air_offset", -30.5), ("P_multiplier", float("inf")),
                         ("P_multiplier", -1e-300)):
        bad = torch.full((N,), value, dtype=torch.float64, device=cuda_device)
        a = _lib.ForcingAdjust(**{field: bad.data_ptr()})
        assert e.lib.tfg_bind_forcing_adjust(e.ctx, C.byref(a), e.stream_ptr) != 0
        msg = e.lib.tfg_last_error()
        assert field.encode() in msg and [k for k in KEYS if k.encode() in msg] == [field], msg
    # before statics
    ctx = C.c_void_p()
    _lib.check(e.lib.tfg_create(C.byref(ctx), 0, _lib.F64_STRICT), "tfg_create")
    ok = torch.zeros(N, dtype=torch.float64, device=cuda_device)
    a = _lib.ForcingAdjust(T_air_offset=ok.data_ptr())
    assert e.lib.tfg_bind_forcing_adjust(ctx, C.byref(a), None) != 0
    assert b"tfg_bind_static" in e.lib.tfg_last_error()
    e.lib.tfg_destroy(ctx)
    # binding statics again unbinds: the next run is the unbound one
    f = torch.as_tensor(_setup(n_per_col=64, M=2, T=40, seed=47, odd=False)[1][:, :, col]).to(cuda_device).contiguous()
    e.set_forcing_adjust(adj)
    sd = e.state_dict()
    e._bind_static()
    e.run(f)
    plain = _engine(statics, "f64", 40)
    plain.load_state_dict(sd)
    plain.run(f)
    torch.cuda.synchronize()
    assert _same(e.state, plain.state)
    e.close()
    plain.close()
