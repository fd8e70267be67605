"""Per-cell surface parameters (dust_atten, canopy_factor, cloud_factor, z0_air, em_surf): one engine running many
parameter sets equals one engine per set, bit for bit, in every mode and kernel route; the oracle agrees with per-cell
arrays; the BMI ensemble gives every member its own values and refuses members that differ in anything else."""

import ctypes as C

import numpy as np
import pytest

from helpers import ATOL, default_constants, err_report, knife_edge_mask, load_case, make_engine

KEYS = ("dust_atten", "canopy_factor", "cloud_factor", "z0_air", "em_surf")
# defaults, the cfgspace golden case's values, and two opposite corners of the schema ranges
SETS = [
    {"dust_atten": 0.08, "canopy_factor": 0.0, "cloud_factor": 0.0, "z0_air": 0.01, "em_surf": 0.985},
    {"dust_atten": 0.05, "canopy_factor": 0.2, "cloud_factor": 0.4, "z0_air": 0.02, "em_surf": 0.97},
    {"dust_atten": 0.0, "canopy_factor": 0.0, "cloud_factor": 0.0, "z0_air": 1e-4, "em_surf": 0.9},
    {"dust_atten": 0.2, "canopy_factor": 1.0, "cloud_factor": 1.0, "z0_air": 0.1, "em_surf": 1.0},
]
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


def _stack(sets, n):
    """Per-cell arrays of K parameter sets, each repeated over n cells (set s owns cells [s*n, (s+1)*n))."""
    return {k: np.repeat([s[k] for s in sets], n) for k in KEYS}


# ---------------------------------------------------------------------------------------------------- host only
def test_check_cell_params_ranges():
    import torch

    from topoflow_glacier_b200.config import CELL_PARAM_KEYS, CELL_PARAM_RANGES, check_cell_params

    assert CELL_PARAM_KEYS == KEYS
    ends = {k: np.array([lo, hi, 0.5 * (lo + hi)]) for k, (lo, hi) in CELL_PARAM_RANGES.items()}
    assert set(check_cell_params(ends)) == set(KEYS)
    check_cell_params({k: torch.as_tensor(v) for k, v in ends.items()})
    for k, (lo, hi) in CELL_PARAM_RANGES.items():
        for bad in (np.nan, np.inf, -np.inf, lo - 1e-12, np.nextafter(hi, np.inf)):
            with pytest.raises(ValueError, match=k):
                check_cell_params({k: np.array([0.5 * (lo + hi), bad])})
    with pytest.raises(ValueError, match="rho_snow"):
        check_cell_params({"rho_snow": np.array([50.0])})


@pytest.mark.parametrize("key,value", [("rho_snow", 60.0), ("T0", -0.1), ("Cp_ice", 2000.0), ("SATTERLUND", True)])
def test_ensemble_members_differing_in_other_constants_are_refused(key, value, tmp_path):
    """Raised before any CUDA call (on a machine without a GPU the engine would raise RuntimeError instead)."""
    import yaml

    from topoflow_glacier_b200 import BmiTopoflowGlacier

    with pytest.raises(ValueError, match=key):
        BmiTopoflowGlacier().initialize_ensemble([BASE_CONFIG, dict(BASE_CONFIG, **{key: value})])
    (tmp_path / "b.yaml").write_text(yaml.dump(dict(BASE_CONFIG, **{key: value})))
    (tmp_path / "a.yaml").write_text(yaml.dump(dict(BASE_CONFIG, ensemble=["b.yaml"])))
    with pytest.raises(ValueError, match=key):
        BmiTopoflowGlacier().initialize(str(tmp_path / "a.yaml"))


def test_ensemble_members_keep_their_own_surface_parameters():
    from topoflow_glacier_b200.bmi import ensemble_cell_params
    from topoflow_glacier_b200.config import TopoflowGlacierConfig

    cfgs = [TopoflowGlacierConfig.model_validate(dict(BASE_CONFIG, **s)) for s in SETS]
    got = ensemble_cell_params(cfgs)
    assert set(got) == set(KEYS)
    for k in KEYS:
        assert got[k].dtype == np.float64 and np.array_equal(got[k], [s[k] for s in SETS])


def test_bind_cell_params_is_declared():
    from pathlib import Path

    from topoflow_glacier_b200 import _lib

    assert "tfg_bind_cell_params" in _lib.PROTOTYPES
    assert [f for f, _ in _lib.CellParams._fields_] == list(KEYS)
    header = (Path(__file__).resolve().parent.parent / "include" / "tfglacier.h").read_text()
    assert "TFG_API int tfg_bind_cell_params(" in header


# ---------------------------------------------------------------------------------------------------- GPU
def _run_all(e, f, T, n_basin):
    import torch

    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.sharding import BasinAggregates

    agg = BasinAggregates(T, n_basin, device=e.device, exponents=e.agg_exponents())
    rec = e.run(f, T, record=_lib.REC_NAMES, basin_agg=agg.accumulator)
    torch.cuda.synchronize()
    return rec, e.state.clone(), e.ring.clone(), agg.decode().clone(), e.column_term_launches


def _ensemble_equals_separate_engines(statics, f, sets, mode, consts=None, forcing_index=None, n_cols=None):
    """One engine over len(sets) copies of the cells with per-cell parameters against one scalar engine per set."""

    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.engine import MeltEngine

    n, K, T = statics["lat"].size, len(sets), f.shape[0]
    base = dict(default_constants(), **(consts or {}))
    kw = dict(zones=[-8.0], mode=mode, horizon_steps=T + 1)
    big = {k: np.tile(v, K) for k, v in statics.items()}
    fmap = {} if forcing_index is None else dict(forcing_index=np.tile(forcing_index, K), n_forcing_cols=n_cols)
    fb = f if forcing_index is not None else f.repeat(1, 1, K).contiguous()
    ens = MeltEngine(big, base, "2013040100", basin_id=np.repeat(np.arange(K, dtype=np.int32), n), n_basin=K,
                     cell_params=_stack(sets, n), **fmap, **kw)
    assert ens.cell_params is not None
    got = _run_all(ens, fb, T, K)
    ens.close()
    fmap1 = {} if forcing_index is None else dict(forcing_index=forcing_index, n_forcing_cols=n_cols)
    for s, ps in enumerate(sets):
        one = MeltEngine(statics, dict(base, **ps), "2013040100", basin_id=np.zeros(n, np.int32), n_basin=1, **fmap1, **kw)
        assert one.cell_params is None
        want = _run_all(one, f, T, 1)
        one.close()
        cells = slice(s * n, (s + 1) * n)
        for name in _lib.REC_NAMES:
            assert _same(got[0][name][:, cells], want[0][name]), (s, name)
        assert _same(got[1][:, cells], want[1]), s                  # state and diagnostic integrals
        assert _same(got[2][:, cells], want[2]), s                  # snowfall window
        assert _same(got[3][:, s], want[3][:, 0]), s                # exact basin sums
        assert (got[4] > 0) == (want[4] > 0)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_ensemble_equals_separate_engines(mode, cuda_device):
    import torch

    case = load_case("rand64")
    dtype = torch.float32 if mode == "f32" else torch.float64
    f = torch.as_tensor(case["forcing"]).to(cuda_device, dtype).contiguous()
    _ensemble_equals_separate_engines(case["statics"], f, SETS, mode, consts=case["consts"])


@pytest.mark.gpu
@pytest.mark.parametrize("mode,consts", [("f64", {}), ("f64_fast", {}), ("f64", {"SATTERLUND": True})])
def test_ensemble_with_forcing_map_and_column_terms(mode, consts, cuda_device):
    """Each cell's K copies share its forcing column; the column-term pass carries the parameter-free factors."""
    import torch

    import bench

    # 768 cells per set: whole warps, so that every warp of the ensemble sums one basin as the scalar engines' warps do
    # (exact basin sums are independent of the order of the atomics, not of how cells are grouped into warps)
    n, M, T = 768, 24, 150                                          # 150 steps: two launches (128 + 22)
    statics, _ = bench.synthetic_host_sample(n, 1, seed=21)
    _, fcols = bench.synthetic_host_sample(M, T, seed=22)
    col = (np.arange(n) * M // n).astype(np.int32)
    col[::7] = np.random.default_rng(5).integers(0, M, col[::7].size)
    f = torch.as_tensor(np.ascontiguousarray(fcols)).to(cuda_device, torch.float64).contiguous()
    got = _ensemble_equals_separate_engines(statics, f, SETS, mode, consts=consts, forcing_index=col, n_cols=M)
    assert got[4] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mode,column_terms", [("f64", True), ("f64", False), ("f64_fast", True), ("f64_fast", False),
                                               ("f32", False)])
def test_uniform_parameters_equal_no_parameters(mode, column_terms, cuda_device):
    """Arrays equal to the context constants, bound through the C ABI (the engine itself would not bind them), give
    the bits of the engine without them: the per-cell factors are derived exactly as the constants are."""
    import torch

    import bench
    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.engine import MeltEngine

    N, M, T = 2000, 16, 130
    statics, _ = bench.synthetic_host_sample(N, 1, seed=31)
    _, fcols = bench.synthetic_host_sample(M, T, seed=32)
    col = (np.arange(N) * M // N).astype(np.int32)
    dtype = torch.float32 if mode == "f32" else torch.float64
    f = torch.as_tensor(np.ascontiguousarray(fcols)).to(cuda_device, dtype).contiguous()
    consts = dict(default_constants(), **SETS[1])
    out = []
    for bind in (False, True):
        e = MeltEngine(statics, consts, "2013040100", zones=[-8.0], mode=mode, horizon_steps=T + 1, forcing_index=col,
                       n_forcing_cols=M, column_terms=column_terms, basin_id=np.zeros(N, np.int32), n_basin=1)
        if bind:
            arrs = {k: torch.full((N,), consts[k], dtype=torch.float64, device=cuda_device) for k in KEYS}
            p = _lib.CellParams(**{k: arrs[k].data_ptr() for k in KEYS})
            _lib.check(e.lib.tfg_bind_cell_params(e.ctx, C.byref(p), e.stream_ptr), "tfg_bind_cell_params")
        out.append(_run_all(e, f, T, 1))
        e.close()
    for name in _lib.REC_NAMES:
        assert _same(out[0][0][name], out[1][0][name]), name
    for i in (1, 2, 3):
        assert _same(out[0][i], out[1][i])
    assert (out[0][4] > 0) == (out[1][4] > 0) == (column_terms and mode != "f32")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast"])
def test_per_cell_parameters_match_oracle(mode, cuda_device):
    """Per-cell arrays that include the ends of every range, against the NumPy oracle with the same arrays."""
    import torch

    import bench
    from oracle.np_ref import CellStatics, Constants, OracleModel
    from topoflow_glacier_b200.config import CELL_PARAM_RANGES
    from topoflow_glacier_b200.engine import MeltEngine

    N, T = 8192, 36
    statics, forcing = bench.synthetic_host_sample(N, T, seed=41)
    statics["h0_swe"][::7] *= 1e-3
    statics["h0_snow"][::7] *= 1e-3
    rng = np.random.default_rng(42)
    params = {}
    for k, (lo, hi) in CELL_PARAM_RANGES.items():
        v = rng.uniform(lo, hi, N)
        v[rng.integers(0, 4, N) == 0] = lo
        v[rng.integers(0, 4, N) == 0] = hi
        params[k] = v
    ora = OracleModel(CellStatics(**statics, tz=[-8.0]), Constants(**params), "2013040100", strict_pow=False)
    keys = ["h_swe", "h_iwe", "h_snow", "h_ice", "SM", "IM", "M_total", "RH", "Q_sum", "Qn_SW", "Qn_LW", "Qh", "Qe",
            "albedo", "Eccs", "Ecci", "T_surf"]
    want = {k: np.empty((T, N)) for k in keys}
    for t in range(T):
        d = ora.step(*forcing[t])
        for k in keys:
            want[k][t] = d[k]
    eng = MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode=mode, horizon_steps=T + 1,
                     cell_params=params)
    got = {k: v.cpu().numpy() for k, v in eng.run(torch.as_tensor(forcing).to(cuda_device), record=keys).items()}
    eng.close()
    mask = knife_edge_mask(got, want)
    # the log-law singularity at h_snow = z - z0_air moves with the cell's z0_air (see test_large_random_sample_with_knife_edges)
    hs = np.vstack([statics["h0_snow"][None, :], want["h_snow"][:-1]])
    arg = (10.0 - hs) / params["z0_air"]
    with np.errstate(divide="ignore", invalid="ignore"):
        cond = np.where(arg > 0.01, 2.0 * hs / (np.abs(10.0 - hs) * np.abs(np.log(np.maximum(arg, 1e-300)))), 0.0)
    singular = np.maximum.accumulate(np.nan_to_num(cond, posinf=np.inf) > 500.0, axis=0)
    mask |= singular
    melted = int(((want["h_swe"][0] > 0) & (want["h_swe"][-1] == 0)).sum())
    knife = int(mask[-1].sum() - singular[-1].sum())
    # z0_air up to 0.1 m widens the ill-conditioned band below the singularity (a smaller log in the denominator)
    assert knife <= max(5, 0.15 * melted) and singular[-1].sum() <= 0.04 * N, (knife, melted, singular[-1].sum())
    bad = []
    for k in keys:
        ok, ratio, dabs, drel = err_report(got[k][~mask], want[k][~mask], ATOL[k])
        if not ok:
            bad.append((k, ratio, dabs, drel))
    assert not bad, bad


@pytest.mark.gpu
def test_bmi_yaml_ensemble_per_step_equals_fused_and_single_members(tmp_path, cuda_device):
    """An `ensemble:` yaml whose members differ in the five parameters, advanced by update() step by step, equals the
    same ensemble advanced by update_until in one launch, and every member equals a model of its own yaml alone."""
    import torch
    import yaml

    from topoflow_glacier_b200 import BmiTopoflowGlacier

    case = load_case("cats288")
    K, T = len(SETS), 30
    names = []
    for i, s in enumerate(SETS):
        c = dict(BASE_CONFIG, **s, **{k: float(v[i]) for k, v in case["statics"].items()})
        (tmp_path / f"m{i}.yaml").write_text(yaml.dump(c))
        names.append(f"m{i}.yaml")
    head = yaml.safe_load((tmp_path / names[0]).read_text())
    (tmp_path / "ens.yaml").write_text(yaml.dump(dict(head, ensemble=names[1:])))
    forcing = case["forcing"][:T, :, :K]
    set_order = ("atmosphere_water__liquid_equivalent_precipitation_rate", "land_surface_air__temperature",
                 "land_surface_air__pressure", "atmosphere_air_water~vapor__relative_saturation", "wind_speed_UV")
    step = BmiTopoflowGlacier()
    step.initialize(str(tmp_path / "ens.yaml"))
    assert step._engine.cell_params is not None
    for t in range(T):
        for name, v in zip(set_order, forcing[t]):
            step.set_value(name, np.ascontiguousarray(v))
        step.update()
    fused = BmiTopoflowGlacier()
    fused.initialize_ensemble([str(tmp_path / n) for n in names])
    fused.load_forcing(torch.as_tensor(np.ascontiguousarray(forcing)).cuda())
    fused.update_until(T * 3600.0)
    torch.cuda.synchronize()
    assert _same(step._engine.state, fused._engine.state)
    assert _same(step._engine.ring, fused._engine.ring)
    for i in range(K):
        one = BmiTopoflowGlacier()
        one.initialize(str(tmp_path / names[i]))
        assert one._engine.cell_params is None
        one.load_forcing(torch.as_tensor(np.ascontiguousarray(forcing[:, :, i:i + 1])).cuda())
        one.update_until(T * 3600.0)
        torch.cuda.synchronize()
        assert _same(one._engine.state[:, 0], fused._engine.state[:, i]), i
        one.finalize()
    step.finalize()
    fused.finalize()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_rebinding_between_launches_equals_checkpoint_handover(mode, cuda_device):
    """set_cell_params(p2) after t1 steps with p1 == a scalar engine with p1 for t1 steps, checkpointed into a scalar
    engine with p2 for the rest (the calibration loop: run, score, new parameters, run again)."""
    import torch

    case = load_case("rand64")
    T, t1 = case["forcing"].shape[0], 20
    N = case["N"]
    dtype = torch.float32 if mode == "f32" else torch.float64
    f = torch.as_tensor(case["forcing"]).to(cuda_device, dtype).contiguous()
    p1, p2 = SETS[2], SETS[3]
    e = make_engine(case, mode=mode, cell_params={k: np.full(N, v) for k, v in p1.items()})
    assert e.cell_params is not None
    e.run(f[:t1].contiguous())
    e.set_cell_params({k: np.full(N, v) for k, v in p2.items()})
    e.run(f[t1:].contiguous())
    a = make_engine(case, mode=mode, consts=p1)
    a.run(f[:t1].contiguous())
    b = make_engine(case, mode=mode, consts=p2)
    b.load_state_dict(a.state_dict())
    b.run(f[t1:].contiguous())
    torch.cuda.synchronize()
    assert _same(e.state, b.state) and _same(e.ring, b.ring)
    e.set_cell_params(None)                                         # unbinding restores the constants
    assert e.cell_params is None
    for x in (e, a, b):
        x.close()


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_sharded_engine_with_cell_params_two_ranks_equal_one(tmp_path, cuda_device):
    import os
    import subprocess
    import sys

    import torch

    import bench
    from topoflow_glacier_b200.engine import MeltEngine
    from topoflow_glacier_b200.sharding import BasinAggregates

    N, T, NB = 5000, 14, 13
    statics, forcing = bench.synthetic_host_sample(N, T, seed=12)
    basin = np.random.default_rng(4).integers(0, NB, N).astype(np.int32)
    rng = np.random.default_rng(6)
    from topoflow_glacier_b200.config import CELL_PARAM_RANGES

    params = {k: rng.uniform(lo, hi, N) for k, (lo, hi) in CELL_PARAM_RANGES.items()}
    np.savez(tmp_path / "in.npz", forcing=forcing, basin=basin, **{f"s_{k}": v for k, v in statics.items()},
             **{f"p_{k}": v for k, v in params.items()})
    one = MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", basin_id=basin,
                     n_basin=NB, horizon_steps=T + 1, cell_params=params)
    agg = BasinAggregates(T, NB, device=cuda_device, exponents=one.agg_exponents())
    one.run(torch.as_tensor(forcing).cuda(), basin_agg=agg.zero())
    agg.reduce()
    torch.cuda.synchronize()
    root = str(__import__("pathlib").Path(__file__).resolve().parent.parent)
    script = tmp_path / "w.py"
    script.write_text(f'''
import os, sys
sys.path.insert(0, {root!r})
os.environ["NGEN_EWTS_LOGGING"] = "DISABLED"
import numpy as np, torch, torch.distributed as dist
from topoflow_glacier_b200.config import default_constants
from topoflow_glacier_b200.sharding import ShardedMeltEngine
dist.init_process_group("gloo")
rank = dist.get_rank()
z = np.load({str(tmp_path / "in.npz")!r})
statics = {{k[2:]: z[k] for k in z.files if k.startswith("s_")}}
params = {{k[2:]: z[k] for k in z.files if k.startswith("p_")}}
f = torch.as_tensor(z["forcing"]).cuda()
T = f.shape[0]
sh = ShardedMeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", basin_id=z["basin"],
                       n_basin={NB}, horizon_steps=T + 1, device=0, cell_params=params)
_, g = sh.run(sh.local(f).contiguous())
lo, hi = sh.bounds
np.savez({str(tmp_path)!r} + f"/out{{rank}}.npz", agg=g.cpu().numpy(), state=sh.state.cpu().numpy(), lo=lo, hi=hi)
dist.destroy_process_group()
sys.stdout.write("rank %d ok\\n" % rank)
''')
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29617", str(script)],
                       capture_output=True, text=True, env=env, timeout=560)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    outs = [np.load(tmp_path / f"out{k}.npz") for k in range(2)]
    want = agg.buffer.cpu().numpy()
    for o in outs:
        assert np.array_equal(o["agg"], want)
        assert np.array_equal(o["state"], one.state[:, int(o["lo"]):int(o["hi"])].cpu().numpy())
    one.close()


@pytest.mark.gpu
def test_bind_errors(cuda_device):
    import torch

    case = load_case("rand64")
    N = case["N"]
    e = make_engine(case, mode="f64")
    with pytest.raises(ValueError, match="z0_air"):
        e.set_cell_params({"z0_air": np.full(N, 0.5)})
    with pytest.raises(ValueError, match="one value per cell"):
        e.set_cell_params({"dust_atten": np.full(N + 1, 0.1)})
    # the library checks on the device too: a NaN that reaches it directly is refused and leaves nothing bound
    from topoflow_glacier_b200 import _lib

    bad = torch.full((N,), float("nan"), dtype=torch.float64, device=cuda_device)
    p = _lib.CellParams(em_surf=bad.data_ptr())
    assert e.lib.tfg_bind_cell_params(e.ctx, C.byref(p), e.stream_ptr) != 0
    assert b"em_surf" in e.lib.tfg_last_error()
    e.close()
