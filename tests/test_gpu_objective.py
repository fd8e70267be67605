"""The objective (tfg_bind_objective, MeltEngine.set_objective): per-cell sums of a BMI output against observations,
accumulated inside the melt kernel.  The sums equal a host float64 loop over the recorded series bit for bit in every
mode and kernel route, change nothing else, do not depend on the launch split or the sharding, and give the twin
experiment's truth NSE = 1 exactly; the scores follow one definition (objective.py) for sums and series alike."""

import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from helpers import default_constants

ROOT = Path(__file__).resolve().parent.parent


def _np_scores(s, o):
    """Direct NumPy statement of each metric for one series pair (NaN observations dropped)."""
    m = np.isfinite(o)
    s, o = s[m], o[m]
    nse = 1.0 - np.sum((s - o) ** 2) / np.sum((o - o.mean()) ** 2)
    r = np.corrcoef(s, o)[0, 1]
    alpha, beta = s.std() / o.std(), s.mean() / o.mean()
    kge = 1.0 - np.sqrt((r - 1) ** 2 + (alpha - 1) ** 2 + (beta - 1) ** 2)
    return {"n": m.sum(), "nse": nse, "kge": kge, "r": r, "alpha": alpha, "beta": beta,
            "rmse": np.sqrt(np.mean((s - o) ** 2)), "bias": np.mean(s - o)}


# ---------------------------------------------------------------------------------------------------- host only
def test_skill_scores_equal_series_scores_and_numpy():
    from topoflow_glacier_b200.objective import SCORE_NAMES, series_scores, series_sums, skill_scores

    rng = np.random.default_rng(3)
    T, M = 240, 9
    o = 0.4 + rng.gamma(2.0, 0.1, (T, M)) + np.sin(np.arange(T) / 17.0)[:, None]
    s = o * rng.uniform(0.7, 1.3, M) + rng.normal(0, 0.05, (T, M))
    o[rng.uniform(size=(T, M)) < 0.3] = np.nan
    o[:20] = np.nan                                                  # spin-up
    o[::24, 2] = np.inf                                              # non-finite = not observed, of either kind
    acc, mom = series_sums(s, o)
    a = skill_scores(acc, mom)
    b = series_scores(s, o)
    assert set(a) == set(SCORE_NAMES)
    for k in SCORE_NAMES:
        assert np.array_equal(a[k].numpy(), b[k].numpy()), k
    for j in range(M):
        want = _np_scores(s[:, j], o[:, j])
        for k in SCORE_NAMES:
            assert abs(a[k][j].item() - want[k]) <= 1e-12 * abs(want[k]), (j, k, a[k][j].item(), want[k])
        r, al, be = a["r"][j].item(), a["alpha"][j].item(), a["beta"][j].item()
        assert a["kge"][j].item() == 1.0 - np.sqrt((r - 1) ** 2 + (al - 1) ** 2 + (be - 1) ** 2)


def test_series_sums_are_the_sequential_float64_loop():
    from topoflow_glacier_b200.objective import series_sums

    rng = np.random.default_rng(8)
    s, o = rng.normal(size=(50, 4)), rng.normal(size=(50, 4))
    o[rng.uniform(size=o.shape) < 0.2] = np.nan
    acc, _ = series_sums(s, o)
    for j in range(4):
        w = [0.0, 0.0, 0.0, 0.0]
        for t in range(50):
            if np.isfinite(o[t, j]):
                d = s[t, j] - o[t, j]
                w = [w[0] + s[t, j], w[1] + s[t, j] * s[t, j], w[2] + s[t, j] * o[t, j], w[3] + d * d]
        assert acc[:, j].tolist() == w


def test_degenerate_series_give_nan_not_inf():
    import torch

    from topoflow_glacier_b200.objective import SCORE_NAMES, series_scores, skill_scores

    T = 30
    s = np.linspace(0.1, 0.9, T)[:, None].repeat(4, axis=1)
    o = np.empty((T, 4))
    o[:, 0] = 0.5                     # constant observations: var_o = 0
    o[:, 1] = np.nan                  # nothing observed: n = 0
    o[:, 2] = np.tile([-1.0, 1.0], T // 2)   # mean_o = 0
    o[:, 3] = np.linspace(0.2, 0.8, T)
    s[:, 3] = 0.3                     # constant simulation: var_s = 0
    sc = series_scores(s, o)
    for k in SCORE_NAMES:
        assert not torch.isinf(sc[k]).any(), k
    assert torch.isnan(sc["nse"][0]) and torch.isnan(sc["kge"][0]) and torch.isnan(sc["alpha"][0])
    assert np.isfinite(sc["rmse"][0].item()) and np.isfinite(sc["bias"][0].item())
    assert sc["n"][1].item() == 0 and all(torch.isnan(sc[k][1]) for k in SCORE_NAMES if k != "n")
    assert torch.isnan(sc["beta"][2]) and torch.isnan(sc["kge"][2]) and np.isfinite(sc["nse"][2].item())
    assert torch.isnan(sc["r"][3]) and sc["alpha"][3].item() == 0.0 and np.isfinite(sc["nse"][3].item())
    z = torch.zeros(4)
    assert all(torch.isnan(v).all() for k, v in skill_scores((z, z, z, z), (z, z, z)).items() if k != "n")


def test_objective_is_declared_and_the_ctypes_structure_matches_the_header():
    from topoflow_glacier_b200 import _lib

    header = (ROOT / "include" / "tfglacier.h").read_text()
    assert "TFG_API int tfg_bind_objective(tfg_ctx* ctx, const tfg_objective* o, void* stream);" in header
    assert "tfg_bind_objective" in _lib.PROTOTYPES
    assert int(re.search(r"#define TFG_N_OBJ (\d+)", header).group(1)) == _lib.N_OBJ == 4
    body = re.search(r"typedef struct tfg_objective \{(.*?)\} tfg_objective;", header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            ctype = re.match(r"(const )?(\w+)", decl).group(2)
            for name in decl.split(",") if "," in decl else [decl]:
                fields.append((re.findall(r"\w+", name)[-1], "ptr" if "*" in decl else ctype))
    want = {"int32_t": C.c_int32, "int64_t": C.c_int64, "ptr": C.c_void_p}
    assert [f for f, _ in _lib.Objective._fields_] == [f for f, _ in fields]
    for (name, ct), (_, t) in zip(_lib.Objective._fields_, fields):
        assert ct is want[t], name
    assert C.sizeof(_lib.Objective) == 56


def test_observation_csv_round_trip_is_exact(tmp_path):
    """The example's --write-obs / --obs files give back the same float64 bits, NaN where a value is missing."""
    import importlib.util

    import pandas as pd

    spec = importlib.util.spec_from_file_location("calib", ROOT / "examples" / "calibrate_topoflow_glacier.py")
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    rng = np.random.default_rng(12)
    obs = rng.uniform(0.0, 3e-6, (100, 3)) * rng.uniform(0.1, 10.0, (100, 3))
    obs[rng.uniform(size=obs.shape) < 0.3] = np.nan
    start = pd.Timestamp("2013-03-20 00:00")
    ex.write_obs_csv(tmp_path / "o.csv", obs, ["a", "b", "c"], start)
    assert np.array_equal(ex.read_obs_csv(tmp_path / "o.csv", ["a", "b", "c"], start, 100), obs, equal_nan=True)


# ---------------------------------------------------------------------------------------------------- GPU
QUANTITIES = ("h_swe", "M_total", "RH")


def _bits(x):
    import torch

    x = x.contiguous()
    return x.view(torch.int32 if x.element_size() == 4 else torch.int64)


def _same(a, b):
    import torch

    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _setup(N=1536, M=12, T=300, seed=51):
    """Cells, per-cell forcing, catchment forcing (M columns) and a map; per-cell parameters for half of the runs."""
    import bench
    from topoflow_glacier_b200.config import CELL_PARAM_RANGES

    statics, fcell = bench.synthetic_host_sample(N, T, seed=seed)
    _, fcols = bench.synthetic_host_sample(M, T, seed=seed + 1)
    col = (np.arange(N) * M // N).astype(np.int32)
    rng = np.random.default_rng(seed + 2)
    params = {k: rng.uniform(lo, hi, N) for k, (lo, hi) in CELL_PARAM_RANGES.items()}
    return statics, fcell, np.ascontiguousarray(fcols), col, params


def _obs(T_obs, n_cols, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    o = rng.uniform(0.0, scale, (T_obs, n_cols))
    o[rng.uniform(size=o.shape) < 0.25] = np.nan
    o[::5] = np.nan                                                  # whole rows unobserved
    return o


def _engine(statics, mode, T, route, col, M, params, **kw):
    from topoflow_glacier_b200.engine import MeltEngine

    fmap = {} if route == "cell" else dict(forcing_index=col, n_forcing_cols=M, column_terms=(route == "map_ct"))
    return MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode=mode, horizon_steps=T + 1,
                      basin_id=np.zeros(statics["lat"].size, np.int32), n_basin=1, cell_params=params, **fmap, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
@pytest.mark.parametrize("route", ["cell", "map", "map_ct"])
@pytest.mark.parametrize("with_params", [False, True])
def test_sums_equal_host_loop_over_recorded_series(mode, route, with_params, cuda_device):
    """REC+OBJ in one run: the device sums equal the host's sequential float64 loop over the recorded quantity."""
    import torch

    from topoflow_glacier_b200.objective import series_sums

    if mode == "f32" and route == "map_ct":
        pytest.skip("the float32 mode has no column-term pass")
    T, M = 260, 12
    statics, fcell, fcols, col, params = _setup(T=T)
    N = col.size
    dtype = torch.float32 if mode == "f32" else torch.float64
    f = torch.as_tensor(fcell if route == "cell" else fcols).to(cuda_device, dtype).contiguous()
    step0, T_obs = 37, 180                                            # window starts after the run, ends before it
    for qi, q in enumerate(QUANTITIES):
        e = _engine(statics, mode, T, route, col, M, params if with_params else None)
        n_obs_cols = N if route == "cell" else M
        obs = _obs(T_obs, n_obs_cols, seed=qi, scale={"h_swe": 1.0, "M_total": 1e-6, "RH": 1.0}[q])
        e.set_objective(q, obs, obs_step0=step0)
        rec = e.run(f, record=(q,))[q]
        torch.cuda.synchronize()
        assert (e.column_term_launches > 0) == (route == "map_ct")
        # the observation each cell saw, per step of the run
        o_cell = np.full((T, N), np.nan)
        o_cell[step0:step0 + T_obs] = obs[:, np.arange(N) if route == "cell" else col]
        want, _ = series_sums(rec.double().cpu(), o_cell)
        got = torch.stack(e.objective_sums()).cpu()
        assert _same(got, want), (q, (got != want).sum().item())
        assert e.objective["row_counts"].tolist() == [1] * T_obs
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_objective_changes_nothing_else(mode, cuda_device):
    import torch

    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.sharding import BasinAggregates

    T, M = 200, 12
    statics, _, fcols, col, params = _setup(T=T, seed=61)
    dtype = torch.float32 if mode == "f32" else torch.float64
    f = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    out = []
    for bind in (False, True):
        e = _engine(statics, mode, T, "map_ct", col, M, params)
        if bind:
            e.set_objective("h_swe", _obs(T, M, seed=4), obs_step0=0)
        agg = BasinAggregates(T, 1, device=e.device, exponents=e.agg_exponents())
        rec = e.run(f, record=_lib.REC_NAMES, basin_agg=agg.accumulator)
        torch.cuda.synchronize()
        out.append((rec, e.state.clone(), e.ring.clone(), e.window_carry.clone(), agg.decode().clone()))
        e.close()
    for name in _lib.REC_NAMES:
        assert _same(out[0][0][name], out[1][0][name]), name
    for i in (1, 2, 3, 4):                      # state + integrals, window, running window sum, exact basin sums
        assert _same(out[0][i], out[1][i]), i


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_launch_split_does_not_matter(mode, cuda_device):
    """One 300-step run (three launches), 300 step() calls and runs of 7 + 121 + 172 steps give the same sums."""
    import torch

    T, M = 300, 12
    statics, _, fcols, col, params = _setup(N=640, T=T, seed=71)
    dtype = torch.float32 if mode == "f32" else torch.float64
    f = torch.as_tensor(fcols).to(cuda_device, dtype).contiguous()
    obs = _obs(280, M, seed=5)
    sums, scores = [], []
    for how in ("one", "steps", "split"):
        e = _engine(statics, mode, T, "map", col, M, params)
        e.set_objective("h_swe", obs, obs_step0=10)
        if how == "one":
            e.run(f)
        elif how == "steps":
            for t in range(T):
                e.inputs[:5].copy_(f[t])
                e.step()
        else:
            t0 = 0
            for n in (7, 121, 172):
                e.run(f[t0:t0 + n].contiguous())
                t0 += n
        torch.cuda.synchronize()
        sums.append(torch.stack(e.objective_sums()).clone())
        scores.append(e.scores())
        e.close()
    for i in (1, 2):
        assert _same(sums[0], sums[i]), i
        for k, v in scores[0].items():
            assert _same(v, scores[i][k]), (i, k)


@pytest.mark.gpu
def test_rewind_counts_rows_twice_and_reset_zeroes(cuda_device):
    import torch

    T, M = 40, 12
    statics, _, fcols, col, _ = _setup(N=256, T=T, seed=81)
    f = torch.as_tensor(fcols).to(cuda_device, torch.float64).contiguous()
    e = _engine(statics, "f64_fast", T, "map", col, M, None)
    sd = e.state_dict()
    e.set_objective("h_swe", _obs(T, M, seed=6))
    e.run(f)
    n1 = e.scores()["n"].clone()
    e.load_state_dict(sd)
    e.run(f)
    assert torch.equal(e.scores()["n"], 2 * n1)
    assert e.objective["row_counts"].tolist() == [2] * T
    e.load_state_dict(sd)
    e.reset_objective()
    e.run(f)
    assert torch.equal(e.scores()["n"], n1)
    e.set_objective(None)
    with pytest.raises(RuntimeError, match="no objective"):
        e.scores()
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f64_fast", "f32"])
def test_twin_experiment_truth_scores_one(mode, tmp_path, cuda_device):
    import importlib.util

    spec = importlib.util.spec_from_file_location("calib", ROOT / "examples" / "calibrate_topoflow_glacier.py")
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    for daily in (False, True):
        csv = tmp_path / f"obs_{daily}.csv"
        r = ex.run(sets=160, mode=mode, quantity="M_total", daily=daily, write_obs=csv, seed=1, verbose=False)
        K = r["sets"]
        assert r["column_terms"] == (mode != "f32")
        obs = r["obs"]
        for c, b in enumerate(r["best"]):
            o = obs[:, c]
            assert np.nanvar(o) > 0, c
            ti = c * K + r["truth_index"][c]
            assert r["scores"]["rmse"][ti] == 0.0 and r["scores"]["nse"][ti] == 1.0, (c, r["scores"]["nse"][ti])
            assert abs(r["scores"]["kge"][ti] - 1.0) <= 1e-12
            assert b["index"] == r["truth_index"][c], (c, b)
            assert b["n"] == np.isfinite(o).sum()
        again = ex.run(sets=160, mode=mode, quantity="M_total", obs_csv=csv, seed=1, verbose=False)
        assert np.array_equal(again["obs"], obs, equal_nan=True)
        for k, v in r["scores"].items():
            assert np.array_equal(again["scores"][k], v, equal_nan=True), k


@pytest.mark.gpu
def test_bind_errors_name_the_field(cuda_device):
    import torch

    from topoflow_glacier_b200 import _lib

    T, M = 10, 12
    statics, _, _, col, _ = _setup(N=256, T=T, seed=91)
    N = col.size
    e = _engine(statics, "f64", T, "map", col, M, None)
    obs = _obs(T, M, seed=7)
    with pytest.raises(ValueError, match="quantity"):
        e.set_objective("Qh", obs)
    with pytest.raises(ValueError, match="obs must be"):
        e.set_objective("h_swe", obs[:, 0])
    e.set_forcing_map(None)                                          # no map: the default is column = cell
    with pytest.raises(ValueError, match="obs must have one column per cell"):
        e.set_objective("h_swe", obs)
    acc = torch.zeros(4, N, dtype=torch.float64, device=cuda_device)
    o_dev = torch.as_tensor(obs).to(cuda_device).contiguous()
    bad_col = torch.as_tensor(col).to(cuda_device).contiguous()
    bad_col[N // 2] = M                                              # out of range: caught on the device
    b = _lib.Objective(quantity=1, obs=o_dev.data_ptr(), obs_step0=0, n_obs_steps=T, n_obs_cols=M,
                       obs_col=bad_col.data_ptr(), acc=acc.data_ptr())
    assert e.lib.tfg_bind_objective(e.ctx, C.byref(b), e.stream_ptr) != 0
    assert b"obs_col" in e.lib.tfg_last_error()
    b.obs_col = None
    b.quantity = 8
    assert e.lib.tfg_bind_objective(e.ctx, C.byref(b), e.stream_ptr) != 0
    assert b"quantity" in e.lib.tfg_last_error()
    b.quantity = 1
    assert e.lib.tfg_bind_objective(e.ctx, C.byref(b), e.stream_ptr) != 0       # column = cell needs n_obs_cols == N
    assert b"n_obs_cols" in e.lib.tfg_last_error()
    e.close()
    ctx = C.c_void_p()
    lib = _lib.load()
    _lib.check(lib.tfg_create(C.byref(ctx), 0, 0), "tfg_create")
    assert lib.tfg_bind_objective(ctx, C.byref(b), None) != 0                 # before tfg_bind_static
    assert b"tfg_bind_static" in lib.tfg_last_error()
    lib.tfg_destroy(ctx)


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_sharded_two_ranks_equal_one_engine(tmp_path, cuda_device):
    import os
    import subprocess
    import sys

    import torch

    N, T, M = 1000, 150, 10
    statics, _, fcols, _, params = _setup(N=N, M=M, T=T, seed=101)
    col = np.random.default_rng(3).integers(0, M, N).astype(np.int32)
    obs = _obs(T, M, seed=8)
    np.savez(tmp_path / "in.npz", fcols=fcols, col=col, obs=obs, **{f"s_{k}": v for k, v in statics.items()},
             **{f"p_{k}": v for k, v in params.items()})
    from topoflow_glacier_b200.engine import MeltEngine

    one = MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", horizon_steps=T + 1,
                     forcing_index=col, n_forcing_cols=M, cell_params=params)
    one.set_objective("h_swe", obs)
    one.run(torch.as_tensor(fcols).to(cuda_device).contiguous())
    want_sums = torch.stack(one.objective_sums()).cpu().numpy()
    want = {k: v.cpu().numpy() for k, v in one.scores().items()}
    one.close()
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
params = {{k[2:]: z[k] for k in z.files if k.startswith("p_")}}
f = torch.as_tensor(z["fcols"]).cuda()
sh = ShardedMeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode="f64_fast", horizon_steps=f.shape[0] + 1,
                       forcing_index=z["col"], n_forcing_cols={M}, device=0, cell_params=params)
sh.set_objective("h_swe", z["obs"], obs_index=z["col"])
sh.run(f, aggregate=False)
sc = sh.scores(gather=True)
lo, hi = sh.bounds
np.savez({str(tmp_path)!r} + f"/out{{rank}}.npz", sums=torch.stack(sh.objective_sums()).cpu().numpy(), lo=lo, hi=hi,
         **{{k: v.cpu().numpy() for k, v in sc.items()}})
dist.destroy_process_group()
''')
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29631", str(script)],
                       capture_output=True, text=True, env=env, timeout=560)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for k in range(2):
        o = np.load(tmp_path / f"out{k}.npz")
        lo, hi = int(o["lo"]), int(o["hi"])
        assert np.array_equal(o["sums"], want_sums[:, lo:hi])
        for name, v in want.items():
            assert np.array_equal(o[name], v, equal_nan=True), (k, name)
