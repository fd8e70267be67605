"""CPU: host-side logic of the product (time tables, cell tables, config schema, forcing parsing, sharding)
against the oracle / the reference's documented behaviour.  No GPU, no compute calls into the library."""

import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pandas as pd
import pytest

from helpers import load_case, make_oracle

ROOT = Path(__file__).resolve().parent.parent


def test_time_tables_bit_equal_oracle():
    from oracle.np_ref import I_SC, OMEGA, time_row
    from topoflow_glacier_b200.timebase import parse_start, time_tables, utc_offsets

    for start in ("2012100100", "2013032000", "20191231-22"):
        st = parse_start(start)
        tt = time_tables(st, 1, 24 * 40)
        for k in range(0, 24 * 40, 7):
            tr = time_row(st + pd.to_timedelta(k + 1, unit="h"))
            assert tt["clock_hour"][k] == tr.clock_hour and tt["TE"][k] == tr.TE
            assert tt["sin_decl"][k] == np.sin(tr.delta) and tt["cos_decl"][k] == np.cos(tr.delta)
            assert tt["tan_decl"][k] == np.tan(tr.delta) and tt["isc_e0"][k] == I_SC * tr.E0
            assert tt["cos_hour"][k] == np.cos(OMEGA * ((tr.clock_hour - 12.0) - tr.TE))
    tt = time_tables(parse_start("2012100100"), 1, 8760)
    g = utc_offsets(tt["when"], ["America/Los_Angeles", -8.0, "UTC"])
    assert set(np.unique(g[:, 0])) == {-8.0, -7.0} and (g[:, 1] == -8).all() and (g[:, 2] == 0).all()
    # DST ends 2012-11-04 09:00 UTC, begins 2013-03-10 10:00 UTC
    when = tt["when"]
    assert g[when == pd.Timestamp("2012-11-04 08:00"), 0] == -7 and g[when == pd.Timestamp("2012-11-04 09:00"), 0] == -8
    assert g[when == pd.Timestamp("2013-03-10 09:00"), 0] == -8 and g[when == pd.Timestamp("2013-03-10 10:00"), 0] == -7


def test_dt_other_than_one_hour_tables():
    from oracle.np_ref import time_row
    from topoflow_glacier_b200.timebase import parse_start, time_tables

    st = parse_start("2013032000")
    tt = time_tables(st, 3, 50)
    for k in (0, 7, 49):
        assert tt["TE"][k] == time_row(st + pd.to_timedelta(3 * (k + 1), unit="h")).TE


def test_cell_tables_bit_equal_oracle():
    from topoflow_glacier_b200.statics import cell_tables

    case = load_case("rand64")
    s = case["statics"]
    ora = make_oracle(case)
    t = cell_tables(s["lat"], s["lon"], s["slope"], s["aspect"], s["elev"], s["da"], s["T_rain_snow"],
                    M_mass_air=0.0289644, g=9.81)
    assert np.array_equal(t["sin_lat"], np.sin(ora.lat_rad)) and np.array_equal(t["cos_lat"], np.cos(ora.lat_rad))
    assert np.array_equal(t["sin_lat_eq"], np.sin(ora.lat_eq)) and np.array_equal(t["cos_lat_eq"], np.cos(ora.lat_eq))
    assert np.array_equal(t["dlon"], ora.dlon) and np.array_equal(t["t_noon"], ora.t_noon)
    assert np.array_equal(t["neg_tan_lat"], -1.0 * np.tan(ora.lat_rad))
    assert np.array_equal(t["neg_tan_lat_eq"], -1.0 * np.tan(ora.lat_eq_rt))
    assert np.array_equal(t["a_elev"], -0.0289644 * 9.81 * s["elev"]) and np.array_equal(t["da_m2"], ora.da_m2)
    with pytest.raises(ValueError):
        cell_tables([46.0], [-121.0], [-5.0], [0.0], [100.0], [1.0], [0.0], M_mass_air=0.0289644, g=9.81)


def test_config_schema_matches_reference_contract():
    from pydantic import ValidationError

    from topoflow_glacier_b200.config import KERNEL_CONSTANTS, TopoflowGlacierConfig, default_constants

    base = {"site_prefix": "x", "forcing_file": "f.csv", "dt": 1, "start_time": 2013032000, "end_time": "2013033123",
            "da": 16.9, "slope": 88.4, "lat": 46.8, "lon": -121.7, "h0_snow": 0.02, "h0_ice": 2.0, "h0_swe": 0.001,
            "h0_iwe": 1.834, "elev": 2365.7}
    cfg = TopoflowGlacierConfig.model_validate(base)
    assert cfg.start_time == "2013032000" and isinstance(cfg.start_time, str)  # int coerced (reference rejects it)
    assert cfg.T_rain_snow == 1.0 and cfg.aspect == 0.0 and cfg.dust_atten == 0.08 and cfg.rho_snow == 50.0
    assert cfg.sigma == 5.67 * 10 ** (-8) and cfg.Lv == 2500000 and cfg.SATTERLUND is False and cfg.z0_air == 0.01
    for bad in ({"dust_atten": 0.3}, {"canopy_factor": 1.5}, {"z0_air": 1.0}, {"em_surf": 0.5}, {"dt": -1}):
        with pytest.raises(ValidationError):
            TopoflowGlacierConfig.model_validate({**base, **bad})
    missing = dict(base)
    del missing["lat"]
    with pytest.raises(ValidationError):
        TopoflowGlacierConfig.model_validate(missing)
    d = default_constants()
    assert all(k in d for k in KERNEL_CONSTANTS) and d["Cp_snow"] == 2090.0 and d["kappa"] == 0.408


def test_forcing_csv_header_keyed_and_windowed(tmp_path):
    from topoflow_glacier_b200.forcing import RAW_COLUMNS, convert_on_host, read_forcing_csv, stack_catchments

    when = pd.date_range("2013-03-20", periods=30, freq="h")
    rng = np.random.default_rng(0)
    df = pd.DataFrame({"Time": when, "RAINRATE": rng.random(30), "Q2D": rng.random(30) * 1e-2, "T2D": 270 + rng.random(30),
                       "U2D": rng.normal(size=30), "V2D": rng.normal(size=30), "LWDOWN": 300.0, "SWDOWN": 100.0,
                       "PSFC": 88000 + rng.random(30)})
    a = tmp_path / "a.csv"
    df.to_csv(a, index=False)
    b = tmp_path / "b.csv"  # the other column order used in the reference's fixtures
    df[["Time", "RAINRATE", "T2D", "Q2D", "U2D", "V2D", "PSFC", "SWDOWN", "LWDOWN"]].to_csv(b, index=False)
    ra = read_forcing_csv(a, pd.Timestamp("2013-03-20 02:00"), pd.Timestamp("2013-03-20 11:00"))
    rb = read_forcing_csv(b, pd.Timestamp("2013-03-20 02:00"), pd.Timestamp("2013-03-20 11:00"))
    assert ra.shape == (10, len(RAW_COLUMNS)) and np.array_equal(ra, rb)
    blk = stack_catchments([ra, rb[:8]])
    assert blk.shape == (8, 6, 2)
    f = convert_on_host(blk)
    sub = pd.read_csv(a).iloc[2:10]  # what the reference driver itself would read back
    assert np.array_equal(f[:, 0, 0], sub["RAINRATE"].values * 10 ** (-3))
    assert np.array_equal(f[:, 1, 0], -273.15 + sub["T2D"].values)
    assert np.array_equal(f[:, 4, 0], ((sub["U2D"] ** 2 + sub["V2D"] ** 2) ** 0.5).values)
    with pytest.raises(KeyError):
        df.drop(columns=["PSFC"]).to_csv(a, index=False)
        read_forcing_csv(a)


def test_shipped_forcing_samples_and_configs():
    """The committed data fixtures (scripts/import_reference_data.py): both forcing samples of the reference parse by
    header name although their columns come in different orders; all five catchment yamls validate (three hold integer
    times the reference's own schema rejects) and name a forcing file that exists."""
    import yaml

    from topoflow_glacier_b200.config import TopoflowGlacierConfig
    from topoflow_glacier_b200.forcing import RAW_COLUMNS, read_forcing_csv
    from topoflow_glacier_b200.timebase import parse_start

    a = read_forcing_csv(ROOT / "tests" / "data" / "sample-cat-3062920.csv")
    b = read_forcing_csv(ROOT / "tests" / "data" / "mock-forcing-june2012.csv")
    assert a.shape == (288, 6) and b.shape == (168, 6)
    assert a[0, RAW_COLUMNS.index("PSFC")] == 88313.5625 and a[0, RAW_COLUMNS.index("T2D")] == 275.2267761230469
    assert b[0, RAW_COLUMNS.index("PSFC")] == 99472.1 and b[0, RAW_COLUMNS.index("T2D")] == 290.82
    assert b[0, RAW_COLUMNS.index("U2D")] == 0.681 and b[0, RAW_COLUMNS.index("V2D")] == -3.783
    names = sorted(p.name for p in (ROOT / "config").glob("cat-*.yaml"))
    assert names == ["cat-3062784.yaml", "cat-3062920-const.yaml", "cat-3062920.yaml", "cat-3062924.yaml", "cat-3062927.yaml"]
    for n in names:
        raw = yaml.safe_load(open(ROOT / "config" / n))
        cfg = TopoflowGlacierConfig.model_validate(raw)
        assert isinstance(cfg.start_time, str) and (ROOT / cfg.forcing_file).exists() and cfg.tz_name == "America/Los_Angeles"
        window = read_forcing_csv(ROOT / cfg.forcing_file, parse_start(cfg.start_time), parse_start(cfg.end_time))
        assert window.shape[0] == 288   # the sample ends 2013-03-31 23:00; every shipped window contains it
    assert isinstance(yaml.safe_load(open(ROOT / "config" / "cat-3062784.yaml"))["start_time"], int)


def test_netcdf_forcing_reader_packed_and_float(tmp_path):
    """NetCDF forcing files behind the same [T, 6, N] block contract as the CSV reader: the file's own int16 packing is
    handed on unchanged (scale_factor / add_offset), a float file or packed=False gives float64 columns; the time window
    is applied; the unpacked values equal the CSV's within the resolution of the packing."""
    import pandas as pd

    from topoflow_glacier_b200.forcing import (DEFAULT_PACKING, RAW_COLUMNS, read_forcing_csv, read_forcing_netcdf,
                                                 unpack_forcing, write_forcing_netcdf)

    csv = ROOT / "tests" / "data" / "sample-cat-3062920.csv"
    raw = read_forcing_csv(csv)                                          # [288, 6]
    when = pd.to_datetime(pd.read_csv(csv)["Time"])
    block = np.repeat(raw[:, :, None], 3, axis=2) * np.array([1.0, 1.001, 0.999])[None, None, :]
    nc = tmp_path / "forcing.nc"
    write_forcing_netcdf(nc, pd.DatetimeIndex(when), block)
    packed, packing = read_forcing_netcdf(nc)
    assert packed.dtype == np.int16 and packed.shape == (288, 6, 3)
    assert np.array_equal(packing[0], DEFAULT_PACKING[0]) and np.array_equal(packing[1], DEFAULT_PACKING[1])
    err = np.abs(unpack_forcing(packed, packing) - block).max(axis=(0, 2))
    assert (err <= DEFAULT_PACKING[0] / 2 + 1e-9).all(), err
    flt, none = read_forcing_netcdf(nc, packed=False)
    assert none is None and flt.dtype == np.float64 and np.array_equal(flt, unpack_forcing(packed, packing))
    win, _ = read_forcing_netcdf(nc, pd.Timestamp("2013-03-21 00:00"), pd.Timestamp("2013-03-21 23:00"))
    assert win.shape == (24, 6, 3) and np.array_equal(win, packed[24:48])
    assert RAW_COLUMNS == ("RAINRATE", "T2D", "PSFC", "Q2D", "U2D", "V2D")


def test_shard_bounds_cover_all_cells():
    from topoflow_glacier_b200.sharding import shard_bounds, shard_sizes

    for n in (1, 4, 127, 128, 100_000_000, 16_777_216, 12345):
        for world in (1, 2, 3, 4, 8):
            if -(-n // 128) < world:  # fewer 128-cell groups than ranks: a rank without cells would hang the
                with pytest.raises(ValueError):  # collectives of the others (ADVICE r1) -> loud error instead
                    shard_sizes(n, world)
                continue
            sizes = shard_sizes(n, world)
            assert sum(sizes) == n and all(s > 0 for s in sizes)
            assert all(s % 128 == 0 for s in sizes[:-1])
            assert max(sizes) - min(sizes) <= 128 + 127   # dealt out evenly: at most one group (+ the partial one) apart
            hi_prev = 0
            for r in range(world):
                lo, hi = shard_bounds(n, world, r)
                assert lo == hi_prev and hi - lo == sizes[r]
                hi_prev = hi
            assert hi_prev == n


def test_perihelion_table_and_timezone_default():
    from topoflow_glacier_b200.timebase import PERIHELION, default_timezone

    assert PERIHELION[1981] == (2, 2) and PERIHELION[2012] == (5, 0) and PERIHELION[2024] == (3, 1)
    assert default_timezone(46.82, -121.74) == "America/Los_Angeles"
    assert default_timezone(40.0, -105.0) == "America/Denver"
    assert default_timezone(61.0, -149.0) == "America/Anchorage"
    assert default_timezone(-33.0, 151.0) == 10.0


@pytest.mark.timeout(300)
def test_basin_aggregate_allreduce_two_ranks_gloo(tmp_path):
    """world_size 2 on CPU (gloo): per-rank partial basin sums -> all_reduce == the single-process sums."""
    script = tmp_path / "w.py"
    script.write_text(f'''
import os, sys
sys.path.insert(0, {str(ROOT)!r})
import numpy as np, torch, torch.distributed as dist
from topoflow_glacier_b200.sharding import BasinAggregates, basin_sums_host, shard_bounds, dist_info
dist.init_process_group("gloo")
rank, world = dist_info()
assert world == 2
N, NB, T = 1000, 7, 3
rng = np.random.default_rng(0)
vals = rng.random((T, 3, N)); da = rng.random(N) * 1e3; basin = rng.integers(0, NB, N)
lo, hi = shard_bounds(N, world, rank)
agg = BasinAggregates(T, NB)
for t in range(T):
    for j in range(3):
        agg.buffer[t, :, j] = torch.as_tensor(basin_sums_host(vals[t, j, lo:hi], da[lo:hi], basin[lo:hi], NB))
agg.reduce()
# exact mode: the int64 words are all-reduced (exactly) and decoded; value = hi * 2^(E-40) + lo * 2^(E-82)
ex = BasinAggregates(T, NB, exponents=(3, 20, 20))
words = torch.as_tensor(rng.integers(-2**40, 2**40, (2, T * NB * 3 * 2 + 1)))  # same draw on both ranks
ex.accumulator.copy_(words[rank])
ex.reduce()
tot = (words[0] + words[1])[:-1].view(T, NB, 3, 2).double()
e = torch.tensor([3.0, 20.0, 20.0], dtype=torch.float64)
assert torch.equal(ex.buffer, tot[..., 0] * torch.exp2(e - 40) + tot[..., 1] * torch.exp2(e - 82))
assert ex.n_left_out == int(words[0, -1] + words[1, -1])
area = agg.basin_area(torch.as_tensor(da[lo:hi]), torch.as_tensor(basin[lo:hi]))
for t in range(T):
    for j in range(3):
        np.testing.assert_allclose(agg.buffer[t, :, j].numpy(), basin_sums_host(vals[t, j], da, basin, NB), rtol=1e-13)
np.testing.assert_allclose(area.numpy(), np.bincount(basin, weights=da, minlength=NB), rtol=1e-13)
dist.destroy_process_group()
sys.stdout.write("rank %d ok\\n" % rank)  # one write: two ranks share the pipe
''')
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", str(script)],
                       capture_output=True, text=True, env=env, timeout=280)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "rank 0 ok" in r.stdout and "rank 1 ok" in r.stdout


def test_bench_reference_arm_runs_on_cpu():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-cells", "2048", "--cpu-steps", "4"], capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr
    import json

    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline_port"]["kind"] == "port"


def _toy_gpkg(path):
    import sqlite3

    con = sqlite3.connect(path)
    con.execute("create table divides (fid integer primary key, geom blob, divide_id text, toid text, type text, "
                "ds_id real, areasqkm real, vpuid text, id text, lengthkm real, tot_drainage_areasqkm real, has_flowline int)")
    con.execute("create table network (fid integer primary key, id text, toid text, divide_id text, areasqkm real)")
    #   cat-1 -> nex-2 -> wb-2 -> nex-3 -> wb-3 -> nex-9 (terminal)      cat-2 -> nex-3     cat-3 -> nex-9     cat-7 -> nex-8 (other basin)
    rows = [("cat-1", "nex-2", 10.0, 10.0, "wb-1"), ("cat-2", "nex-3", 5.0, 15.0, "wb-2"), ("cat-3", "nex-9", 2.5, 17.5, "wb-3"),
            ("cat-7", "nex-8", 4.0, 4.0, "wb-7")]
    for i, (d, t, a, tot, wb) in enumerate(rows):
        con.execute("insert into divides (fid, divide_id, toid, areasqkm, id, tot_drainage_areasqkm) values (?,?,?,?,?,?)",
                    (i + 1, d, t, a, wb, tot))
        con.execute("insert into network (id, toid, divide_id, areasqkm) values (?,?,?,?)", (wb, t, d, a))
    con.commit()
    con.close()


def test_hydrofabric_topology_and_basin_ids(tmp_path):
    from topoflow_glacier_b200.hydrofabric import read_hydrofabric

    p = tmp_path / "toy.gpkg"
    _toy_gpkg(p)
    h = read_hydrofabric(p)
    assert h.divide_id == ["cat-1", "cat-2", "cat-3", "cat-7"] and h.areasqkm.sum() == 21.5
    assert h.path_to_outlet("cat-1") == ["cat-1", "nex-2", "wb-2", "nex-3", "wb-3", "nex-9"]
    assert h.terminal("cat-7") == "nex-8" and h.upstream_divides("nex-3") == ["cat-1", "cat-2"]
    b, names = h.basin_ids(h.divide_id)
    assert list(b) == [0, 0, 0, 1] and names == ["nex-9", "nex-8"]
    b, names = h.basin_ids(["cat-1", "cat-2", "cat-3"], outlets=["nex-3"])
    assert list(b) == [0, 0, 1] and names == ["nex-3", "nex-9"]
    assert np.array_equal(h.area_of(["cat-2", "cat-7"]), [5.0, 4.0])
    with pytest.raises(FileNotFoundError):
        read_hydrofabric(tmp_path / "missing.gpkg")


def test_pinned_block_needs_the_cuda_library():
    """forcing.pinned_block allocates through the C ABI (cudaHostAlloc): without a GPU it fails loudly instead of handing
    out pageable memory; tfg_host_is_pinned answers 0 for ordinary host memory."""
    import torch

    from topoflow_glacier_b200 import _lib
    from topoflow_glacier_b200.forcing import pinned_block

    lib = _lib.load()
    a = np.zeros(16)
    assert lib.tfg_host_is_pinned(a.ctypes.data) == 0 and lib.tfg_host_is_pinned(None) == 0
    if torch.cuda.is_available():
        blk = pinned_block((4, 6, 8), torch.int16)
        assert lib.tfg_host_is_pinned(blk.data_ptr()) == 1
    else:
        with pytest.raises(RuntimeError, match="tfg_host_alloc"):
            pinned_block((4, 6, 8), torch.int16)
