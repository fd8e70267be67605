"""bench.py contract, CPU side: the reference arm prints ONE JSON line with the keys the driver reads."""

import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-cells", "4096", "--cpu-steps", "2"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "cell_timesteps_per_sec" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    # the unmodified reference when its copy exists (scripts/install_reference.py -> baseline/_ref), else the NumPy port;
    # the port is reported beside it either way
    have_ref = (ROOT / "baseline" / "_ref" / "topoflow_glacier").is_dir()
    assert d["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert d["cpu_baseline_port"]["kind"] == "port" and d["cpu_baseline_port"]["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_times_exactly_steps_runs(monkeypatch, capsys):
    """With the reference copy present, --warmup runs go untimed and exactly --steps runs are timed and averaged
    (the port beside it likewise); each run here reports its own index as its throughput."""
    import bench

    ref, port = [], []

    def fake_ref(cores, inst, n_steps):
        ref.append(len(ref) + 1)
        return float(ref[-1]), 1e-3 * ref[-1], {}

    def fake_port(statics, forcing, start, cores):
        port.append(len(port) + 1)
        return float(port[-1]), 0.0, None

    monkeypatch.setattr(bench, "reference_available", lambda: True)
    monkeypatch.setattr(bench, "reference_throughput", fake_ref)
    monkeypatch.setattr(bench, "cpu_port_throughput", fake_port)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "5", "--warmup", "2",
                                      "--cpu-cells", "64", "--cpu-steps", "2"])
    assert bench.main() == 0
    d = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert len(ref) == 7 and len(port) == 7 and d["steps"] == 5
    assert d["cpu_baseline"]["kind"] == "reference" and d["value"] == sum(range(3, 8)) / 5
    assert d["ms_per_step"] == pytest.approx(sum(range(3, 8)) / 5, rel=1e-12)


def test_gpu_arm_refuses_to_run_without_cuda():
    """The product path has no CPU fallback: without a CUDA device the GPU arm must fail loudly."""
    import torch

    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--no-cpu", "--steps", "1"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_launch(tmp_path, cuda_device):
    """--dump-outputs holds what the last timed launch left: the same bits whether or not the coherent-weather leg (which
    advances the same engine afterwards) runs, a different state with one more timed step, and basin sums of the last
    timestep that are the sums of the dumped state over the basin's cells (all cells dumped below DUMP_CELLS).  Above
    DUMP_CELLS the rows are a sample of DUMP_CELLS cells; everything stays float and within 64 MB."""
    import bench
    from topoflow_glacier_b200.sharding import AGG_NAMES

    def dump(tag, cells, steps, *extra):
        d = tmp_path / tag
        cmd = [sys.executable, str(ROOT / "bench.py"), "--no-cpu", "--no-modes", "--no-strong", "--no-shared",
               "--cells", str(cells), "--chunk", "16", "--warmup", "3", "--steps", str(steps), "--agg", "exact",
               "--dump-outputs", str(d), *extra]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert sum(p.stat().st_size for p in d.iterdir()) <= 64 << 20
        out = {p.stem: np.load(p) for p in d.glob("*.npy")}
        assert set(out) == set(bench.BMI_OUTPUTS) | {f"basin_{n}" for n in AGG_NAMES}
        for name, v in out.items():
            assert v.dtype == np.float64 and np.isfinite(v).all(), name
            assert v.shape == ((min(cells, bench.DUMP_CELLS),) if name in bench.BMI_OUTPUTS else (16, bench.N_BASIN)), name
        return out

    n = 200_000
    a = dump("a", n, 2)
    b = dump("b", n, 2, "--no-coherent")
    c = dump("c", n, 3)
    for name in a:
        assert np.array_equal(a[name].view(np.int64), b[name].view(np.int64)), name
    assert not np.array_equal(a["h_swe"], c["h_swe"])
    basin = np.arange(n) // -(-n // bench.N_BASIN)          # bench.py's raster basins, one GPU
    da_m2 = np.full(n, 9e-4) * 1e6                          # synthetic.synthetic_cells: 30 m cells
    for row, agg in zip(("M_total", "h_swe", "h_iwe"), AGG_NAMES):
        want = np.bincount(basin, weights=a[row] * da_m2, minlength=bench.N_BASIN)
        np.testing.assert_allclose(a[f"basin_{agg}"][-1], want, rtol=1e-12, atol=1e-12 * want.max(), err_msg=agg)
    dump("sampled", bench.DUMP_CELLS + 40_000, 1)
