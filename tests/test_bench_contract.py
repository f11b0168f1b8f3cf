"""bench.py contract on CPU: the reference arm prints ONE JSON line with the agreed keys; rank != 0 of a multi-rank
launch prints nothing; the refio writers produce the reference's row formats."""
import io
import json
import os
import subprocess
import sys

import numpy as np

import mg2d


def _run(env_extra, repo_root):
    env = dict(os.environ, MG2D_CPU_SAMPLE_L="64", **env_extra)
    return subprocess.run([sys.executable, os.path.join(repo_root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                           "--gpus", "1"], capture_output=True, text=True, env=env, timeout=600, cwd=repo_root)


def test_reference_arm_json(repo_root):
    out = _run({}, repo_root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is False and d["vs_baseline"] is None
    assert d["metric"] == "wilson_mg_time_to_solution_1e-10" and d["unit"] == "ms" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_are_silent(repo_root):
    out = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, repo_root)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_files(repo_root, tmp_path, monkeypatch):
    """--dump-outputs: float64 files only, the window centred on the point source, the same seeded sample on every call."""
    import importlib.util
    import torch
    # loading bench.py runs its module-level settings: undo them when the test ends
    monkeypatch.setattr(sys, "path", list(sys.path))
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(repo_root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    L = 1024             # more sites than the sample takes
    x = torch.complex(torch.arange(L * L * 2.0), -torch.arange(L * L * 2.0)).reshape(L * L, 2)
    info = {"resnorms": [1.0, 1e-3, 1e-11], "true_resnorm": 2e-11}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), x, info, L)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["resnorms.npy", "true_resnorm.npy", "x_sample.npy", "x_sample_site.npy", "x_window.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float64 and np.array_equal(a, b), n
    w = np.load(tmp_path / "a" / "x_window.npy")
    c, h = L // 2, bench.DUMP_WINDOW // 2
    assert w.shape == (2 * h, 2 * h, 2, 2) and tuple(w[h, h, 1]) == (2.0 * (c + c * L) + 1, -(2.0 * (c + c * L) + 1))
    site = np.load(tmp_path / "a" / "x_sample_site.npy").astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "x_sample.npy")[:, 0, 0], 2.0 * site)
    assert len(np.unique(site)) == len(site) == bench.DUMP_SAMPLE


def test_refio_row_formats():
    L = 4
    phi = (np.arange(L * L * 2) + 1j * np.arange(L * L * 2)).reshape(L * L, 2)
    f = io.StringIO()
    mg2d.refio.write_results_phi_row(f, 7, phi, L)
    row = f.getvalue().rstrip(",\n").split(",")
    assert row[0] == "7" and len(row) == 1 + L * L * 2
    # x outer, y inner (S6/level.h:293-296): second site written is (x=0, y=1) = index L
    a, b = row[3].split("+i")
    assert float(a) == phi[L, 0].real and float(b) == phi[L, 0].imag
    assert mg2d.refio.gen_scaling_row(32, 3, -0.015, 2, 4, 3, 27) == "32\t3\t-0.015000\t2\t2\t4\t3\t27\n"   # S6/modules_main.h:472
    assert mg2d.refio.near_null_filename(32, 2, 4) == "Near-null_L32_blk2_ndof4.txt"                        # S6/modules_main.h:43
