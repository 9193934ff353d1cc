"""bench.py's driver contract, checked without a GPU: the reference arm prints one JSON line with the agreed keys (and times
the restatement, the only thing bench.py may execute from oracle/), the CUDA arm refuses to run without a device instead
of falling back to the CPU, and the roofline's algorithmic-bytes model is the one DESIGN.md states."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_reference_arm_line_has_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "C4", "--steps", "1",
                          "--warmup", "0", "--ref-problems-per-step", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "registrations/sec" and line["higher_is_better"] is True
    assert line["gpu_launches"] == 0 and line["vs_baseline"] is None and line["dtype"] == "f64"
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert set(cb["stage_ms_per_problem"]) >= {"tims", "scale_test", "graph", "clique", "rotation", "translation"}
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["value"] > 0 and "workload" in line["config"]


def test_cuda_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert "no CPU fallback" in (out.stderr + out.stdout)
    assert not any(l.startswith("{") for l in out.stdout.splitlines())  # no number is printed


def _fake_records(B, n, rng):
    import numpy as np
    capi = importlib.import_module("teaser-plusplus_b200.capi")
    sols = np.zeros(B, dtype=capi.SOLUTION_DTYPE)
    sols["clique_size"] = rng.integers(0, n + 1, size=B)
    sols["rotation"] = rng.normal(size=(B, 9))
    sols["n_edges"] = rng.integers(0, 2**40, size=B)
    sols["gnc_cost"] = np.where(rng.random(B) < 0.5, np.inf, rng.random(B))  # +inf: GNC stopped at initialisation
    sols["stage_ms"] = 1.0
    return sols, rng.integers(0, n, size=(B, n)).astype(np.int32)


def test_dump_outputs_formats_and_size_cap(tmp_path):
    import numpy as np
    b = _bench_module()
    rng = np.random.default_rng(3)
    sols, clq = _fake_records(5, 7, rng)
    b.dump_outputs(str(tmp_path / "small"), sols, clq, np.arange(5) + 100)
    d = {f[:-4]: np.load(tmp_path / "small" / f) for f in os.listdir(tmp_path / "small")}
    assert set(d) == set(b.DUMP_FIELDS) | {"clique", "problem"}  # stage_ms (timings) is not a result
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in d.values())
    assert np.array_equal(d["gnc_cost"], np.where(np.isinf(sols["gnc_cost"]), -1.0, sols["gnc_cost"]))
    assert np.array_equal(d["problem"], np.arange(5) + 100) and np.array_equal(d["n_edges"], sols["n_edges"])
    assert np.array_equal(d["rotation"][2], sols[2]["rotation"].reshape(3, 3).T)
    for k in range(5):
        m = sols[k]["clique_size"]
        assert np.array_equal(d["clique"][k, :m], clq[k, :m]) and np.all(d["clique"][k, m:] == -1)

    # a batch over the budget: a seeded sample of whole rows that depends on the batch shape only, under 64 MB on disk
    B, n = 3000, 6000
    big = [_fake_records(B, n, np.random.default_rng(s)) for s in (4, 5)]
    for s, (sols, clq) in enumerate(big):
        b.dump_outputs(str(tmp_path / f"big{s}"), sols, clq, np.arange(B))
    p0, p1 = (np.load(tmp_path / f"big{s}" / "problem.npy") for s in (0, 1))
    assert np.array_equal(p0, p1) and 0 < len(p0) < B and np.all(np.diff(p0) > 0)
    assert sum(os.path.getsize(tmp_path / "big0" / f) for f in os.listdir(tmp_path / "big0")) <= 64_000_000
    rows = p0.astype(np.int64)
    got = np.load(tmp_path / "big0" / "clique.npy")
    assert got.shape == (len(rows), n)
    m = big[0][0]["clique_size"][rows[0]]
    assert np.array_equal(got[0, :m], big[0][1][rows[0], :m])


def test_algorithmic_bytes_model_and_config_table():
    b = _bench_module()
    # SURVEY §8d / DESIGN §3.1: 48 n (points in) + 8 n ceil(n/64) (bitset rows out) + 4 n (degrees out)
    assert b.bytes_graph(5000) == 48 * 5000 + 8 * 5000 * 79 + 4 * 5000 == 3_420_000
    assert b.bytes_graph(64) == 48 * 64 + 8 * 64 * 1 + 4 * 64
    # BASELINE.json's configs are all selectable, C2 is the default the metric is quoted on
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert {"C1", "C2", "C3", "C4", "C5"} <= set(b.CONFIGS)
    assert b.CONFIGS["C2"]["n"] == 5000 and b.CONFIGS["C3"]["n"] == 10000
    assert b.CONFIGS["C4"]["scaling"] == "strong" and b.CONFIGS["C5"]["scaling"] == "strong" and b.CONFIGS["C2"]["scaling"] == "weak"
    assert "registrations" in json.dumps(base).lower()
