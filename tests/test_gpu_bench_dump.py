"""bench.py --dump-outputs on the GPU: the files hold what the timed device-pointer path returned for the seeded batch,
and they agree with the host-pointer call on the same problems."""
import importlib
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

capi = importlib.import_module("teaser-plusplus_b200.capi")
synth = importlib.import_module("teaser-plusplus_b200.synth")

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_dump_outputs_holds_the_timed_results(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "C4", "--batch", "6", "--steps", "2",
                          "--warmup", "0", "--no-cpu-baseline", "--parity-problems", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2
    d = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    b = _bench_module()
    assert set(d) == set(b.DUMP_FIELDS) | {"clique", "problem"}
    assert all(a.dtype in (np.float32, np.float64) and a.shape[0] == 6 and np.isfinite(a).all() for a in d.values())
    assert np.array_equal(d["problem"], np.arange(6))

    src, dst, _, nb = b.make_batch("C4", range(6), synth)
    ctx = capi.Context(0)
    try:
        sols, cliques = ctx.solve_batch(list(src), list(dst), b.solver_params(capi, "C4", nb, False))
    finally:
        ctx.close()
    for k in range(6):
        m = int(sols[k]["clique_size"])
        assert d["clique_size"][k] == m and np.array_equal(d["clique"][k, :m], cliques[k])
        assert np.all(d["clique"][k, m:] == -1)
        assert np.allclose(d["rotation"][k], capi.rotation_from_solution_record(sols[k]), rtol=0, atol=1e-9)
        assert d["gnc_cost"][k] == (-1.0 if np.isposinf(sols[k]["gnc_cost"]) else sols[k]["gnc_cost"])
        assert np.allclose(d["translation"][k], sols[k]["translation"], rtol=0, atol=1e-9)
