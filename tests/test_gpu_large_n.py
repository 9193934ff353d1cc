"""Problems with 32 768 < n <= 131 072 correspondences: full-size graph stage, clique stage on the compacted
(L-1)-core, and every layer above it (ctypes, C++ façade, pybind).  Checked against the CPU graph builder of
tests/cpp/graph_fused_oracle.cc (the oracle's predicate without materialised TIMs) and the oracle's clique search."""
import functools
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_fused
import oracle_lib as orc

capi = importlib.import_module("teaser-plusplus_b200.capi")
synth = importlib.import_module("teaser-plusplus_b200.synth")

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "teaser-plusplus_b200", "host")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def fixed_params(nb, **kw):
    d = dict(noise_bound=nb, cbar2=1.0, estimate_scaling=0, rotation_estimation_algorithm=0,
             rotation_gnc_factor=1.4, rotation_max_iterations=100, rotation_cost_threshold=1e-12)
    d.update(kw)
    return capi.default_params(**d)


@functools.lru_cache(maxsize=None)
def ball(n, ratio, seed):
    return synth.make_problem(n, ratio, seed, "ball")


@functools.lru_cache(maxsize=4)
def fused(n, ratio, seed, want_bits):
    pr = ball(n, ratio, seed)
    return oracle_fused.build_graph_bits_fused(pr["src"], pr["dst"], pr["noise_bound"], want_bits=want_bits)


def exact_rows(pr, rows):
    """Rows of the inlier graph from a direct float64 evaluation of the predicate (registration.cc:427-443)."""
    n = pr["src"].shape[0]
    beta = 2 * pr["noise_bound"]
    out = []
    for r in rows:
        a = (pr["src"] - pr["src"][r]) ** 2
        b = (pr["dst"] - pr["dst"][r]) ** 2
        want = np.abs(np.sqrt((a[:, 0] + a[:, 1]) + a[:, 2]) - np.sqrt((b[:, 0] + b[:, 1]) + b[:, 2])) <= beta
        want[r] = False
        out.append(want)
    return np.array(out).reshape(len(rows), n)


def unpack(rows, n):
    return np.unpackbits(np.ascontiguousarray(rows).view(np.uint8), axis=-1, bitorder="little")[..., :n].astype(bool)


def is_clique(bits, n, clique):
    sub = unpack(bits[clique], n)[:, clique]
    return bool((sub | np.eye(len(clique), dtype=bool)).all())


# ------------------------------------------------------------------ graph stage
@pytest.mark.parametrize("n,ratio", [(40000, 0.95), (65537, 0.99)])
def test_graph_bit_exact_large(ctx, n, ratio):
    pr = ball(n, ratio, 17)
    obits, odeg, oe = fused(n, ratio, 17, True)
    ctx.set_flags(2)  # verify the FP32 filter against FP64 for every pair
    bits, deg, ne = ctx.graph_build(pr["src"], pr["dst"], 2 * pr["noise_bound"])
    assert ctx.filter_mismatches() == 0
    ctx.set_flags(0)
    assert np.array_equal(bits, obits)
    bits, deg, ne = ctx.graph_build(pr["src"], pr["dst"], 2 * pr["noise_bound"])  # default kernel, fused degrees
    assert np.array_equal(bits, obits) and np.array_equal(deg, odeg) and ne == oe


def test_graph_max_size(ctx):
    n, ratio = 131072, 0.995
    pr = ball(n, ratio, 17)
    _, odeg, oe = fused(n, ratio, 17, False)
    ctx.set_flags(2)
    bits, deg, ne = ctx.graph_build(pr["src"], pr["dst"], 2 * pr["noise_bound"])
    assert ctx.filter_mismatches() == 0
    ctx.set_flags(0)
    bits, deg, ne = ctx.graph_build(pr["src"], pr["dst"], 2 * pr["noise_bound"])
    assert np.array_equal(deg, odeg) and ne == oe
    rows = np.random.default_rng(0).choice(n, size=64, replace=False)
    assert np.array_equal(unpack(bits[rows], n), exact_rows(pr, rows))


def test_graph_debug_kernels_fall_back_above_65535(ctx):
    """The tensor-core (1024) and v7 (2048) kernels pack j in 16 bits: above 65 535 the default kernel runs."""
    n = 70000
    pr = ball(n, 0.99, 23)
    ref, rdeg, re_ = ctx.graph_build(pr["src"], pr["dst"], 2 * pr["noise_bound"])
    for flag in (1024, 2048):
        ctx.set_flags(flag | 4)
        bits, deg, ne = ctx.graph_build(pr["src"], pr["dst"], 2 * pr["noise_bound"])
        assert ctx.debug_counters()["tc_problems"] == 0
        ctx.set_flags(0)
        assert np.array_equal(bits, ref) and np.array_equal(deg, rdeg) and ne == re_


# ------------------------------------------------------------------ whole solve, PMC_EXACT on the compacted core
@pytest.mark.parametrize("n,ratio", [(40000, 0.95), (65537, 0.99), (131072, 0.995)])
def test_solve_ball_large(ctx, n, ratio):
    pr = ball(n, ratio, 17)
    inl = np.sort(pr["inliers"])
    p = fixed_params(pr["noise_bound"])
    ctx.set_flags(4)
    g = ctx.solve(pr["src"], pr["dst"], p)
    counters = ctx.debug_counters()
    ctx.set_flags(0)
    assert g["valid"] and g["sol"].clique_proven_optimal == 1
    assert np.array_equal(g["clique"], inl)
    assert counters["clique_stage_vertices"] == len(inl)  # the (L-1)-core is exactly the inlier set
    if n <= 65537:  # the oracle's exact search on its own bitset (2 GiB at n = 131 072: degrees are checked instead)
        obits, _, _ = fused(n, ratio, 17, True)
        oc, _ = orc.max_clique_bits(obits, n)
        assert np.array_equal(g["clique"], oc)
    else:
        _, odeg, _ = fused(n, ratio, 17, False)
        _, deg = ctx.last_graph(0, n)
        assert np.array_equal(deg, odeg)
    # the clique induces a complete graph: the ordinary path on the clique alone builds the same chain TIMs
    sub = ctx.solve(pr["src"][g["clique"]], pr["dst"][g["clique"]], p)
    assert np.array_equal(sub["clique"], np.arange(len(inl)))
    assert np.array_equal(g["R"], sub["R"]) and np.array_equal(g["t"], sub["t"]) and g["scale"] == sub["scale"]
    assert synth.angular_error(g["R"], pr["R"]) < 0.02 and np.linalg.norm(g["t"] - pr["t"]) < 0.02


def _planted_graph(n, cliques, deg_avg, seed):
    rng = np.random.default_rng(seed)
    m = n * deg_avg // 2
    a = rng.integers(0, n, size=m)
    b = rng.integers(0, n, size=m)
    keep = a != b
    a, b = a[keep], b[keep]
    for K in cliques:
        i, j = np.triu_indices(len(K), 1)
        a = np.concatenate([a, K[i]])
        b = np.concatenate([b, K[j]])
    W = (n + 63) // 64
    bits = np.zeros(n * W, dtype=np.uint64)
    one = np.uint64(1)
    for x, y in ((a, b), (b, a)):
        np.bitwise_or.at(bits, x.astype(np.int64) * W + y // 64, np.left_shift(one, (y % 64).astype(np.uint64)))
    return bits.reshape(n, W)


@pytest.mark.parametrize("two", [False, True])
def test_max_clique_caller_bitset_large(ctx, two):
    n = 50000
    rng = np.random.default_rng(3)
    perm = rng.permutation(n)
    cliques = [np.sort(perm[:150]), np.sort(perm[150:300])] if two else [np.sort(perm[:150])]
    bits = _planted_graph(n, cliques, 12, 4)
    oc, _ = orc.max_clique_bits(bits, n)
    gc, proven = ctx.max_clique(bits, n, mode=0)
    assert proven and np.array_equal(gc, oc)
    assert np.array_equal(gc, min(cliques, key=lambda K: K.tolist()))  # canonical tie-break


def test_ragged_batch_large(ctx):
    prs = [ball(n, 0.95 if n < 60000 else 0.99, 40 + k) for k, n in enumerate((20000, 40000, 70000))]
    p = fixed_params(prs[0]["noise_bound"])
    sols, cliques = ctx.solve_batch([q["src"] for q in prs], [q["dst"] for q in prs], p)
    for b, q in enumerate(prs):
        one = ctx.solve(q["src"], q["dst"], p)
        assert np.array_equal(cliques[b], one["clique"]) and np.array_equal(one["clique"], np.sort(q["inliers"]))
        assert np.array_equal(sols[b]["rotation"], one["sol"].rotation[:])
        assert np.array_equal(sols[b]["translation"], one["sol"].translation[:])
        assert sols[b]["clique_proven_optimal"] == one["sol"].clique_proven_optimal == 1


# ------------------------------------------------------------------ KCORE_HEU / PMC_HEU at n = 50 000
def test_heuristic_modes_large(ctx):
    n = 50000
    pr = ball(n, 0.95, 29)
    bits, deg, ne = ctx.graph_build(pr["src"], pr["dst"], 2 * pr["noise_bound"])
    oc, info = orc.max_clique_bits(bits, n, mode=2, kcore_thr=0.01)
    gc, proven = ctx.max_clique(bits, n, mode=2, kcore_thr=0.01)
    assert info["max_core"] > 0.01 * n and not proven
    assert np.array_equal(gc, oc)  # the innermost core, ascending
    inner = unpack(bits[gc], n)[:, gc].sum(axis=1)
    assert int(inner.min()) == info["max_core"]  # the innermost core's minimum degree is the max core number
    gc, _ = ctx.max_clique(bits, n, mode=2, kcore_thr=0.5)  # max core below int(0.5 n): the greedy clique
    assert len(gc) >= 2 and is_clique(bits, n, gc)
    gc, proven = ctx.max_clique(bits, n, mode=1)
    assert not proven and len(gc) >= 2 and is_clique(bits, n, gc)
    g = ctx.solve(pr["src"], pr["dst"], fixed_params(pr["noise_bound"], inlier_selection_mode=2,
                                                       kcore_heuristic_threshold=0.01))
    assert np.array_equal(g["clique"], oc) and not g["proven"]


# ------------------------------------------------------------------ what stays out of reach
def test_refusals_large(ctx):
    n = 40000
    pr = synth.make_problem(n, 0.99, 31, "incube")  # ~15 % dense: every vertex is in the (L-1)-core
    with pytest.raises(capi.TzrError, match="core"):
        ctx.solve(pr["src"], pr["dst"], fixed_params(pr["noise_bound"]))
    g = ctx.solve(pr["src"], pr["dst"], fixed_params(pr["noise_bound"], inlier_selection_mode=1))
    bits, _ = ctx.last_graph(0, n)
    assert g["valid"] and len(g["clique"]) >= 2 and is_clique(bits, n, g["clique"])
    q = ball(n, 0.95, 17)
    with pytest.raises(capi.TzrError, match="estimate_scaling"):
        ctx.solve(q["src"], q["dst"], fixed_params(q["noise_bound"], estimate_scaling=1))
    big = synth.make_problem(131073, 0.99, 1, "ball")
    with pytest.raises(capi.TzrError):
        ctx.solve(big["src"], big["dst"], fixed_params(big["noise_bound"]))


# ------------------------------------------------------------------ drop-in surfaces
FACADE_MAIN = r"""
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "teaser/registration.h"
int main(int argc, char** argv) {
  const int n = std::atoi(argv[1]);
  std::vector<double> s(3 * (size_t)n), d(3 * (size_t)n);
  FILE* f = std::fopen(argv[2], "rb");
  if (!f || std::fread(s.data(), 8, s.size(), f) != s.size() || std::fread(d.data(), 8, d.size(), f) != d.size()) return 2;
  std::fclose(f);
  teaser::Mat3X src(3, n), dst(3, n);
  for (int i = 0; i < n; ++i)
    for (int r = 0; r < 3; ++r) {
      src(r, i) = s[3 * (size_t)i + r];
      dst(r, i) = d[3 * (size_t)i + r];
    }
  teaser::RobustRegistrationSolver::Params p;
  p.noise_bound = std::atof(argv[3]);
  p.estimate_scaling = false;
  p.rotation_cost_threshold = 1e-12;
  teaser::RobustRegistrationSolver solver(p);
  auto sol = solver.solve(src, dst);
  auto clique = solver.getInlierMaxClique();
  std::printf("%d %zu\n", (int)sol.valid, clique.size());
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) std::printf("%a\n", sol.rotation(r, c));
  for (int r = 0; r < 3; ++r) std::printf("%a\n", sol.translation(r));
  for (auto v : clique) std::printf("%d\n", (int)v);
  return 0;
}
"""


def test_facade_and_pybind_large(ctx, tmp_path):
    n = 40000
    pr = ball(n, 0.95, 17)
    g = ctx.solve(pr["src"], pr["dst"], fixed_params(pr["noise_bound"]))
    subprocess.check_call(["make", "-s", "-C", HOST])
    sys.path.insert(0, os.path.join(HOST, "python"))
    import teaserpp_python as tp
    p = tp.RobustRegistrationSolver.Params()
    p.noise_bound = pr["noise_bound"]
    p.estimate_scaling = False
    p.rotation_cost_threshold = 1e-12
    s = tp.RobustRegistrationSolver(p)
    sol = s.solve(pr["src"].T, pr["dst"].T)
    assert sol.valid and s.getInlierMaxClique() == g["clique"].tolist()
    assert np.array_equal(np.asarray(sol.rotation), g["R"]) and np.array_equal(np.asarray(sol.translation), g["t"])
    # the C++ class library itself
    main = tmp_path / "large_n.cc"
    main.write_text(FACADE_MAIN)
    exe = str(tmp_path / "large_n")
    csrc = os.path.join(ROOT, "teaser-plusplus_b200", "csrc")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-I", os.path.join(HOST, "include"), "-I", os.path.join(ROOT, "include"),
                           str(main), "-L", HOST, "-lteaser_registration", "-L", csrc, "-lteaser_b200",
                           f"-Wl,-rpath,{HOST}:{csrc}", "-o", exe])
    data = tmp_path / "pts.bin"
    with open(data, "wb") as fh:
        fh.write(np.ascontiguousarray(pr["src"]).tobytes())
        fh.write(np.ascontiguousarray(pr["dst"]).tobytes())
    out = subprocess.check_output([exe, str(n), str(data), repr(pr["noise_bound"])], text=True).split()
    valid, m = int(out[0]), int(out[1])
    vals = [float.fromhex(x) for x in out[2:14]]
    assert valid == 1 and m == len(g["clique"])
    assert np.array_equal(np.array(vals[:9]).reshape(3, 3).T, g["R"]) and np.array_equal(np.array(vals[9:]), g["t"])
    assert [int(x) for x in out[14:]] == g["clique"].tolist()
