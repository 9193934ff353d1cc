"""The fused graph builder of tests/cpp/graph_fused_oracle.cc (used to check problems too large to materialise their
TIMs) equals the oracle's orc_build_graph_bits bit for bit."""
import importlib

import numpy as np
import pytest

import oracle_fused
import oracle_lib as orc

synth = importlib.import_module("teaser-plusplus_b200.synth")


def _check(src, dst, nb):
    obits, odeg, oe = orc.build_graph_bits(src, dst, nb)
    fbits, fdeg, fe = oracle_fused.build_graph_bits_fused(src, dst, nb)
    assert np.array_equal(fbits, obits)
    assert np.array_equal(fdeg, odeg)
    assert fe == oe
    _, ddeg, de = oracle_fused.build_graph_bits_fused(src, dst, nb, want_bits=False)
    assert np.array_equal(ddeg, odeg) and de == oe


@pytest.mark.parametrize("cfg", ["C2", "C3", "C5"])
@pytest.mark.parametrize("n", [1, 2, 37, 500, 3000])
def test_fused_graph_equals_oracle(cfg, n):
    pr = synth.config_problem(cfg, 1, n=max(n, 2))
    _check(pr["src"][:n], pr["dst"][:n], pr["noise_bound"])


def test_fused_graph_duplicates_and_nan():
    pr = synth.config_problem("C2", 5, n=300)
    src, dst = pr["src"].copy(), pr["dst"].copy()
    src[10] = src[11]
    dst[10] = dst[11]  # zero-length TIM
    src[20] = src[21]
    _check(src, dst, pr["noise_bound"])
    src[5, 1] = np.nan
    dst[7, 2] = np.nan
    _check(src, dst, pr["noise_bound"])


@pytest.mark.parametrize("shift,scale,nb", [(1e4, 1.0, None), (0.0, 1e-3, 3.3682e-5), (-3e6, 50.0, None),
                                             (0.0, 1.0, 1e-9), (0.0, 1.0, 10.0)])
def test_fused_graph_conditioning(shift, scale, nb):
    pr = synth.config_problem("C2cube", 11, n=400)
    src = pr["src"] * scale + shift
    dst = pr["dst"] * scale - 0.5 * shift
    _check(src, dst, pr["noise_bound"] * scale if nb is None else nb)
