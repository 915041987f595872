"""CPU: the TreePM short-range factor g(r) of csrc/treepm.cuh compiled for the host, and the numpy TreePM oracle
(oracle/treepm_np.py: the short range with softening, cut-off and a neighbour-list path) against an Ewald sum."""
import os
import subprocess

import numpy as np
import pytest
from scipy.special import erfc

from conftest import ROOT
from oracle import pm_np, treepm_np

L = 100.0
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def _set(kind, seed=1, n=2048):
    """The two 2 048-particle sets of DESIGN 3.12: uniform, and 16 Gaussian clumps (sigma = 3)."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        return rng.uniform(0, L, (n, 3))
    c = rng.uniform(0, L, (16, 3))
    return (c[rng.integers(0, 16, n)] + rng.normal(0, 3.0, (n, 3))) % L


def test_short_g_host_matches_float64(tmp_path):
    """g(u) = erfc(u) + 2u/sqrt(pi) exp(-u^2) from the header, built by nvcc for the host, within 2e-5 relative of
    float64 over [0, r_cut] at the default r_cut = 4.5 r_s (u = r / 2 r_s <= 2.25), on 10^5 points."""
    src = tmp_path / "g.cu"
    src.write_text('#include <stdio.h>\n#include "treepm.cuh"\n'
                   "int main() { for (int k = 0; k < 100000; ++k) { float u = 2.25f * (float)k / 99999.0f;\n"
                   '  float g = b200::treepm_short_g(u); fwrite(&u, 4, 1, stdout); fwrite(&g, 4, 1, stdout); } }\n')
    exe = tmp_path / "g"
    subprocess.run([NVCC, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I",
                    os.path.join(ROOT, "lambda-cdm-raytracing_b200", "csrc"), str(src), "-o", str(exe)], check=True)
    out = np.frombuffer(subprocess.run([str(exe)], check=True, capture_output=True).stdout, np.float32)
    u, g = out[0::2].astype(np.float64), out[1::2].astype(np.float64)
    assert len(u) == 100000 and u[-1] == np.float32(2.25)
    ref = erfc(u) + 2 * u / np.sqrt(np.pi) * np.exp(-u * u)
    err = np.abs(g / ref - 1).max()
    print(f"g(u) host max relative error over [0, 2.25]: {err:.2e}")
    assert err <= 2e-5, err


def test_short_range_defaults_match_pm_np():
    """eps = 0 and no cut-off: the remainder pm_np.short_range sums, over every minimum-image pair."""
    rng = np.random.default_rng(5)
    p = rng.uniform(0, L, (600, 3))
    m = rng.uniform(0.5, 2.0, 600)
    got = treepm_np.short_range(p[:50], p, m, L, 4.0)
    exp = pm_np.short_range(p[:50], p, m, L, 4.0)
    assert np.abs(got - exp).max() <= 1e-14 * np.abs(exp).max()


@pytest.mark.parametrize("kind", ["uniform", "clumps"])
def test_short_range_neighbour_list_equals_brute_force(kind):
    p = _set(kind, seed=7, n=4000)
    m = np.random.default_rng(8).uniform(0.5, 2.0, len(p))
    rs = 1.25 * L / 32
    for eps in (0.0, 0.01):
        a = treepm_np.short_range(p[:500], p, m, L, rs, eps=eps, r_cut=4.5 * rs)
        b = treepm_np.short_range(p[:500], p, m, L, rs, eps=eps, r_cut=4.5 * rs, neighbours=True)
        assert np.abs(a - b).max() <= 1e-12 * np.abs(a).max()
    with pytest.raises(ValueError):
        treepm_np.short_range(p[:5], p, m, L, rs, neighbours=True)


def test_short_range_cutoff_and_softening():
    """r_cut drops exactly the pairs at r >= r_cut; eps softens the denominator, not g."""
    p = np.array([[0.0, 0.0, 0.0], [3.0, 0.0, 0.0], [0.0, 7.0, 0.0], [99.0, 0.0, 0.0]])
    m = np.array([1.0, 2.0, 3.0, 4.0])
    rs, eps = 2.0, 0.5
    g = lambda r: erfc(r / (2 * rs)) + r / (rs * np.sqrt(np.pi)) * np.exp(-r * r / (4 * rs * rs))
    a = treepm_np.short_range(p[:1], p, m, L, rs, eps=eps, r_cut=5.0)[0]
    exp = 2 * g(3.0) * np.array([3.0, 0, 0]) / (9 + eps * eps) ** 1.5 + 4 * g(1.0) * np.array([-1.0, 0, 0]) / (
        1 + eps * eps) ** 1.5
    assert np.allclose(a, exp, rtol=1e-14, atol=0)


@pytest.mark.parametrize("kind", ["uniform", "clumps"])
def test_numpy_treepm_against_ewald(kind):
    """PM + exact short range cut off at 4.5 r_s, r_s = 1.25 h, is within 6e-3 relative L2 of Ewald (256 targets)."""
    p = _set(kind)
    m = np.ones(len(p))
    t = p[:256]
    ew = pm_np.ewald(t, p, m, L)
    for grid in (32, 64):
        rs = 1.25 * L / grid
        tp = pm_np.pm_forces(p, m, t, grid, L, rs) + treepm_np.short_range(t, p, m, L, rs, r_cut=4.5 * rs)
        err = np.linalg.norm(tp - ew) / np.linalg.norm(ew)
        print(f"numpy TreePM {kind} G={grid}: {err:.2e} from Ewald")
        assert err <= 6e-3, (grid, err)
