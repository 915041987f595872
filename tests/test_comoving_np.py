"""CPU suite: the comoving KDK factors of the C ABI (b200_comoving_kdk_factors, a host scalar) against scipy quad and
the Einstein-de Sitter closed forms, its argument checks, the float64 oracle's second-order convergence on the 1-D
Zel'dovich plane wave, and the oracle's TreePM potential convention against its Ewald sum."""
import ctypes as C

import numpy as np
import pytest

from oracle import comoving_np, pm_np

PAIRS = [(0.01, 0.02), (0.02, 1.0), (0.5, 0.51), (1.0, 2.0)]
COSMOS = [(0.31, 0.0, 0.69), (0.3, 0.1, 0.6), (0.35, -0.1, 0.75)]


@pytest.fixture(scope="module")
def lib():
    import b200grav
    return b200grav.load_library()


def _factors(lib, a0, a1, cosmo):
    d, k = C.c_double(), C.c_double()
    rc = lib.b200_comoving_kdk_factors(a0, a1, *cosmo, C.byref(d), C.byref(k))
    return rc, d.value, k.value


@pytest.mark.parametrize("cosmo", COSMOS)
@pytest.mark.parametrize("a0,a1", PAIRS)
def test_factors_match_quad(lib, a0, a1, cosmo):
    rc, d, k = _factors(lib, a0, a1, cosmo)
    dr, kr = comoving_np.kdk_factors(a0, a1, cosmo)
    assert rc == 0
    assert abs(d / dr - 1) <= 1e-12 and abs(k / kr - 1) <= 1e-12, (d / dr - 1, k / kr - 1)


@pytest.mark.parametrize("a0,a1", PAIRS)
def test_factors_einstein_de_sitter_closed_form(lib, a0, a1):
    """D = 2 (a0^-1/2 - a1^-1/2), K = 2 (a1^1/2 - a0^1/2), written without cancellation."""
    rc, d, k = _factors(lib, a0, a1, (1.0, 0.0, 0.0))
    s0, s1 = np.sqrt(a0), np.sqrt(a1)
    k_exact = 2 * (a1 - a0) / (s1 + s0)
    d_exact = k_exact / (s0 * s1)
    assert rc == 0
    assert abs(d / d_exact - 1) <= 1e-14 and abs(k / k_exact - 1) <= 1e-14, (d / d_exact - 1, k / k_exact - 1)


def test_factors_zero_interval(lib):
    assert _factors(lib, 0.3, 0.3, (0.31, 0.0, 0.69)) == (0, 0.0, 0.0)


def test_factors_invalid_arguments(lib):
    lcdm = (0.31, 0.0, 0.69)
    d = C.c_double()
    for a0, a1 in [(0.0, 1.0), (-0.1, 1.0), (0.5, 0.4), (float("nan"), 1.0), (0.5, float("inf"))]:
        assert _factors(lib, a0, a1, lcdm)[0] == 1, (a0, a1)
    assert lib.b200_comoving_kdk_factors(0.1, 1.0, *lcdm, None, C.byref(d)) == 1
    assert lib.b200_comoving_kdk_factors(0.1, 1.0, *lcdm, C.byref(d), None) == 1
    assert _factors(lib, 0.1, 1.0, (0.3, -2.0, 0.0))[0] == 1          # E^2 < 0 at a1
    # E^2 = 0.3 a^-3 - 2 a^-2 + 10 is positive at 0.1 and 1 but negative around its minimum at a = 0.225
    closed = (0.3, -2.0, 10.0)
    assert _factors(lib, 0.1, 1.0, closed)[0] == 1
    assert _factors(lib, 0.5, 1.0, closed)[0] == 0


def test_growth_rate_is_log_derivative():
    for cosmo in COSMOS:
        for a in (0.05, 0.5, 1.0):
            h = 1e-5
            fd = (np.log(comoving_np.growth(a * (1 + h), cosmo)) - np.log(comoving_np.growth(a * (1 - h), cosmo))) / (
                np.log1p(h) - np.log1p(-h))
            assert abs(comoving_np.growth_rate(a, cosmo) / fd - 1) < 1e-8


def test_plane_wave_kdk_converges_at_second_order():
    """Om = 0.31, a = 0.02 -> 0.5 in log-uniform steps, shell crossing at a = 1: the relative position error falls
    by 4 per halving of the step (1.0e-2 / 2.6e-3 / 6.4e-4 / 1.6e-4 at 16 / 32 / 64 / 128 steps)."""
    box, a0, a1 = 1.0, 0.02, 0.5
    amp = box / (2 * np.pi * comoving_np.growth(1.0))
    q = np.array([0.25 * box])                                          # sin = 1: the largest displacement
    x0, p0 = comoving_np.plane_wave(q, a0, amp, box)
    x1, p1 = comoving_np.plane_wave(q, a1, amp, box)
    errs = []
    for n in (16, 32, 64, 128):
        disp, p = comoving_np.kdk_plane(x0 - q, p0, np.geomspace(a0, a1, n + 1))
        errs.append(abs(disp[0] - (x1 - q)[0]) / (x1 - q)[0])
        assert abs(p[0] - p1[0]) / abs(p1[0]) < 3 * errs[-1]
    print("plane-wave KDK position error at 16 / 32 / 64 / 128 steps: " + " / ".join(f"{e:.1e}" for e in errs))
    assert errs[0] < 1.5e-2 and errs[-1] < 2.5e-4, errs
    for a, b in zip(errs, errs[1:]):
        assert 3.5 < a / b < 4.5, errs


def test_pm_plus_short_potential_is_ewald():
    """The convention of the TreePM potential: the numpy PM potential (own smoothed self term included, k = 0 mode
    zero) plus short_potential (minus the self term m / (sqrt(pi) r_s) and the background's 4 pi r_s^2 M / L^3)
    against the Ewald potential, 600 clumped particles, G = 32: within 1.5 % r.m.s. of phi's spread and with a mean
    offset below 0.3 % of it (without the background term the offset would be 4 pi r_s^2 M / L^3 ~ 10 %)."""
    L, n, grid = 100.0, 600, 32
    rng = np.random.default_rng(3)
    c = rng.uniform(0, L, (16, 3))
    pos = (c[rng.integers(0, 16, n)] + rng.normal(0, 3.0, (n, 3))) % L
    m = rng.uniform(0.5, 2.0, n)
    rs = 1.25 * L / grid
    _, phi_pm = pm_np.pm_forces(pos, m, pos, grid, L, rs, potential=True)
    phi = phi_pm + comoving_np.short_potential(np.arange(n), pos, m, L, rs, 0.0, 4.5 * rs)
    ew = comoving_np.ewald_potential(pos, pos, m, L)
    d = phi - ew
    rms, mean = np.sqrt((d * d).mean()) / ew.std(), abs(d.mean()) / ew.std()
    print(f"numpy PM + short potential vs Ewald: rms {rms:.2e}, mean {mean:.2e} of the spread")
    assert rms < 1.5e-2 and mean < 3e-3, (rms, mean)


def test_ewald_potential_madelung():
    """One particle per box: the lattice's regularised self potential -2.837297 / L (simple-cubic Madelung constant
    with a neutralising background), independent of the Ewald splitting."""
    x = np.array([[1.0, 2.0, 3.0]])
    for alpha in (0.3, 0.5):
        assert abs(comoving_np.ewald_potential(x, x, np.ones(1), 10.0, alpha=alpha)[0] * 10 + 2.8372975) < 1e-6
