"""CPU suite for the block (hierarchical) time steps of the comoving KDK (DESIGN 3.14): the factor table of
b200grav.block_factor_table (the C ABI's host-scalar factors) against the whole-step factors, the binning rule of the
numpy restatement on hand-made cases, and the float64 oracle scheme (oracle/blockstep_np.py): the global KDK at
max_bins = 1, second order with the bins held fixed."""
import numpy as np
import pytest

from oracle import blockstep_np as bs
from oracle import comoving_np

COSMOS = [(0.31, 0.0, 0.69), (0.3, 0.1, 0.6), (0.35, -0.1, 0.75)]


@pytest.fixture(scope="module")
def lib():
    import b200grav
    return b200grav.load_library()


def _kdk(lib):
    import b200grav
    return lambda a0, a1, cosmo: b200grav.comoving_kdk_factors(lib, a0, a1, *cosmo)


@pytest.mark.parametrize("cosmo", COSMOS)
@pytest.mark.parametrize("a0,a1", [(0.02, 0.03), (0.5, 1.0)])
def test_factor_table_sums(lib, a0, a1, cosmo):
    """For every bin b <= 5 the opening plus closing kicks of its steps sum to K(a0, a1); the sub-step drifts sum to
    D(a0, a1); the table matches the oracle's layout."""
    import b200grav
    kicks, nodes = b200grav.block_factor_table(lib, a0, a1, 6, cosmo)
    D, K = b200grav.comoving_kdk_factors(lib, a0, a1, *cosmo)
    assert nodes[0] == a0 and nodes[-1] == a1 and len(nodes) == 33
    assert len(kicks) == 2 * (2 ** 6 - 1)
    for b in range(6):
        s = sum(kicks[bs.ko_index(b, j)] + kicks[bs.kc_index(b, j, 6)] for j in range(2 ** b))
        assert abs(s / K - 1) <= 1e-14, (b, s / K - 1)
    d = sum(b200grav.comoving_kdk_factors(lib, nodes[k], nodes[k + 1], *cosmo)[0] for k in range(32))
    assert abs(d / D - 1) <= 1e-14, d / D - 1
    ok, on = bs.factor_table(a0, a1, 6, cosmo, _kdk(lib))
    assert np.array_equal(ok, kicks) and np.array_equal(on, nodes)


def test_factor_table_one_bin_is_the_global_step(lib):
    """max_bins = 1: the doubles of ComovingSimulation's global step, K(a0, am), K(am, a1), am = sqrt(a0 a1)."""
    import b200grav
    a0, a1 = 0.0217, 0.0341
    kicks, nodes = b200grav.block_factor_table(lib, a0, a1, 1)
    am = np.sqrt(a0 * a1)
    assert list(nodes) == [a0, a1]
    assert kicks[0] == b200grav.comoving_kdk_factors(lib, a0, am)[1]
    assert kicks[1] == b200grav.comoving_kdk_factors(lib, am, a1)[1]
    with pytest.raises(ValueError):
        b200grav.block_factor_table(lib, a0, a1, 17)


def test_binning_thresholds_and_limits():
    """dlna = 1/2, crit = 1: |g| = 4^(b+1) sits exactly on bin b's threshold (float(dlna^2 / 4^b) |g| = 1 <= crit);
    one ulp above it needs bin b + 1; |g| = 0 is bin 0; huge, inf and NaN are clamped at L."""
    L = 5
    gs = []
    want = []
    for b in range(L):
        g = np.float32(4.0 ** (b + 1))
        gs += [g, np.nextafter(g, np.float32(np.inf))]
        want += [b, b + 1]
    gs += [0.0, 1e30, np.inf, np.nan]
    want += [0, L, L, L]
    g3 = np.zeros((len(gs), 3), np.float32)
    g3[:, 0] = gs
    got = bs.desired_bin32(g3, 0.5, np.float32(1.0), L)
    assert list(got) == want, (list(got), want)
    # the norm: components in a fixed order, sqrt last
    g3 = np.array([[3.0, 4.0, 12.0]], np.float32)
    assert bs.gnorm32(g3)[0] == np.float32(13.0)


@pytest.mark.parametrize("k,lo", [(1, 3), (2, 2), (4, 1), (6, 2)])
def test_rebinning_alignment(k, lo):
    """A particle whose step ends at 0 < k < S and that wants bin 0 gets L - ctz(k) (L = 3): the longest step that
    starts on its own grid there.  One that wants a finer bin keeps it."""
    L = 3
    n = 2
    fac = np.arange(1, 2 * (2 ** 4 - 1) + 1, dtype=np.float32) * np.float32(1e-3)
    bins = np.array([L, L], np.uint8)                       # bin L ends at every k
    gl = np.zeros((n, 3), np.float32)
    gs = np.zeros((n, 3), np.float32)
    gs[1, 0] = 1e30                                         # wants bin L
    mom, acc, b, hist, _ = bs.sync_pass32(k, 4, np.ones(n, np.float32), np.zeros((n, 3), np.float32),
                                       np.zeros((n, 3), np.float32), gl, gs, bins, fac, np.float32(1.0), 0.5)
    assert bs.lowest_bin(k, L) == lo
    assert list(b) == [lo, L]
    assert hist.sum() == n and hist[lo] >= 1 and hist[L] >= 1


def _smooth_forces(box):
    """A smooth periodic acceleration field standing in for the PM and short-range forces."""
    kx = 2 * np.pi / box

    def f(pos, idx, with_long):
        gl = -0.5 * np.sin(kx * pos) if with_long else None
        p = pos[idx]
        gs = 0.2 * np.sin(2 * kx * p[:, [1, 2, 0]]) * np.cos(kx * p)
        return gl, gs
    return f


def test_scheme_one_bin_is_global_kdk():
    """max_bins = 1: the oracle scheme is the global comoving KDK, exactly."""
    rng = np.random.default_rng(4)
    box, n = 1.0, 50
    pos, mom = rng.uniform(0, box, (n, 3)), rng.normal(0, 0.1, (n, 3))
    f = _smooth_forces(box)
    grid = np.geomspace(0.1, 0.3, 5)
    x, p, bins = bs.scheme(pos, mom, np.ones(n), box, grid, 1, f)
    gl, gs = f(pos, np.arange(n), True)
    acc = gl + gs
    xr, pr = pos.copy(), mom.copy()
    for a0, a1 in zip(grid[:-1], grid[1:]):
        am = np.sqrt(a0 * a1)
        pr += acc * comoving_np.kdk_factors(a0, am)[1]
        xr = xr + pr * comoving_np.kdk_factors(a0, a1)[0]
        xr -= box * np.floor(xr / box)
        gl, gs = f(xr, np.arange(n), True)
        acc = gl + gs
        pr += acc * comoving_np.kdk_factors(am, a1)[1]
    assert np.array_equal(x, xr) and np.array_equal(p, pr)
    assert np.all(bins == 0)


def test_scheme_fixed_bins_second_order():
    """Bins 0..3 held fixed (max_bins = 4), a clumped set under the float64 TreePM force (eps = 0.05, a = 0.2 -> 0.3,
    smooth enough for the asymptotic regime): |x_N - x_4N| / |x_2N - x_4N| in [3, 5.5] (5 for a second-order
    scheme)."""
    rng = np.random.default_rng(9)
    box, n = 1.0, 96
    c = rng.uniform(0, box, (4, 3))
    pos = (c[rng.integers(0, 4, n)] + rng.normal(0, 0.08, (n, 3))) % box
    mass = np.full(n, 3 * 0.31 / (8 * np.pi * n))
    mom = np.zeros((n, 3))
    bins = rng.integers(0, 4, n)
    rs = 1.25 / 8
    f = bs.treepm_forces(mass, box, 8, rs, 0.05, 4.5 * rs)
    out = {}
    for steps in (2, 4, 8):
        out[steps] = bs.scheme(pos, mom, mass, box, np.geomspace(0.2, 0.3, steps + 1), 4, f, fixed_bins=bins)[0]

    def dist(a, b):
        d = a - b
        d -= box * np.round(d / box)
        return np.sqrt((d * d).mean())
    ratio = dist(out[2], out[8]) / dist(out[4], out[8])
    assert 3.0 <= ratio <= 5.5, ratio
