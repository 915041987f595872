"""CPU suite: the numpy restatement of the reference's P(k) estimator (oracle/pk_np.py) on cases with a
known answer."""
import numpy as np

from oracle import pk_np


def test_plane_wave_lands_in_its_bin():
    """delta(x) = A cos(2 pi m x / L) sampled by a fine particle lattice with weights: all the power sits in
    bin m with P = A^2/2 * V / (modes in the bin) * (CIC window)^2."""
    G, box, m_wave, A = 32, 100.0, 3, 0.2
    g = (np.arange(G) + 0.0) * (box / G)                       # particles exactly on mesh points: CIC is exact
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    pos = np.stack([x.ravel(), y.ravel(), z.ravel()], 1).astype(np.float32)
    mass = (1.0 + A * np.cos(2 * np.pi * m_wave * pos[:, 0] / box)).astype(np.float32)
    k, pk, c = pk_np.power_spectrum(pos, mass, G, box, mass_weighted=True, shot_noise_correction=False)
    # |delta_k|^2 = (A/2)^2 at k = +-m: the +m mode is in the kz = 0 plane (multiplicity 1), and so is -m
    expect = 2 * (A / 2) ** 2 * box ** 3 / c[m_wave]
    assert abs(pk[m_wave] / expect - 1.0) < 1e-4
    others = np.delete(pk, m_wave)
    assert np.abs(others).max() < 1e-6 * pk[m_wave]
    assert abs(k[m_wave] - (m_wave + 0.5) * 2 * np.pi / box) < 1e-6
    assert c[0] == 0 and c[1] == 26          # bin = int(|n|): bin 0 holds only the skipped DC mode; 6 + 12 + 8 modes have 1 <= |n| < 2


def test_white_noise_is_shot_noise():
    """Uniform random particles: P(k) = V / N at low k (before the CIC window bites)."""
    rng = np.random.default_rng(3)
    n, G, box = 200000, 32, 100.0
    pos = rng.uniform(0, box, (n, 3)).astype(np.float32)
    k, pk, c = pk_np.power_spectrum(pos, np.ones(n, np.float32), G, box, shot_noise_correction=False)
    lo = slice(1, 5)
    w = c[lo] / c[lo].sum()
    assert abs((pk[lo] * w).sum() / (box ** 3 / n) - 1.0) < 0.12
    k2, pk2, _ = pk_np.power_spectrum(pos, np.ones(n, np.float32), G, box, shot_noise_correction=True)
    assert np.allclose(pk - pk2, box ** 3 / G ** 3)              # the reference subtracts V / G^3 (:271)


def test_cic_grid_is_periodic_in_whole_boxes():
    """The CIC mesh of positions moved by whole periods, -3L .. +3L, is the mesh of the originals.  Below -L the
    reference's fmod(x G / L + G, G) is negative; unwrapped, that mesh differs by more than its largest value."""
    rng = np.random.default_rng(17)
    G, box, n = 32, 100.0, 20000
    pos = rng.uniform(0, box, (n, 3)).astype(np.float32)
    mass = rng.uniform(0.5, 2.0, n).astype(np.float32)
    g0 = pk_np.cic_grid(pos, mass, G, box)
    for k in (-3, -2, -1, 1, 2, 3):
        g = pk_np.cic_grid((pos + np.float32(k * box)).astype(np.float32), mass, G, box)
        # float32 positions near 3L carry ~1e-5 of rounding, i.e. ~4e-6 of a cell
        assert np.abs(g - g0).max() <= 1e-4 * g0.max(), (k, np.abs(g - g0).max(), g0.max())
        assert abs(g.sum() - g0.sum()) <= 1e-9 * g0.sum(), k


def test_force_error_measure():
    ref = np.array([[3.0, 4.0, 0.0], [0.0, 0.0, 2.0]], np.float32)
    tst = np.array([[3.0, 4.5, 0.0], [0.0, 0.0, 2.0]], np.float32)
    avg, mx = pk_np.force_error(tst, ref)
    assert abs(mx - 0.1) < 1e-6 and abs(avg - 0.05) < 1e-6
