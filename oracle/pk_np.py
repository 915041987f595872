"""pk_np.py -- numpy restatement of the reference's power-spectrum estimator and force-error measure.

TEST INFRASTRUCTURE ONLY (imported by tests/).  Follows
  PowerSpectrumAnalyzer::compute_power_spectrum  src/analysis/power_spectrum.cu:53-84
    assign_particles_to_grid_cic :86-134, compute_density_contrast :161-180,
    apply_fft_forward :182-205 (forward FFT / G^3), bin_power_spectrum :207-285, compute_k_binning :287-299
  the tree-vs-direct error loop of examples/barnes_hut_test.cu:173-189.
Parity status: unpinned by reference outputs -- power_spectrum.cu needs FFTW (absent here) and has no
fixtures; the restatement follows the source line by line and is checked against analytic cases
(tests/test_diag.py: a single plane wave, white noise = shot noise level).
"""
import numpy as np


def cic_grid(pos, mass, grid, box, mass_weighted=True):
    G = grid
    g = np.zeros((G, G, G), np.float64)
    x = np.fmod(pos.astype(np.float32) * np.float32(G / box) + np.float32(G), np.float32(G)).astype(np.float32)  # :93-101
    x = np.where(x < 0, x + np.float32(G), x).astype(np.float32)     # below -box fmod stays negative (not in :93-101)
    i = x.astype(np.int64)
    f = (x - i.astype(np.float32)).astype(np.float32)
    m = mass.astype(np.float32) if mass_weighted else np.ones(len(pos), np.float32)
    for dx in (0, 1):
        for dy in (0, 1):
            for dz in (0, 1):
                w = ((f[:, 0] if dx else 1 - f[:, 0]) * (f[:, 1] if dy else 1 - f[:, 1]) *
                     (f[:, 2] if dz else 1 - f[:, 2])).astype(np.float32)                                  # :113-117
                np.add.at(g, ((i[:, 0] + dx) % G, (i[:, 1] + dy) % G, (i[:, 2] + dz) % G), (m * w).astype(np.float64))
    return g


def power_spectrum(pos, mass, grid, box, mass_weighted=True, shot_noise_correction=True):
    """(k centres, P(k), modes per bin), grid/2 bins of width 2 pi / box."""
    G = grid
    rho = cic_grid(pos, mass, G, box, mass_weighted)
    mean = rho.sum() / G ** 3
    delta = (rho - mean) / mean if mean > 0 else np.zeros_like(rho)                                       # :161-180
    dk_field = np.fft.rfftn(delta) / G ** 3                                                               # :200-204
    dk = np.float32(2.0) * np.float32(np.pi) / np.float32(box)                                             # float, :215
    n = np.fft.fftfreq(G, 1.0 / G)
    n[G // 2] = G // 2                                                                                     # :225-226
    nz = np.arange(G // 2 + 1)
    f32 = np.float32
    kx, ky, kz = np.meshgrid(n.astype(f32) * dk, n.astype(f32) * dk, nz.astype(f32) * dk, indexing="ij")   # float per op
    kmag = np.sqrt((kx * kx + ky * ky) + kz * kz)                                                          # :230
    assert kmag.dtype == np.float32
    b = (kmag / dk).astype(np.int64)                                                                       # :236
    nb = G // 2
    mult = np.where((np.arange(G // 2 + 1) == 0) | (np.arange(G // 2 + 1) == G // 2), 1, 2)[None, None, :] * np.ones_like(b)
    ok = (kmag > 0) & (b < nb)
    p = np.bincount(b[ok], weights=(np.abs(dk_field[ok]) ** 2 * mult[ok]), minlength=nb)
    c = np.bincount(b[ok], weights=mult[ok], minlength=nb).astype(np.int64)
    vol = float(box) ** 3
    pk = np.where(c > 0, p / np.maximum(c, 1), 0.0) * vol                                                  # :262-267
    if shot_noise_correction:
        pk = pk - vol / G ** 3                                                                             # :271-277
    k = (np.arange(nb).astype(f32) * dk + (np.arange(nb) + 1).astype(f32) * dk) * f32(0.5)                 # :296-298
    return k.astype(np.float32), pk, c


def force_error(a_test, a_ref):
    """(mean, max) of |a_test - a_ref| / (|a_ref| + 1e-10)  (examples/barnes_hut_test.cu:173-189)."""
    e = np.abs(a_test.astype(np.float32) - a_ref.astype(np.float32))
    mag = np.sqrt((a_ref.astype(np.float32) ** 2).sum(1))
    rel = np.sqrt((e ** 2).sum(1)) / (mag + np.float32(1e-10))
    return float(rel.astype(np.float64).mean()), float(rel.max())
