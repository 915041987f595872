"""-m gpu: device-side diagnostics (SURVEY 8f N4): the force-error measure and the CIC + FFT power
spectrum against their numpy restatements (oracle/pk_np.py), and an end-to-end physical check --
the measured P(k) of the device-generated Zel'dovich particles follows D^2 x the input spectrum."""
import numpy as np
import pytest
import torch

from inputs import masses_np, uniform_mt
from oracle import ics_np, pk_np

pytestmark = pytest.mark.gpu


def test_force_error_vs_numpy(engine):
    rng = np.random.default_rng(5)
    ref = rng.normal(0, 1, (10001, 3)).astype(np.float32)
    tst = (ref * (1 + rng.normal(0, 1e-3, ref.shape))).astype(np.float32)
    tst[77] *= 3.0
    avg, mx = engine.force_error_dev(torch.from_numpy(tst).cuda(), torch.from_numpy(ref).cuda())
    a0, m0 = pk_np.force_error(tst, ref)
    assert abs(avg / a0 - 1) < 1e-5 and abs(mx / m0 - 1) < 1e-6
    assert engine.force_error_dev(torch.from_numpy(ref).cuda(), torch.from_numpy(ref).cuda()) == (0.0, 0.0)


def test_tree_vs_direct_error_sampler(engine):
    """The reference example's headline number: tree (fixed physics) against the direct sum."""
    n = 50000
    pos, mass = uniform_mt(n, seed=9), masses_np(n, seed=10)
    posm = torch.from_numpy(np.concatenate([pos, mass[:, None]], 1)).cuda()
    a_d = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    a_t = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.direct_forces_dev(posm, a_d, eps=0.01)
    engine.tree_build_fixed_dev(posm, n, 8, 20, eps=0.01)
    errs = []
    for theta in (0.8, 0.5, 0.3):
        engine.tree_walk_dev(a_t, 0, n, theta=theta)
        errs.append(engine.force_error_dev(a_t, a_d))
    assert errs[0][0] > errs[1][0] > errs[2][0] and errs[1][0] < 5e-3 and errs[2][0] < 1e-3, errs
    assert all(mx >= avg for avg, mx in errs)


@pytest.mark.parametrize("grid,n,weighted,shot,centred", [(32, 20000, True, True, False), (64, 100000, False, False, True),
                                                          (16, 5, True, False, False)])
def test_power_spectrum_vs_numpy(engine, grid, n, weighted, shot, centred):
    rng = np.random.default_rng(grid)
    pos = rng.uniform(-50, 50, (n, 3)).astype(np.float32) if centred else rng.uniform(0, 100, (n, 3)).astype(np.float32)
    mass = masses_np(n, seed=grid + 1)
    posm = torch.from_numpy(np.concatenate([pos, mass[:, None]], 1)).cuda()
    k, p, c = engine.power_spectrum_dev(posm, grid, 100.0, weighted, shot)
    k0, p0, c0 = pk_np.power_spectrum(pos, mass, grid, 100.0, weighted, shot)
    assert np.array_equal(c, c0) and np.allclose(k, k0, rtol=1e-6)
    scale = np.abs(p0).max()
    assert np.abs(p - p0).max() < 2e-4 * scale          # float atomics / float FFT vs double


def test_power_spectrum_periodic_in_whole_boxes(engine):
    """Positions moved by -2L, -3L and +5L give the P(k) of the originals, and match pk_np on the moved positions
    (below -L the deposit must wrap the negative fmod result back into the grid)."""
    G, box, n = 32, 100.0, 20000
    rng = np.random.default_rng(23)
    pos = rng.uniform(0, box, (n, 3)).astype(np.float32)
    mass = masses_np(n, seed=24)
    k0, p0, c0 = engine.power_spectrum_dev(torch.from_numpy(np.concatenate([pos, mass[:, None]], 1)).cuda(), G, box)
    scale = np.abs(p0).max()
    for shift in (-2, -3, 5):
        moved = (pos + np.float32(shift * box)).astype(np.float32)
        k, p, c = engine.power_spectrum_dev(torch.from_numpy(np.concatenate([moved, mass[:, None]], 1)).cuda(), G, box)
        assert np.array_equal(c, c0) and np.array_equal(k, k0)
        assert np.abs(p - p0).max() < 2e-4 * scale, (shift, np.abs(p - p0).max() / scale)
        _, pn, cn = pk_np.power_spectrum(moved, mass, G, box)
        assert np.array_equal(c, cn) and np.abs(p - pn).max() < 2e-4 * scale, (shift, np.abs(p - pn).max() / scale)


def test_zeldovich_particles_carry_the_input_spectrum(engine):
    """ICs -> CIC -> FFT -> P(k): at wavelengths well above the mesh, P_measured = D^2 P_linear."""
    G = 128
    n = G ** 3
    posm = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    vel = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    _, _, D, _ = engine.zeldovich_ics_dev(posm, vel, grid=G, box=100.0, z_initial=9.0, seed=4242)
    k, p, c = engine.power_spectrum_dev(posm, G, 100.0, mass_weighted=False, shot_noise_correction=False)
    sel = (np.arange(G // 2) >= 2) & (np.arange(G // 2) <= 10)      # k <= 0.17 k_Nyquist: CIC window > 0.97
    kk = np.arange(G // 2)[sel] * 2 * np.pi / 100.0                  # bin b holds |n| in [b, b+1)
    # average the linear spectrum over each shell like the estimator does (power-law inside a shell is enough)
    want = np.array([np.mean(ics_np.power(np.linspace(k0, k0 + 2 * np.pi / 100.0, 16) )) for k0 in kk]) * D * D
    ratio = p[sel] / want
    tol = 4.0 / np.sqrt(c[sel]) + 0.08                               # sample variance + shell-average / window slack
    assert np.all(np.abs(ratio - 1.0) < tol), (ratio, tol)
