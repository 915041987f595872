"""-m gpu: comoving LambdaCDM integration with the periodic PM and TreePM forces (DESIGN 3.13) -- the TreePM
short-range potential (b200_tree_potential_short_dev), the TreePM energy (b200_treepm_energy_dev) and
ComovingSimulation against exact solutions: the float64 short potential and the Ewald potential
(oracle/comoving_np.py), the Zel'dovich pancake, linear growth of P(k) and the Layzer-Irvine equation."""
import numpy as np
import pytest
import torch

import b200grav
from oracle import comoving_np

pytestmark = pytest.mark.gpu

L = 100.0
EPS = 0.01
FACTOR = 4.5
LCDM = (0.31, 0.0, 0.69)


def _posm(pos, mass):
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([pos, mass[:, None]], 1), np.float32)).cuda()


def _set(kind, n, seed):
    """The sets of test_gpu_treepm.py: uniform, or 16 Gaussian clumps (sigma = 3), in [0, L)^3; masses 0.5 .. 2."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        pos = rng.uniform(0, L, (n, 3))
    else:
        c = rng.uniform(0, L, (16, 3))
        pos = (c[rng.integers(0, 16, n)] + rng.normal(0, 3.0, (n, 3))) % L
    pos = pos.astype(np.float32)
    pos[pos >= L] = 0.0
    return pos, rng.uniform(0.5, 2.0, n).astype(np.float32)


def _short_phi(engine, posm, theta, rs, build=True):
    n = posm.shape[0]
    if build:
        engine.tree_build_fixed_dev(posm, n, 8, 20, EPS)
    phi = torch.zeros(n, dtype=torch.float32, device="cuda")
    engine.tree_potential_short_dev(phi, 0, n, theta, L, rs, FACTOR * rs)
    torch.cuda.synchronize()
    return phi.cpu().numpy().astype(np.float64)


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


# ---- the short-range potential ------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind,seed", [("uniform", 11), ("clumps", 12)])
def test_short_potential_exact_limit_and_theta(engine, kind, seed):
    """theta = 0: the exact truncated sum of comoving_np.short_potential to FP32 accuracy; the error falls with theta."""
    pos, mass = _set(kind, 8192, seed)
    rs = 1.25 * L / 32
    posm = _posm(pos, mass)
    ref = comoving_np.short_potential(np.arange(len(pos)), pos, mass, L, rs, EPS, FACTOR * rs)
    err0 = _rel(_short_phi(engine, posm, 0.0, rs), ref)
    errs = [_rel(_short_phi(engine, posm, th, rs, build=False), ref) for th in (0.55, 0.4, 0.25)]
    print(f"short potential {kind}: theta=0 {err0:.2e}; theta 0.55 / 0.4 / 0.25: " + " / ".join(f"{e:.2e}" for e in errs))
    assert err0 <= 1e-5, err0
    assert all(b <= a for a, b in zip(errs, errs[1:])), errs
    assert errs[-1] <= 1e-3, errs


def test_short_potential_errors(engine):
    pos, mass = _set("uniform", 4096, 3)
    posm = _posm(pos, mass)
    n, rs = len(pos), 1.25 * L / 32
    phi = torch.zeros(n, dtype=torch.float32, device="cuda")
    L_ = engine.L
    fresh = b200grav.Engine(0)                                       # no tree at all
    assert L_.b200_tree_potential_short_dev(fresh._h, 0, n, 0.5, L, rs, FACTOR * rs, phi.data_ptr(), None) == 3
    fresh.close()
    engine.tree_build_dev(posm, n, L, 8, 20)                          # the reference-faithful tree
    assert L_.b200_tree_potential_short_dev(engine._h, 0, n, 0.5, L, rs, FACTOR * rs, phi.data_ptr(), None) == 3
    engine.tree_build_fixed_dev(posm, n, 8, 20, EPS)
    assert L_.b200_tree_potential_short_dev(engine._h, 0, n, 0.58, L, rs, FACTOR * rs, phi.data_ptr(), None) == 5
    assert L_.b200_tree_potential_short_dev(engine._h, 0, n, 0.5, L, rs, 0.5 * L, phi.data_ptr(), None) == 1
    assert L_.b200_tree_potential_short_dev(engine._h, 0, n, 0.5, L, 0.0, FACTOR * rs, phi.data_ptr(), None) == 1
    assert L_.b200_tree_potential_short_dev(engine._h, 0, n + 1, 0.5, L, rs, FACTOR * rs, phi.data_ptr(), None) == 1
    assert L_.b200_tree_potential_short_dev(engine._h, 0, n, 0.5, L, rs, FACTOR * rs, None, None) == 1
    other = posm.clone()                                              # energy of an array the tree was not built from
    with pytest.raises(b200grav.B200Error, match="status 3"):
        engine.treepm_energy_dev(other, torch.zeros((n, 3), device="cuda"), 0, n, 32, L)


# ---- the TreePM potential: PM + short range = Ewald ---------------------------------------------------------------

@pytest.mark.parametrize("kind,grid", [("uniform", 32), ("clumps", 32), ("clumps", 64)])
def test_treepm_potential_matches_ewald(engine, kind, grid):
    """theta = 0: PM potential + short potential against the Ewald potential, 1 000 particles; the r.m.s. difference
    relative to the spread of phi.  Also: treepm_energy_dev returns -1/2 sum m phi of that phi, 1/2 sum m v^2."""
    pos, mass = _set(kind, 1000, 21)
    n, rs = len(pos), 1.25 * L / grid
    posm = _posm(pos, mass)
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    phi = torch.empty(n, dtype=torch.float32, device="cuda")
    engine.tree_build_fixed_dev(posm, n, 8, 20, EPS)
    engine.pm_forces_dev(posm, acc, 0, n, grid, L, rs, phi=phi)
    engine.tree_potential_short_dev(phi, 0, n, 0.0, L, rs, FACTOR * rs)
    torch.cuda.synchronize()
    ph = phi.cpu().numpy().astype(np.float64)
    ew = comoving_np.ewald_potential(pos, pos, mass, L)
    d = ph - ew
    rms, mean = np.sqrt((d * d).mean()) / ew.std(), d.mean() / ew.std()
    print(f"TreePM potential vs Ewald {kind} G={grid}: rms {rms:.2e}, mean {mean:+.2e} of the spread {ew.std():.3f}")
    assert rms <= 1e-2, rms
    assert abs(mean) <= 3e-3, mean
    vel = torch.from_numpy(np.random.default_rng(2).normal(0, 1, (n, 3)).astype(np.float32)).cuda()
    ke, pe = engine.treepm_energy_dev(posm, vel, 0, n, grid, L, rs, FACTOR * rs, 0.0)
    m64 = mass.astype(np.float64)
    assert abs(pe / (-0.5 * (m64 * ph).sum()) - 1) < 1e-5
    assert abs(ke / (0.5 * (m64 * (vel.cpu().numpy().astype(np.float64) ** 2).sum(1)).sum()) - 1) < 1e-6


# ---- Zel'dovich pancake ---------------------------------------------------------------------------------------------

def _pancake(engine, force, n_steps, nx=32, ny=64, a0=0.02, a1=0.5, theta=0.3):
    """nx sheets of ny^2 particles on a lattice, displaced along x by the growing plane wave, shell crossing at
    a = 1, run with ComovingSimulation; returns (x error, p error) relative to the amplitudes at a1, the largest
    y / z excursion, and the final x.  The in-plane spacing is half the sheet spacing: the field of a square
    lattice sheet differs from a uniform sheet's by ~exp(-2 pi d / spacing) at distance d, 1.9e-3 at d = spacing,
    3.5e-6 at twice it."""
    h = L / ny
    qx, qy, qz = np.meshgrid((np.arange(nx) + 0.5) * L / nx, (np.arange(ny) + 0.5) * h, (np.arange(ny) + 0.5) * h,
                             indexing="ij")
    qx, qy, qz = qx.ravel(), qy.ravel(), qz.ravel()
    amp = L / (2 * np.pi * comoving_np.growth(1.0))
    x0, p0 = comoving_np.plane_wave(qx, a0, amp, L)
    n = len(qx)
    pos = np.stack([x0 % L, qy, qz], 1).astype(np.float32)
    pos[pos >= L] = 0.0
    mom = np.zeros((n, 3))
    mom[:, 0] = p0
    mass = np.full(n, 3 * LCDM[0] * L ** 3 / (8 * np.pi * n))
    sim = b200grav.ComovingSimulation(engine, pos, mom, mass, L, a0, force=force, pm_grid=128, theta=theta,
                                      eps=0.02 * h, cosmo=LCDM)
    for a in np.geomspace(a0, a1, n_steps + 1)[1:]:
        sim.step(a)
    xs, ps = sim.positions().astype(np.float64), sim.momenta().astype(np.float64)
    xe, pe = comoving_np.plane_wave(qx, a1, amp, L)
    dx = xs[:, 0] - xe
    dx -= L * np.round(dx / L)
    scale = comoving_np.growth(a1) * amp
    pscale = np.abs(pe).max()
    yz = max(np.abs(xs[:, 1] - pos[:, 1]).max(), np.abs(xs[:, 2] - pos[:, 2]).max())
    return (np.sqrt((dx * dx).mean()) / scale, np.sqrt(((ps[:, 0] - pe) ** 2).mean()) / pscale, yz, xs[:, 0])


def test_pancake_treepm_and_richardson(engine):
    """TreePM (theta = 0.3), 64 log steps a = 0.02 -> 0.5: x and p within 5e-3 of the exact solution; y, z still;
    |x32 - x128| / |x64 - x128| in [3, 5.5] (second order through the whole stack)."""
    runs = {k: _pancake(engine, "treepm", k) for k in (32, 64, 128)}
    ex, ep, yz, _ = runs[64]
    print(f"pancake TreePM 64 steps: x err {ex:.2e}, p err {ep:.2e}, y/z excursion {yz:.2e} (box {L})")
    for k in (32, 128):
        print(f"pancake TreePM {k} steps: x err {runs[k][0]:.2e}, p err {runs[k][1]:.2e}")

    def dist(a, b):
        d = a - b
        d -= L * np.round(d / L)
        return np.sqrt((d * d).mean())
    ratio = dist(runs[32][3], runs[128][3]) / dist(runs[64][3], runs[128][3])
    print(f"pancake Richardson ratio |x32 - x128| / |x64 - x128| = {ratio:.2f}")
    assert ex <= 5e-3 and ep <= 5e-3, (ex, ep)
    assert yz <= 1e-3 * L / 64, yz
    assert 3.0 <= ratio <= 5.5, ratio


def test_pancake_pm(engine):
    """PM alone (G = 128, r_s = 1.25 h): within 3e-2."""
    ex, ep, yz, _ = _pancake(engine, "pm", 64)
    print(f"pancake PM 64 steps: x err {ex:.2e}, p err {ep:.2e}, y/z excursion {yz:.2e}")
    assert ex <= 3e-2 and ep <= 3e-2, (ex, ep)
    assert yz <= 1e-3 * L / 64, yz


# ---- linear growth and the Layzer-Irvine equation -------------------------------------------------------------------

def _lowest_bins(engine, posm, grid=128, nbins=4):
    k, p, c = engine.power_spectrum_dev(posm, grid, L, shot_noise_correction=False)     # lattice ICs: no Poisson noise
    sel = np.flatnonzero(c > 0)[:nbins]
    return k[sel], p[sel].astype(np.float64)


def test_linear_growth_and_layzer_irvine(engine):
    """128^3 Zel'dovich particles at z = 49, TreePM theta = 0.5.  At a = 0.1 the lowest four P(k) bins have grown
    as (D(a) / D(a0))^2 within 2 %; continued to a = 1 with energies every step, I(a) = a (K + W) + int K da
    (trapezoid) stays within 2 % of |W(a = 1)|."""
    pos, mom, mass, a0 = b200grav.comoving_zeldovich_dev(engine, grid=128, box=L, z_initial=49.0, seed=7)
    sim = b200grav.ComovingSimulation(engine, pos, mom, mass, L, a0, force="treepm", pm_grid=128, theta=0.5,
                                      eps=0.02, cosmo=LCDM)
    del pos, mom
    _, p0 = _lowest_bins(engine, sim.posm)
    grid_a = np.concatenate([np.geomspace(a0, 0.1, 25), np.geomspace(0.1, 1.0, 81)[1:]])
    k_, w_ = sim.energies()
    ks, ws, As = [k_], [w_], [a0]
    for i, a in enumerate(grid_a[1:], 1):
        sim.step(a)
        k_, w_ = sim.energies()
        ks.append(k_); ws.append(w_); As.append(a)
        if i == 24:                                                  # a = 0.1
            k, p1 = _lowest_bins(engine, sim.posm)
            ratio = p1 / p0 / (comoving_np.growth(a) / comoving_np.growth(a0)) ** 2
            print("linear growth to a = 0.1, P / P0 / (D / D0)^2 in the lowest bins: "
                  + ", ".join(f"k={kk:.3f}: {r:.4f}" for kk, r in zip(k, ratio)))
            assert np.all(np.abs(ratio - 1) <= 0.02), ratio
    assert not engine.tree_overflowed()
    As, ks, ws = np.array(As), np.array(ks), np.array(ws)
    cumk = np.concatenate([[0.0], np.cumsum(0.5 * (ks[1:] + ks[:-1]) * np.diff(As))])
    I = As * (ks + ws) + cumk
    dev = np.abs(I - I[0]).max() / abs(ws[-1])
    print(f"Layzer-Irvine: max |I - I0| / |W(1)| = {dev:.2e}; K(1) = {ks[-1]:.4e}, W(1) = {ws[-1]:.4e}")
    assert dev <= 0.02, dev


def test_production_size(engine):
    """2^24 particles (256^3 Zel'dovich at z = 49), four comoving TreePM steps to a = 0.03: finite, no tree
    overflow, and the lowest P(k) bins grow as D^2 within 2 %."""
    pos, mom, mass, a0 = b200grav.comoving_zeldovich_dev(engine, grid=256, box=L, z_initial=49.0, seed=3)
    sim = b200grav.ComovingSimulation(engine, pos, mom, mass, L, a0, force="treepm", pm_grid=256, theta=0.5,
                                      eps=0.01, cosmo=LCDM)
    del pos, mom
    _, p0 = _lowest_bins(engine, sim.posm, grid=256)
    for a in np.geomspace(a0, 0.03, 5)[1:]:
        sim.step(a)
    torch.cuda.synchronize()
    assert torch.isfinite(sim.posm).all() and torch.isfinite(sim.mom).all() and torch.isfinite(sim.acc).all()
    assert not engine.tree_overflowed()
    _, p1 = _lowest_bins(engine, sim.posm, grid=256)
    ratio = p1 / p0 / (comoving_np.growth(0.03) / comoving_np.growth(a0)) ** 2
    print("2^24 particles, a = 0.02 -> 0.03: P / P0 / (D / D0)^2 in the lowest bins " + ", ".join(f"{r:.4f}" for r in ratio))
    assert np.all(np.abs(ratio - 1) <= 0.02), ratio
