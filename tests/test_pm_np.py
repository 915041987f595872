"""CPU: the numpy restatement of the periodic particle-mesh force (oracle/pm_np.py) and its Ewald yardstick.

The Ewald sum reduces to Newton at small separations and is converged; the PM force conserves momentum, vanishes on
a uniform lattice and is invariant under whole-cell shifts; and PM(r_s = 1.25 h) plus the analytic short-range
remainder reproduces the Ewald force of a pair to the published TreePM accuracy (Springel 2005)."""
import numpy as np
import pytest

from oracle import pm_np

L = 100.0


def test_ewald_reduces_to_newton_at_small_separation():
    rng = np.random.default_rng(1)
    src = rng.uniform(0, L, (8, 3))
    u = rng.normal(size=(8, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    for r in (1e-3, 1e-2 * L):
        tgt = src + r * u
        for i in range(8):
            a = pm_np.ewald(tgt[i:i + 1], src[i:i + 1], [1.0], L)[0]
            newton = -u[i] / (r * r)
            assert np.linalg.norm(a - newton) <= 1e-5 * np.linalg.norm(newton)


def test_ewald_is_converged():
    rng = np.random.default_rng(2)
    src = rng.uniform(0, L, (16, 3))
    m = rng.uniform(0.5, 2.0, 16)
    tgt = rng.uniform(0, L, (8, 3))
    a = pm_np.ewald(tgt, src, m, L)
    scale = np.abs(a).max()
    # more real-space images / more k vectors change nothing ...
    assert np.abs(pm_np.ewald(tgt, src, m, L, n_real=3) - a).max() <= 1e-10 * scale
    assert np.abs(pm_np.ewald(tgt, src, m, L, n_k=8) - a).max() <= 1e-10 * scale
    # ... and moving weight between the two sums (another alpha) gives the same force
    assert np.abs(pm_np.ewald(tgt, src, m, L, alpha=2.5 / L, n_real=3, n_k=8) - a).max() <= 1e-9 * scale


def _cloud(n, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0, L, (n, 3)), rng.uniform(0.5, 2.0, n)


def test_pm_momentum_conserved():
    pos, m = _cloud(500, 3)
    a = pm_np.pm_forces(pos, m, pos, 32, L, 1.25 * L / 32)
    assert np.abs((m[:, None] * a).sum(0)).max() <= 1e-12 * (m * np.linalg.norm(a, axis=1)).sum()


def test_pm_uniform_lattice_has_no_force():
    G = 16
    g = (np.arange(G) + 0.37) * (L / G)
    pos = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    a, phi = pm_np.pm_forces(pos, np.ones(len(pos)), pos, G, L, 1.25 * L / G, potential=True)
    assert np.abs(a).max() <= 1e-12


@pytest.mark.parametrize("shift_cells", [(1, 0, 0), (3, -5, 7), (16, 16, 16)])
def test_pm_whole_cell_shift_leaves_forces_unchanged(shift_cells):
    G = 32
    pos, m = _cloud(300, 4)
    a0, p0 = pm_np.pm_forces(pos, m, pos, G, L, 1.25 * L / G, potential=True)
    moved = pos + np.asarray(shift_cells, np.float64) * (L / G)          # (16,16,16): the origin-centred frame
    a1, p1 = pm_np.pm_forces(moved, m, moved, G, L, 1.25 * L / G, potential=True)
    assert np.abs(a1 - a0).max() <= 1e-10 * np.abs(a0).max()
    assert np.abs(p1 - p0).max() <= 1e-10 * np.abs(p0).max()


def test_pm_plus_short_range_matches_ewald():
    """G = 32, L = 100, r_s = 1.25 h: r.m.s. (max) relative error of the pair force per separation."""
    G = 32
    h = L / G
    rs = 1.25 * h
    rng = np.random.default_rng(0)
    for q in (0.5, 1, 2, 4, 8, 12):
        n = 48
        src = rng.uniform(0, L, (n, 3))
        u = rng.normal(size=(n, 3))
        u /= np.linalg.norm(u, axis=1)[:, None]
        tgt = src + q * h * u
        errs = []
        for i in range(n):
            s, t = src[i:i + 1], tgt[i:i + 1]
            a = pm_np.pm_forces(s, [1.0], t, G, L, rs) + pm_np.short_range(t, s, [1.0], L, rs)
            e = pm_np.ewald(t, s, [1.0], L)
            errs.append(np.linalg.norm(a - e) / np.linalg.norm(e))
        errs = np.asarray(errs)
        assert np.sqrt((errs ** 2).mean()) <= 0.015 and errs.max() <= 0.025, (q, errs)
