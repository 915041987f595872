"""-m gpu: periodic particle-mesh gravity (b200_pm_forces_dev / _host) against its float64 numpy restatement
(oracle/pm_np.py), bitwise determinism under source permutation and target sharding, momentum conservation, the
physics end to end against an Ewald sum, KDK stepping through LambdaCDMSimulation(force="pm"), argument checks."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import pm_np

pytestmark = pytest.mark.gpu

L = 100.0


def _posm(pos, mass):
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([pos, mass[:, None]], 1), np.float32)).cuda()


def _cloud(n, seed, centred=False, unit=False, clustered=True):
    rng = np.random.default_rng(seed)
    lo = -L / 2 if centred else 0.0
    pos = rng.uniform(lo, lo + L, (n, 3)).astype(np.float32)
    if clustered:           # half of the particles in a knot: PM is there for structure, not for uniform noise
        k = n // 2
        pos[:k] = (pos[:k] * 0.1 + rng.normal(0, 3.0, (k, 3)) + (lo + L / 2)).astype(np.float32)
    mass = np.ones(n, np.float32) if unit else rng.uniform(0.5, 2.0, n).astype(np.float32)
    return pos, mass


def _pm(engine, posm, grid, rs, phi=True, i0=0, nt=None):
    n = posm.shape[0]
    nt = n - i0 if nt is None else nt
    acc = torch.empty((nt, 3), dtype=torch.float32, device="cuda")
    pot = torch.empty(nt, dtype=torch.float32, device="cuda") if phi else None
    engine.pm_forces_dev(posm, acc, i0, nt, grid=grid, box=L, r_split=rs, phi=pot)
    torch.cuda.synchronize()
    return acc.cpu().numpy(), (pot.cpu().numpy() if phi else None)


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))


# FP32 mesh + cuFFT against float64, measured on a B200: acc 4.3e-7 .. 9.3e-7, phi 7.7e-8 .. 6.5e-7 relative L2
@pytest.mark.parametrize("grid,n,unit,centred,rs_cells", [(32, 4000, True, False, 1.25), (64, 30000, False, True, 1.25),
                                                          (16, 37, False, False, 0.8), (128, 200000, False, True, 2.0)])
def test_pm_vs_numpy(engine, grid, n, unit, centred, rs_cells):
    pos, mass = _cloud(n, grid + n, centred, unit)
    rs = rs_cells * L / grid
    acc, phi = _pm(engine, _posm(pos, mass), grid, rs)
    a0, p0 = pm_np.pm_forces(pos, mass, pos, grid, L, rs, potential=True)
    ea, ep = _rel(acc, a0), _rel(phi, p0)
    print(f"pm vs numpy G={grid} n={n}: acc {ea:.2e} phi {ep:.2e}")
    assert ea < 5e-6 and ep < 5e-6, (ea, ep)


def test_pm_deterministic_under_permutation(engine):
    """Random storage order (the deposit's global-atomic path) and cell-sorted order (its shared-memory table) give
    the same mesh bit for bit, hence bitwise equal forces per particle; two calls are bitwise equal."""
    G = 64
    pos, mass = _cloud(200000, 7)
    posm = _posm(pos, mass)
    a0, p0 = _pm(engine, posm, G, 1.25 * L / G)
    a1, p1 = _pm(engine, posm, G, 1.25 * L / G)
    assert np.array_equal(a0, a1) and np.array_equal(p0, p1)
    cell = np.floor(pm_np.wrap(pos, L) * (G / L)).astype(np.int64) % G
    for perm in (np.random.default_rng(3).permutation(len(pos)),
                 np.lexsort((cell[:, 2], cell[:, 1], cell[:, 0]))):
        ap, pp = _pm(engine, _posm(pos[perm], mass[perm]), G, 1.25 * L / G)
        assert np.array_equal(ap, a0[perm]) and np.array_equal(pp, p0[perm])


def test_pm_sharded_targets_bitwise(engine):
    """Targets split over two contexts on one GPU (the deposit replicated), concatenated == one call."""
    import b200grav
    G = 64
    pos, mass = _cloud(50001, 8)
    posm = _posm(pos, mass)
    a_all, p_all = _pm(engine, posm, G, 1.25 * L / G)
    other = b200grav.Engine(0)
    try:
        h = 50001 // 2
        a0, p0 = _pm(engine, posm, G, 1.25 * L / G, i0=0, nt=h)
        a1, p1 = _pm(other, posm, G, 1.25 * L / G, i0=h, nt=50001 - h)
    finally:
        other.close()
    assert np.array_equal(np.concatenate([a0, a1]), a_all) and np.array_equal(np.concatenate([p0, p1]), p_all)


def test_pm_host_equals_dev(engine):
    G = 32
    pos, mass = _cloud(10000, 9)
    a_dev, _ = _pm(engine, _posm(pos, mass), G, 1.25 * L / G, phi=False)
    assert np.array_equal(engine.pm_forces_host(pos, mass, G, L), a_dev)
    a_unit, _ = _pm(engine, _posm(pos, np.ones_like(mass)), G, 1.25 * L / G, phi=False)
    assert np.array_equal(engine.pm_forces_host(pos, None, G, L), a_unit)


def test_pm_momentum(engine):
    G = 64
    pos, mass = _cloud(100000, 10)
    acc, _ = _pm(engine, _posm(pos, mass), G, 1.25 * L / G, phi=False)
    a = acc.astype(np.float64)
    m = mass.astype(np.float64)
    assert np.abs((m[:, None] * a).sum(0)).max() <= 1e-5 * (m * np.linalg.norm(a, axis=1)).sum()


def test_pm_plus_short_range_matches_ewald(engine):
    """Device long range + numpy short range (r_s = 1.25 h) against the Ewald sum of 256 particles."""
    G = 32
    rs = 1.25 * L / G
    rng = np.random.default_rng(11)
    pos = rng.uniform(0, L, (256, 3)).astype(np.float32)
    mass = rng.uniform(0.5, 2.0, 256).astype(np.float32)
    acc, _ = _pm(engine, _posm(pos, mass), G, rs, phi=False)
    total = acc + pm_np.short_range(pos, pos, mass, L, rs)
    err = _rel(total, pm_np.ewald(pos, pos, mass, L))
    assert err <= 0.015, err


def test_pm_kdk_matches_numpy(engine):
    """LambdaCDMSimulation(force="pm"): 4096 particles, G = 32, 20 KDK steps against a numpy KDK with pm_np forces
    (a = 1 throughout: h = 0 switches the expansion off)."""
    import b200grav
    G, n, dt, steps = 32, 4096, 0.4, 20
    pos, mass = _cloud(n, 12, unit=True, clustered=False)
    pos = pm_np.wrap(pos, L).astype(np.float32)
    vel = np.zeros((n, 3), np.float32)
    sim = b200grav.LambdaCDMSimulation(engine, pos, vel, mass, box=L, force="pm", pm_grid=G, a0=1.0,
                                       cosmo=(0.31, 0.0, 0.69, 0.0))
    for _ in range(steps):
        sim.step(dt)
    x = pos.astype(np.float64)
    v = vel.astype(np.float64)
    a = pm_np.pm_forces(x, mass, x, G, L, 1.25 * L / G)
    for _ in range(steps):
        v += 0.5 * dt * a
        x = pm_np.wrap(x + dt * v, L)
        a = pm_np.pm_forces(x, mass, x, G, L, 1.25 * L / G)
        v += 0.5 * dt * a
    d = sim.positions().astype(np.float64) - x
    d -= L * np.round(d / L)
    moved = np.abs(pm_np.wrap(x - pos + L / 2, L) - L / 2).max()
    assert moved > 0.5 * L / G, moved                  # the particles went somewhere
    assert np.abs(d).max() <= 1e-4 * L, np.abs(d).max()


def test_pm_phase_times(engine):
    G = 32
    pos, mass = _cloud(20000, 13)
    posm = _posm(pos, mass)
    engine.set_timing(True)
    try:
        _pm(engine, posm, G, 1.25 * L / G)
        ms = engine.pm_phase_ms()
    finally:
        engine.set_timing(False)
    assert np.all(ms > 0) and abs(ms[:6].sum() - ms[6]) <= 1e-3 * ms[6] + 1e-2, ms


def test_pm_invalid_arguments(engine):
    lib, h = engine.L, engine._h
    posm = _posm(*_cloud(64, 14))
    acc = torch.empty((64, 3), dtype=torch.float32, device="cuda")
    p, a = posm.data_ptr(), acc.data_ptr()
    ok = dict(n=64, i0=0, nt=64, grid=16, box=L, rs=8.0, acc=a)

    def call(**kw):
        c = dict(ok, **kw)
        return lib.b200_pm_forces_dev(h, p, c["n"], c["i0"], c["nt"], c["grid"], c["box"], c["rs"], c["acc"], None,
                                      None)
    assert call() == 0
    for kw in (dict(grid=15), dict(grid=6), dict(grid=1026), dict(grid=2048), dict(box=0.0), dict(box=-1.0),
               dict(rs=0.0), dict(rs=-1.0), dict(i0=1), dict(nt=65), dict(acc=None)):
        assert call(**kw) == 1, kw
    pos = np.zeros((4, 3), np.float32)
    out = np.zeros((4, 3), np.float32)
    assert lib.b200_pm_forces_host(h, pos.ctypes.data, None, out.ctypes.data, 4, 17, C.c_float(L), 1.0) == 1
    assert lib.b200_pm_forces_host(h, pos.ctypes.data, None, None, 4, 16, C.c_float(L), 1.0) == 1
    torch.cuda.synchronize()
