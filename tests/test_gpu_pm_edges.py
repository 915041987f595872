"""-m gpu: the periodic particle-mesh force (b200_pm_forces_dev) at the edges of what it promises.

Exact properties, compared bit for bit.  The inputs are dyadic: box L = 128, a power-of-two mesh and positions on
a 2^-12 grid, so the wrap, the CIC fractions and every rescaling below are exact in FP32 and anything short of bit
equality is a bug:
  * periodic images -- a source or target moved by k L lands in the same cell with the same fractions;
  * the [0, L) and origin-centred frames;
  * mass scale 2^k -- the fixed-point quantum moves by 2^-k, the integers do not, and the mesh, cuFFT and the
    gather are linear, so the outputs scale by exactly 2^k;
  * mass sign -- round-to-nearest is odd and the int64 sums are two's complement, so the outputs negate exactly;
  * length scale 2^k (positions, L and r_split) -- acceleration x 2^-2k, potential x 2^-k: no hidden length;
  * a uniform lattice and all-zero masses give exactly zero; the plan cache survives a change of mesh.
Against oracle/pm_np.py (float64), at the tolerance of test_gpu_pm.py::test_pm_vs_numpy: boundary coordinates,
odd and non-power-of-two meshes, extreme split radii, signed and widely ranged masses, and deposits crafted to
reach the shared-memory table's fallbacks.  Production size: 2^24 Zel'dovich particles at G = 256 and 512 in
Hilbert storage order, and G = 1024 against an Ewald sum."""
import ctypes as C
import time

import numpy as np
import pytest
import torch

from oracle import pm_np

pytestmark = pytest.mark.gpu

L = 128.0          # dyadic box of the exact tests
Q = 4096.0         # positions on a 1 / Q grid
TOL = 5e-6         # relative L2, as test_pm_vs_numpy
SHIFTS = np.array([-3, -1, 1, 2, 7])


def _posm(pos, mass):
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([pos, np.asarray(mass)[:, None]], 1),
                                                 np.float32)).cuda()


def _pm(engine, posm, grid, box, rs, i0=0, nt=None):
    nt = posm.shape[0] - i0 if nt is None else nt
    acc = torch.empty((nt, 3), dtype=torch.float32, device="cuda")
    pot = torch.empty(nt, dtype=torch.float32, device="cuda")
    engine.pm_forces_dev(posm, acc, i0, nt, grid=grid, box=box, r_split=rs, phi=pot)
    torch.cuda.synchronize()
    return acc.cpu().numpy(), pot.cpu().numpy()


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))


def _dyadic_cloud(n, seed, box=L):
    """Half uniform, half in a knot, on the 1 / Q grid inside [0, box)."""
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0, box, (n, 3))
    pos[: n // 2] = box / 2 + rng.normal(0, box / 32, (n // 2, 3))
    return (np.floor(np.mod(pos, box) * Q) / Q).astype(np.float32)


def _masses(kind, n, seed):
    """'ordinary': uniform in [0.5, 2).  'wide': the same plus two particles of mass +2^20 and -2^20.  The quantum is
    2^(ilogb(n max|m|) - 60): with ordinary masses m W is a whole number of quanta (round-to-nearest never acts);
    here a unit mass is 2^24 quanta, so most contributions are rounded and the light cells' densities resolve one
    quantum in FP32 -- which makes the rounding rule of the deposit visible in the outputs."""
    m = np.random.default_rng(seed).uniform(0.5, 2.0, n).astype(np.float32)
    if kind == "wide":
        m[n // 3], m[2 * n // 3] = 2.0 ** 20, -(2.0 ** 20)
    return m


# ---- exact properties -----------------------------------------------------------------------------------------------

def test_pm_periodic_images_bitwise(engine):
    """Massive sources followed by massless tracers (targets only: every run has the same n and max|m|, hence the
    same quantum).  Moving each source, each tracer, or both by its own k L changes no bit."""
    G, ns, nt = 64, 30000, 5000
    rng = np.random.default_rng(1)
    src, trc = _dyadic_cloud(ns, 2), _dyadic_cloud(nt, 3)
    mass = np.concatenate([_masses("ordinary", ns, 4), np.zeros(nt, np.float32)])
    ks, kt = rng.choice(SHIFTS, (ns, 3)) * L, rng.choice(SHIFTS, (nt, 3)) * L
    a0, p0 = _pm(engine, _posm(np.concatenate([src, trc]), mass), G, L, 1.25 * L / G)
    assert np.abs(a0[:ns]).max() > 0
    for s, t in ((src + ks, trc), (src, trc + kt), (src + ks, trc + kt)):
        a, p = _pm(engine, _posm(np.concatenate([s, t]).astype(np.float32), mass), G, L, 1.25 * L / G)
        assert np.array_equal(a, a0) and np.array_equal(p, p0)


def test_pm_frame_bitwise(engine):
    """The same particles in the [0, L) and in the origin-centred [-L/2, L/2) frame."""
    G = 64
    pos, mass = _dyadic_cloud(40000, 5), _masses("ordinary", 40000, 6)
    a0, p0 = _pm(engine, _posm(pos, mass), G, L, 1.25 * L / G)
    centred = np.where(pos >= L / 2, pos - np.float32(L), pos).astype(np.float32)
    assert centred.min() < 0
    a1, p1 = _pm(engine, _posm(centred, mass), G, L, 1.25 * L / G)
    assert np.array_equal(a1, a0) and np.array_equal(p1, p0)


@pytest.mark.parametrize("kind", ["ordinary", "wide"])
def test_pm_mass_scale_bitwise(engine, kind):
    G, n = 64, 65536
    pos, mass = _dyadic_cloud(n, 7), _masses(kind, n, 8)
    a0, p0 = _pm(engine, _posm(pos, mass), G, L, 1.25 * L / G)
    for k in (-40, -13, 13, 40):
        a, p = _pm(engine, _posm(pos, np.ldexp(mass, k)), G, L, 1.25 * L / G)
        assert np.array_equal(a, np.ldexp(a0, k)) and np.array_equal(p, np.ldexp(p0, k)), k


@pytest.mark.parametrize("kind", ["ordinary", "wide"])
def test_pm_mass_sign_bitwise(engine, kind):
    """Negated masses: every contribution rounds to the negated integer, the int64 mesh and its total negate
    (two's complement), T / cells truncates towards zero, so the density and everything after it negate."""
    G, n = 64, 65536
    pos, mass = _dyadic_cloud(n, 9), _masses(kind, n, 10)
    a0, p0 = _pm(engine, _posm(pos, mass), G, L, 1.25 * L / G)
    a1, p1 = _pm(engine, _posm(pos, -mass), G, L, 1.25 * L / G)
    assert np.array_equal(a1, -a0) and np.array_equal(p1, -p0)


def test_pm_length_scale_bitwise(engine):
    G, n = 64, 40000
    pos, mass = _dyadic_cloud(n, 11), _masses("ordinary", n, 12)
    rs = 1.25 * L / G
    a0, p0 = _pm(engine, _posm(pos, mass), G, L, rs)
    for k in (-20, -5, 1, 20):
        a, p = _pm(engine, _posm(np.ldexp(pos, k), mass), G, np.ldexp(L, k), np.ldexp(rs, k))
        assert np.array_equal(a, np.ldexp(a0, -2 * k)) and np.array_equal(p, np.ldexp(p0, -k)), k


@pytest.mark.parametrize("grid,box", [(8, L), (64, L), (48, 96.0)])
@pytest.mark.parametrize("offset", [0.0, 0.5])
def test_pm_uniform_lattice_is_exactly_zero(engine, grid, box, offset):
    """One particle per cell, on the mesh points (one contribution each) or at the cell centres (eight of m / 8):
    the integer mesh is uniform, equals T / cells, and the density is exactly zero -- so are the outputs."""
    h = box / grid
    i = (np.arange(grid) + offset) * h
    x, y, z = np.meshgrid(i, i, i, indexing="ij")
    pos = np.stack([x.ravel(), y.ravel(), z.ravel()], 1).astype(np.float32)
    pos = pos[np.random.default_rng(grid).permutation(len(pos))]          # spread cells over the CTAs
    a, p = _pm(engine, _posm(pos, np.full(len(pos), 0.7, np.float32)), grid, box, 1.25 * h)
    assert np.all(a == 0) and np.all(p == 0), (np.abs(a).max(), np.abs(p).max())


def test_pm_zero_masses_are_exactly_zero(engine):
    pos = _dyadic_cloud(10000, 13)
    a, p = _pm(engine, _posm(pos, np.zeros(10000, np.float32)), 32, L, 5.0)
    assert np.all(a == 0) and np.all(p == 0)


def test_pm_plan_cache_survives_other_meshes(engine):
    """G = 64, then G = 32, then a P(k) (its own plan and buffers), then G = 64 again: the first result."""
    pos, mass = _dyadic_cloud(30000, 14), _masses("ordinary", 30000, 15)
    posm = _posm(pos, mass)
    a0, p0 = _pm(engine, posm, 64, L, 2.5)
    _pm(engine, posm, 32, L, 5.0)
    engine.power_spectrum_dev(posm, 48, L)
    a1, p1 = _pm(engine, posm, 64, L, 2.5)
    assert np.array_equal(a1, a0) and np.array_equal(p1, p0)


# ---- against the float64 restatement ----------------------------------------------------------------------------

def _cloud(n, seed, box, centred=False):
    rng = np.random.default_rng(seed)
    lo = -box / 2 if centred else 0.0
    pos = rng.uniform(lo, lo + box, (n, 3))
    pos[: n // 2] = lo + box / 2 + rng.normal(0, 0.03 * box, (n // 2, 3))
    return pos.astype(np.float32)


def _check_vs_numpy(engine, pos, mass, grid, box, rs, label, sub=None):
    acc, phi = _pm(engine, _posm(pos, mass), grid, box, rs)
    a0, p0 = pm_np.pm_forces(pos, mass, pos, grid, box, rs, potential=True)
    ea, ep = _rel(acc, a0), _rel(phi, p0)
    print(f"pm vs numpy {label} G={grid} r_s={rs / (box / grid):g} h: acc {ea:.2e} phi {ep:.2e}")
    assert ea < TOL and ep < TOL, (label, ea, ep)
    if sub is not None:
        es, eps = _rel(acc[sub], a0[sub]), _rel(phi[sub], p0[sub])
        assert es < TOL and eps < TOL, (label, es, eps)
    return acc, phi


@pytest.mark.parametrize("grid", [32, 48])
def test_pm_boundary_coordinates_vs_numpy(engine, grid):
    """0, -0.0, L, the float below L, the negative float above 0, cell faces and images up to +-8 L, on all three
    axes, mixed into a clustered cloud.  Checked over all targets and over the boundary targets alone."""
    box = 100.0
    f32 = np.float32
    special = np.array([0.0, -0.0, box, np.nextafter(f32(box), f32(0)), -np.nextafter(f32(0), f32(1))], f32)
    faces = (np.arange(0, grid + 1, 7) * f32(box / grid)).astype(f32)
    rng = np.random.default_rng(grid)
    base = rng.uniform(0, box, (400, 3))
    images = (base + rng.integers(-8, 9, (400, 3)) * box).astype(f32)
    corners = np.stack(np.meshgrid(special, special, special, indexing="ij"), -1).reshape(-1, 3)
    mixed = rng.choice(np.concatenate([special, faces]), (600, 3))
    mixed[np.arange(600), rng.integers(0, 3, 600)] = rng.uniform(0, box, 600)     # one interior coordinate
    edge = np.concatenate([corners, mixed, images]).astype(f32)
    pos = np.concatenate([edge, _cloud(20000, grid + 1, box)]).astype(f32)
    mass = np.random.default_rng(grid + 2).uniform(0.5, 2.0, len(pos)).astype(f32)
    _check_vs_numpy(engine, pos, mass, grid, box, 1.25 * box / grid, "boundary", sub=slice(0, len(edge)))


@pytest.mark.parametrize("grid,rs_cells", [(8, 1.25), (10, 1.25), (10, 0.5), (48, 0.5), (48, 8.0), (96, 1.25),
                                           (96, 0.5), (250, 1.25), (250, 8.0)])
def test_pm_grids_and_splits_vs_numpy(engine, grid, rs_cells):
    """The smallest mesh, non-power-of-two meshes (other cuFFT code paths, inexact G / L) and split radii from half a
    cell (little filtering against the W^-2 deconvolution) to eight cells."""
    box = 100.0
    pos = _cloud(30000, grid, box, centred=grid % 4 == 0)
    mass = np.random.default_rng(grid + 3).uniform(0.5, 2.0, len(pos)).astype(np.float32)
    _check_vs_numpy(engine, pos, mass, grid, box, rs_cells * box / grid, "grid")


@pytest.mark.parametrize("kind", ["zero_total", "negative_total", "ratio_1e4"])
def test_pm_signed_and_ranged_masses_vs_numpy(engine, kind):
    """Mixed signs summing to about zero, a negative total, and masses spread over four decades (zoom runs).
    The quantum is 2^(ilogb(n max|m|) - 60) of the mass unit, so it grows with max|m| / mean|m|: at n = 2^20 one
    quantum is 4.8e-7 of the mean mass at a ratio of 1e6 and 6.1e-5 at 1e8 -- beyond FP32's 6e-8 from about 1e5."""
    box, G, n = 100.0, 64, 50000
    rng = np.random.default_rng(31)
    pos = _cloud(n, 32, box, centred=True)
    m = rng.uniform(0.5, 2.0, n)
    if kind == "zero_total":
        m = np.where(np.arange(n) % 2 == 0, m, -np.roll(m, 1))                # +m_i, -m_i pairs at other places
    elif kind == "negative_total":
        m = np.where(rng.random(n) < 0.7, -m, m)
    else:
        m = 10.0 ** rng.uniform(0, 4, n)
    mass = m.astype(np.float32)
    total = float(mass.astype(np.float64).sum())
    if kind == "zero_total":
        assert total == 0.0
    elif kind == "negative_total":
        assert total < -0.2 * np.abs(mass).sum()
    _check_vs_numpy(engine, pos, mass, G, box, 1.25 * box / G, kind)


def _slot(cell):
    """pm.cu's pm_table_add hash: (cell * 0x9E3779B1 mod 2^32) >> (32 - 12)."""
    return ((np.asarray(cell, np.uint64) * np.uint64(0x9E3779B1)) & np.uint64(0xFFFFFFFF)) >> np.uint64(20)


@pytest.mark.parametrize("kind", ["probe_overflow", "one_cell"])
def test_pm_crafted_deposits(engine, kind):
    """The first CTA's 1 024 sources are crafted, a clustered cloud follows.
    probe_overflow: sources on the mesh points of 1 024 distinct cells whose hash falls in two adjacent slots of
    the 4 096-slot table (G = 128 has 512 cells per slot): each contributes to one cell, the first 16 cells fill
    the probe window and every other one falls back to a global atomic after MAX_PROBE probes.
    one_cell: all 1 024 sources inside one cell, so the CTA's 8 192 contributions pile onto 8 table slots.
    Both against pm_np, and bitwise stable when the crafted block or the whole array is permuted."""
    G, box = 128, L
    h = box / G
    rng = np.random.default_rng(41)
    if kind == "probe_overflow":
        cells = np.arange(G ** 3, dtype=np.int64)
        s = _slot(cells).astype(np.int64)
        per_slot = np.bincount(s, minlength=4096)
        s0 = int(np.argmax(per_slot + np.roll(per_slot, -1)))
        pick = cells[(s == s0) | (s == (s0 + 1) % 4096)][:1024]
        assert len(pick) == 1024 and len(np.unique(_slot(pick))) == 2
        crafted = np.stack([pick // (G * G), (pick // G) % G, pick % G], 1) * h
    else:
        crafted = (np.array([17, 64, 101]) + rng.random((1024, 3))) * h
        crafted = np.floor(crafted * Q) / Q
    pos = np.concatenate([crafted, _cloud(30000, 42, box)]).astype(np.float32)
    mass = rng.uniform(0.5, 2.0, len(pos)).astype(np.float32)
    acc, phi = _check_vs_numpy(engine, pos, mass, G, box, 1.25 * h, kind)
    for perm in (np.concatenate([rng.permutation(1024), np.arange(1024, len(pos))]), rng.permutation(len(pos))):
        a, p = _pm(engine, _posm(pos[perm], mass[perm]), G, box, 1.25 * h)
        assert np.array_equal(a, acc[perm]) and np.array_equal(p, phi[perm])


# ---- production size -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("grid", [256, 512])
def test_pm_production_zeldovich(grid):
    """tools/pm_time.py's setup: 2^24 Zel'dovich particles (256^3, z = 49, box 100), r_s = 1.25 h.  Hilbert storage
    order (b200_spatial_order_dev) and random order give bitwise the same forces per particle; a sample of 4 096
    targets agrees with pm_np.  At G = 512 a Hilbert CTA's particles overflow the shared-memory table into global
    atomics.  The float64 restatement needs ~10 GB of host memory at G = 512."""
    import b200grav
    box, ic = 100.0, 256
    n = ic ** 3
    rs = 1.25 * box / grid
    eng = b200grav.Engine(0)
    try:
        t0 = time.perf_counter()
        posm = torch.empty((n, 4), dtype=torch.float32, device="cuda")
        vel = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        eng.zeldovich_ics_dev(posm, vel, grid=ic, box=box, origin_shift=box / 2)
        del vel
        perm = torch.empty(n, dtype=torch.int32, device="cuda")
        eng.spatial_order_dev(posm, n, box, perm)
        rnd = torch.randperm(n, device="cuda", generator=torch.Generator("cuda").manual_seed(grid))
        out = {}
        for name, order in (("hilbert", perm.long()), ("random", rnd)):
            acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
            phi = torch.empty(n, dtype=torch.float32, device="cuda")
            eng.pm_forces_dev(posm[order].contiguous(), acc, grid=grid, box=box, r_split=rs, phi=phi)
            back_a, back_p = torch.empty_like(acc), torch.empty_like(phi)
            back_a[order], back_p[order] = acc, phi
            out[name] = (back_a, back_p)
        torch.cuda.synchronize()
        t_dev = time.perf_counter() - t0
        assert torch.equal(out["hilbert"][0], out["random"][0]) and torch.equal(out["hilbert"][1], out["random"][1])
        pick = np.random.default_rng(0).choice(n, 4096, replace=False)
        a_dev = out["hilbert"][0][torch.from_numpy(pick).cuda()].cpu().numpy()
        p_dev = out["hilbert"][1][torch.from_numpy(pick).cuda()].cpu().numpy()
        host = posm.cpu().numpy().astype(np.float64)
        del out, posm
        t1 = time.perf_counter()
        a0, p0 = pm_np.pm_forces(host[:, :3], host[:, 3], host[pick, :3], grid, box, rs, potential=True)
        t_np = time.perf_counter() - t1
        ea, ep = _rel(a_dev, a0), _rel(p_dev, p0)
        print(f"pm production G={grid} n=2^24: acc {ea:.2e} phi {ep:.2e}; device part {t_dev:.1f} s, "
              f"pm_np {t_np:.1f} s")
        assert ea <= 1e-5 and ep <= 1e-5, (ea, ep)
    finally:
        eng.close()
        torch.cuda.empty_cache()


def test_pm_grid_1024_vs_ewald():
    """The largest mesh the API takes: 2^30 cells (the int cell index and the table hash at their range; ~41 GB of
    meshes and spectra plus the cuFFT workspace).  PM + the numpy short range against the Ewald sum of 256
    particles, within the 1.5 % of the G = 32 test; particles in the first and last cells included."""
    import b200grav
    G, box = 1024, 100.0
    rs = 1.25 * box / G
    rng = np.random.default_rng(51)
    pos = rng.uniform(0, box, (256, 3)).astype(np.float32)
    pos[0] = 0.0
    pos[1] = np.nextafter(np.float32(box), np.float32(0))
    pos[2] = [0.5 * box / G, box - 0.5 * box / G, 0.0]
    mass = rng.uniform(0.5, 2.0, 256).astype(np.float32)
    eng = b200grav.Engine(0)
    try:
        t0 = time.perf_counter()
        acc, _ = _pm(eng, _posm(pos, mass), G, box, rs)
        t_dev = time.perf_counter() - t0
    finally:
        eng.close()
        torch.cuda.empty_cache()
    err = _rel(acc + pm_np.short_range(pos, pos, mass, box, rs), pm_np.ewald(pos, pos, mass, box))
    print(f"pm G=1024 + short range vs Ewald: {err:.2e} (first call, plans and buffers included: {t_dev:.1f} s)")
    assert err <= 0.015, err


# ---- API edges -----------------------------------------------------------------------------------------------------

def test_pm_empty_calls(engine):
    """n_targets = 0 returns 0 and writes nothing; so does the host entry with n = 0."""
    lib, h = engine.L, engine._h
    posm = _posm(_dyadic_cloud(64, 61), np.ones(64, np.float32))
    acc = torch.full((64, 3), 7.0, device="cuda")
    phi = torch.full((64,), 7.0, device="cuda")
    for i0 in (0, 64):
        assert lib.b200_pm_forces_dev(h, posm.data_ptr(), 64, i0, 0, 32, L, 5.0, acc.data_ptr(), phi.data_ptr(),
                                      None) == 0
    torch.cuda.synchronize()
    assert bool((acc == 7.0).all()) and bool((phi == 7.0).all())
    out = np.full((4, 3), 7.0, np.float32)
    assert lib.b200_pm_forces_host(h, None, None, out.ctypes.data, 0, 32, C.c_float(L), 5.0) == 0
    assert np.all(out == 7.0)
