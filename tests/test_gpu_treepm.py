"""-m gpu: TreePM -- the periodic short-range walk of the fixed-physics tree with a force cut-off
(b200_tree_walk_short_dev) added to the particle-mesh long range (b200_pm_forces_dev), through
Engine.treepm_forces_dev and LambdaCDMSimulation(force="treepm").  References: the float64 numpy definition
pm_np.pm_forces + treepm_np.short_range(eps, r_cut) and the Ewald sum pm_np.ewald."""
import numpy as np
import pytest
import torch

from oracle import pm_np, treepm_np

pytestmark = pytest.mark.gpu

L = 100.0
EPS = 0.01
FACTOR = 4.5


def _posm(pos, mass):
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([pos, mass[:, None]], 1), np.float32)).cuda()


def _set(kind, n, seed):
    """Uniform, or 16 Gaussian clumps (sigma = 3), in [0, L)^3; float32 positions, masses 0.5 .. 2."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        pos = rng.uniform(0, L, (n, 3))
    else:
        c = rng.uniform(0, L, (16, 3))
        pos = (c[rng.integers(0, 16, n)] + rng.normal(0, 3.0, (n, 3))) % L
    pos = pos.astype(np.float32)
    pos[pos >= L] = 0.0                                  # float32 rounding of x just below L
    return pos, rng.uniform(0.5, 2.0, n).astype(np.float32)


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))


def _treepm(engine, posm, grid, theta, i0=0, nt=None, box=L, **kw):
    nt = posm.shape[0] - i0 if nt is None else nt
    acc = torch.empty((nt, 3), dtype=torch.float32, device="cuda")
    engine.treepm_forces_dev(posm, acc, i0, nt, grid, box, theta=theta, eps=EPS, **kw)
    torch.cuda.synchronize()
    return acc


def _short(engine, posm, grid, theta, box=L):
    """The short-range walk alone, added to zeros, on a fresh fixed tree of posm."""
    n = posm.shape[0]
    rs = 1.25 * box / grid
    engine.tree_build_fixed_dev(posm, n, 8, 20, EPS)
    acc = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
    engine.tree_walk_short_dev(acc, 0, n, theta, box, rs, FACTOR * rs)
    torch.cuda.synchronize()
    return acc


def _numpy_treepm(pos, mass, tgt, grid, box=L):
    rs = 1.25 * box / grid
    x, m, t = (np.asarray(a, np.float64) for a in (pos, mass, tgt))
    return pm_np.pm_forces(x, m, t, grid, box, rs) + treepm_np.short_range(t, x, m, box, rs, eps=EPS,
                                                                        r_cut=FACTOR * rs, neighbours=True)


def _clear_of_cut(pos, r_cut, box=L):
    """Per target: no source at |r - r_cut| / r_cut < 1e-5, so FP32 rounding cannot decide whether a pair is in.
    Among 8 192^2 pairs about a hundred are that close, so the comparison samples the targets clear of them."""
    from scipy.spatial import cKDTree
    x = pm_np.wrap(np.asarray(pos, np.float64), box)
    lists = cKDTree(x, boxsize=box).query_ball_point(x, r_cut * 1.001)
    ok = np.ones(len(x), bool)
    for i, js in enumerate(lists):
        d = pm_np._min_image(x[js] - x[i], box)
        ok[i] = np.abs(np.sqrt((d * d).sum(-1)) / r_cut - 1).min() >= 1e-5
    return ok


# ---- accuracy ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind,seed", [("uniform", 11), ("clumps", 12)])
@pytest.mark.parametrize("grid", [32, 64])
def test_exact_limit_matches_numpy(engine, kind, seed, grid):
    """theta = 0 accepts no cell: the walk is the exact truncated short-range sum."""
    pos, mass = _set(kind, 8192, seed)
    rs = 1.25 * L / grid
    sample = np.flatnonzero(_clear_of_cut(pos, FACTOR * rs))
    assert len(sample) >= 0.9 * len(pos), len(sample)
    acc = _treepm(engine, _posm(pos, mass), grid, 0.0).cpu().numpy()
    err = _rel(acc[sample], _numpy_treepm(pos, mass, pos[sample], grid))
    print(f"treepm theta=0 {kind} G={grid}: {err:.2e} from numpy over {len(sample)} targets clear of r_cut")
    assert err <= 2e-5, err


@pytest.mark.parametrize("kind,seed", [("uniform", 11), ("clumps", 12)])
def test_converges_in_theta(engine, kind, seed):
    grid = 32
    pos, mass = _set(kind, 8192, seed)
    posm = _posm(pos, mass)
    ref = _numpy_treepm(pos, mass, pos, grid)
    errs = [_rel(_treepm(engine, posm, grid, th).cpu().numpy(), ref) for th in (0.7, 0.5, 0.35, 0.25)]
    print(f"treepm {kind} G={grid} error at theta 0.7 / 0.5 / 0.35 / 0.25: " + " / ".join(f"{e:.2e}" for e in errs))
    assert all(b <= a for a, b in zip(errs, errs[1:])), errs
    assert errs[1] <= 3e-3, errs


@pytest.mark.parametrize("kind", ["uniform", "clumps"])
@pytest.mark.parametrize("grid", [32, 64])
def test_against_ewald(engine, kind, grid):
    """The 2 048-particle sets of DESIGN 3.12 (unit masses, 256 targets): TreePM at theta = 0.3 within 6e-3 of
    Ewald and at most a quarter of the error of the minimum-image direct sum."""
    rng = np.random.default_rng(1)
    if kind == "uniform":
        pos = rng.uniform(0, L, (2048, 3))
    else:
        c = rng.uniform(0, L, (16, 3))
        pos = (c[rng.integers(0, 16, 2048)] + rng.normal(0, 3.0, (2048, 3))) % L
    pos = pos.astype(np.float32)
    pos[pos >= L] = 0.0
    mass = np.ones(2048, np.float32)
    x = pos.astype(np.float64)
    ew = pm_np.ewald(x[:256], x, mass, L)
    d = pm_np._min_image(x[None] - x[:256, None], L)
    r = np.sqrt((d * d).sum(-1))
    f = np.where(r > 0, 1.0 / np.where(r > 0, r, 1.0) ** 3, 0.0)
    e_direct = _rel((f[..., None] * d).sum(1), ew)
    acc = _treepm(engine, _posm(pos, mass), grid, 0.3, 0, 256).cpu().numpy()
    err = _rel(acc, ew)
    print(f"treepm theta=0.3 {kind} G={grid}: {err:.2e} from Ewald; minimum-image direct sum {e_direct:.2e}")
    assert err <= 6e-3 and err <= 0.25 * e_direct, (err, e_direct)


@pytest.mark.parametrize("grid", [256])
def test_production_zeldovich(grid):
    """2^24 Zel'dovich particles (256^3, z = 49, box 100) in Hilbert storage order, G = 256.  At theta = 0 a sample
    of 4 096 targets is within 2e-5 of the float64 definition (neighbour-list oracle); at theta = 0.5, 0.35, 0.25
    there is no NaN and the error falls with theta.
    theta = 0.5 is not held to a 3e-3 bound here: it measures 7.9e-3 on a B200.  Near-uniform initial conditions make
    the short-range sum cancel 44-fold (sum of |terms| over |sum|), and theta = 0.5 is the first opening angle at
    which the lowest cells (edge about 2.5 particle spacings) become monopoles inside r_cut = 2.2: the short-range
    error is 7e-6 of the total at theta = 0.25, 4e-4 at 0.35 and 7.9e-3 at 0.5 (DESIGN 3.12)."""
    import b200grav
    box, ic = 100.0, 256
    n = ic ** 3
    eng = b200grav.Engine(0)
    try:
        posm = torch.empty((n, 4), dtype=torch.float32, device="cuda")
        vel = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        eng.zeldovich_ics_dev(posm, vel, grid=ic, box=box, origin_shift=box / 2)
        del vel
        perm = torch.empty(n, dtype=torch.int32, device="cuda")
        eng.spatial_order_dev(posm, n, box, perm)
        posm = posm[perm.long()].contiguous()
        del perm
        pick = torch.from_numpy(np.random.default_rng(0).choice(n, 4096, replace=False)).cuda()
        got = {}
        for theta in (0.0, 0.5, 0.35, 0.25):
            acc = _treepm(eng, posm, grid, theta, box=box)
            assert not torch.isnan(acc).any(), theta
            got[theta] = acc[pick].cpu().numpy()
            del acc
        host = posm.cpu().numpy().astype(np.float64)
        del posm
        ref = _numpy_treepm(host[:, :3], host[:, 3], host[pick.cpu().numpy(), :3], grid, box)
        err = {theta: _rel(a, ref) for theta, a in got.items()}
        print(f"treepm production G={grid} n=2^24 vs the numpy theta = 0 definition: " +
              " / ".join(f"theta {t} {e:.2e}" for t, e in err.items()))
        assert err[0.0] <= 2e-5, err
        assert err[0.25] <= err[0.35] <= err[0.5], err
    finally:
        eng.close()
        torch.cuda.empty_cache()


# ---- physics ------------------------------------------------------------------------------------------------------

def test_short_range_momentum(engine):
    pos, mass = _set("clumps", 8192, 21)
    a = _short(engine, _posm(pos, mass), 64, 0.0).cpu().numpy().astype(np.float64)
    tot = np.abs((mass[:, None] * a).sum(0)).max()
    scale = (mass * np.linalg.norm(a, axis=1)).sum()
    print(f"short-range momentum: |sum m a| / sum m |a| = {tot / scale:.2e}")
    assert tot <= 1e-5 * scale


def test_uniform_lattice_feels_no_force(engine):
    """L = 128, G = 64, one particle per cell at even integer coordinates: every separation is exact in FP32."""
    box, grid = 128.0, 64
    h = box / grid
    g = np.arange(grid, dtype=np.float32) * np.float32(h)
    pos = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    mass = np.ones(len(pos), np.float32)
    acc = _treepm(engine, _posm(pos, mass), grid, 0.0, box=box).cpu().numpy()
    worst = np.abs(acc).max()
    print(f"lattice: max |a| = {worst:.2e} (pair force at h: {1 / h ** 2:.2e})")
    assert worst <= 1e-5 / h ** 2, worst


def test_cutoff_prunes(engine):
    """theta = 0, N = 2^16 uniform, G = 64: the pair interactions are at most 1 % of N^2 (r_cut = 4.5 r_s is 0.3 %
    of the volume), and the walk visits fewer nodes and issues fewer pair slots than the periodic fixed walk."""
    n, grid = 1 << 16, 64
    pos, mass = _set("uniform", n, 31)
    posm = _posm(pos, mass)
    rs = 1.25 * L / grid
    engine.tree_set_counting(True)
    try:
        engine.tree_build_fixed_dev(posm, n, 8, 20, EPS)
        acc = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
        engine.tree_walk_short_dev(acc, 0, n, 0.0, L, rs, FACTOR * rs)
        short = engine.tree_walk_stats().astype(np.float64)
        engine.tree_set_periodic(L)
        engine.tree_walk_dev(acc, 0, n, 0.0)
        full = engine.tree_walk_stats().astype(np.float64)
    finally:
        engine.tree_set_periodic(0.0)
        engine.tree_set_counting(False)
    print(f"theta=0 N=2^16 G=64: short walk visits {short[0]:.3e}, pair interactions {short[2] / n ** 2:.2%} of N^2, "
          f"pair slots {short[3] / n ** 2:.2%} of N^2; periodic walk visits {full[0]:.3e}, pairs "
          f"{full[2] / n ** 2:.2%}")
    assert short[2] <= 0.01 * n * n
    assert short[0] < full[0] and short[3] < full[3]


# ---- determinism and state ----------------------------------------------------------------------------------------

def test_split_targets_concatenate_bitwise(engine):
    pos, mass = _set("clumps", 20000, 41)
    posm = _posm(pos, mass)
    one = _treepm(engine, posm, 32, 0.5)
    a = _treepm(engine, posm, 32, 0.5, 0, 7001)
    b = _treepm(engine, posm, 32, 0.5, 7001, 20000 - 7001)
    assert torch.equal(torch.cat([a, b]), one)


def test_short_walk_adds_exactly(engine):
    pos, mass = _set("uniform", 20000, 42)
    posm = _posm(pos, mass)
    grid = 32
    rs = 1.25 * L / grid
    both = _treepm(engine, posm, grid, 0.5)
    short = _short(engine, posm, grid, 0.5)
    pm = torch.empty_like(short)
    engine.pm_forces_dev(posm, pm, 0, posm.shape[0], grid, L, rs)
    torch.cuda.synchronize()
    assert torch.equal(short + pm, both)


def test_other_walks_unchanged_by_treepm(engine):
    """The short walk neither reads nor changes the b200_tree_set_periodic state."""
    pos, mass = _set("clumps", 20000, 43)
    posm = _posm(pos, mass)
    n = posm.shape[0]

    def walk():
        engine.tree_build_fixed_dev(posm, n, 8, 20, EPS)
        acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        engine.tree_walk_dev(acc, 0, n, 0.5)
        torch.cuda.synchronize()
        return acc

    try:
        for box in (L, 0.0):
            engine.tree_set_periodic(box)
            before = walk()
            _treepm(engine, posm, 32, 0.5)
            assert torch.equal(walk(), before), box
    finally:
        engine.tree_set_periodic(0.0)


def test_argument_checks(engine):
    import b200grav
    pos, mass = _set("uniform", 4096, 44)
    posm = _posm(pos, mass)
    n = posm.shape[0]
    acc = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
    fresh = b200grav.Engine(0)
    try:
        with pytest.raises(b200grav.B200Error, match="status 3"):          # no tree
            fresh.tree_walk_short_dev(acc, 0, n, 0.5, L, 4.0, 18.0)
        fresh.tree_build_dev(posm, n, L, 8, 20)                              # the reference-faithful tree
        with pytest.raises(b200grav.B200Error, match="status 3"):
            fresh.tree_walk_short_dev(acc, 0, n, 0.5, L, 4.0, 18.0)
    finally:
        fresh.close()
    engine.tree_build_fixed_dev(posm, n, 8, 20, EPS)
    bad = [(L, 0.0, 18.0), (L, -1.0, 18.0), (L, float("nan"), 18.0), (L, 4.0, 0.0), (L, 4.0, L / 2),
           (L, 4.0, 60.0), (0.0, 4.0, 18.0), (-L, 4.0, 18.0), (L, 4.0, float("nan"))]
    for box, rs, rc in bad:
        with pytest.raises(b200grav.B200Error, match="status 1"):
            engine.tree_walk_short_dev(acc, 0, n, 0.5, box, rs, rc)
    with pytest.raises(b200grav.B200Error, match="status 1"):               # targets beyond the tree
        engine.tree_walk_short_dev(acc, 1, n, 0.5, L, 4.0, 18.0)
    with pytest.raises(b200grav.B200Error, match="status 1"):               # G = 8 with r_s = 1.25 h: r_cut = 0.70 L
        engine.treepm_forces_dev(posm, acc, 0, n, 8, L)
    acc.fill_(3.0)
    engine.tree_walk_short_dev(acc, 0, 0, 0.5, L, 4.0, 18.0)
    engine.tree_walk_short_dev(None, 0, 0, 0.5, L, 4.0, 18.0)
    torch.cuda.synchronize()
    assert bool((acc == 3.0).all())


# ---- driver -------------------------------------------------------------------------------------------------------

def test_kdk_matches_numpy(engine):
    """LambdaCDMSimulation(force="treepm"): 4096 particles in clumps, G = 32, theta = 0, three KDK steps against a
    numpy KDK on the numpy TreePM forces (a = 1 throughout: h = 0 switches the expansion off).  Softening 1.0 keeps
    the comparison well conditioned: a 6e-8 relative change of the initial positions (FP32 rounding) moves the
    float64 result by 7e-6 here, against 0.12 at eps = 0.01, where close encounters amplify any rounding."""
    import b200grav
    G, n, dt, steps, eps = 32, 4096, 0.2, 3, 1.0
    pos, mass = _set("clumps", n, 51)
    vel = np.zeros((n, 3), np.float32)
    sim = b200grav.LambdaCDMSimulation(engine, pos, vel, mass, box=L, force="treepm", pm_grid=G, theta=0.0, eps=eps,
                                       a0=1.0, cosmo=(0.31, 0.0, 0.69, 0.0))
    for _ in range(steps):
        sim.step(dt)
    rs = 1.25 * L / G
    x = pos.astype(np.float64)
    v = vel.astype(np.float64)

    def forces(x):
        return pm_np.pm_forces(x, mass, x, G, L, rs) + treepm_np.short_range(x, x, mass, L, rs, eps=eps,
                                                                         r_cut=FACTOR * rs, neighbours=True)

    a = forces(x)
    for _ in range(steps):
        v += 0.5 * dt * a
        x = pm_np.wrap(x + dt * v, L)
        a = forces(x)
        v += 0.5 * dt * a
    d = sim.positions().astype(np.float64) - x
    d -= L * np.round(d / L)
    moved = np.abs(pm_np.wrap(x - pos + L / 2, L) - L / 2)
    print(f"treepm KDK: median move {np.median(moved):.2e}, max position difference {np.abs(d).max():.2e}")
    assert np.median(moved) > 10 * 1e-4 * L, np.median(moved)        # the particles went somewhere
    assert np.abs(d).max() <= 1e-4 * L, np.abs(d).max()
