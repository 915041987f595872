"""-m gpu: block (hierarchical) time steps of the comoving TreePM integration (DESIGN 3.14) -- the sync-point pass
b200_block_kick_dev and the active short walk b200_tree_walk_short_active_dev against their numpy and device
definitions bit for bit, ComovingSimulation(max_bins=...) against the parent's global step (bitwise) and against the
float64 oracle scheme (oracle/blockstep_np.py), its efficiency at equal accuracy, and the Layzer-Irvine equation."""
import numpy as np
import pytest
import torch

import b200grav
from oracle import blockstep_np as bs
from oracle import comoving_np

pytestmark = pytest.mark.gpu

L = 100.0
LCDM = (0.31, 0.0, 0.69)


def _set(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        pos = rng.uniform(0, L, (n, 3))
    else:
        c = rng.uniform(0, L, (16, 3))
        pos = (c[rng.integers(0, 16, n)] + rng.normal(0, 3.0, (n, 3))) % L
    pos = pos.astype(np.float32)
    pos[pos >= L] = 0.0
    mass = np.full(n, 3 * LCDM[0] * L ** 3 / (8 * np.pi * n), np.float32)
    return pos, rng.normal(0, 0.05, (n, 3)).astype(np.float32), mass


def _bits(t):
    """Bit patterns of a float32 array, every NaN as the one quiet NaN (the device and numpy set different NaN
    payloads)."""
    a = np.array(t.cpu().numpy() if torch.is_tensor(t) else t, np.float32)
    a[np.isnan(a)] = np.nan
    return a.view(np.uint32)


# ---- 1. bitwise reduction to the global step -------------------------------------------------------------------------

def _parent_run(engine, pos, mom, mass, a_grid, G, theta, eps):
    """The global comoving KDK step of ComovingSimulation before block steps, from Engine calls."""
    dev = torch.device("cuda")
    f32 = lambda x: torch.as_tensor(x, dtype=torch.float32, device=dev)
    posm = torch.cat([f32(pos).reshape(-1, 3), f32(mass).reshape(-1, 1)], 1).contiguous()
    mom = f32(mom).reshape(-1, 3).clone()
    n = posm.shape[0]
    acc = torch.zeros((n, 3), dtype=torch.float32, device=dev)
    rs = 1.25 * L / G
    forces = lambda: engine.treepm_forces_dev(posm, acc, 0, n, G, L, rs, theta=theta, eps=eps)
    forces()
    for a0, a1 in zip(a_grid[:-1], a_grid[1:]):
        am = np.sqrt(a0 * a1)
        drift, _ = engine.comoving_kdk_factors(a0, a1, *LCDM)
        _, k0 = engine.comoving_kdk_factors(a0, am, *LCDM)
        _, k1 = engine.comoving_kdk_factors(am, a1, *LCDM)
        engine.leapfrog_dev(posm, mom, acc, n, 1, np.float32(k0), 1.0, np.float32(drift), L)
        forces()
        engine.leapfrog_dev(posm, mom, acc, n, 1, np.float32(k1), 1.0, 0.0, L)
    torch.cuda.synchronize()
    return posm, mom, acc


def _check_reduction(engine, pos, mom, mass, a_grid, G, theta, eps):
    ref = _parent_run(engine, pos, mom, mass, a_grid, G, theta, eps)
    for max_bins, eta in ((1, 0.025), (5, 1e30)):
        sim = b200grav.ComovingSimulation(engine, pos, mom, mass, L, a_grid[0], force="treepm", pm_grid=G,
                                          theta=theta, eps=eps, cosmo=LCDM, max_bins=max_bins, eta=eta)
        for a in a_grid[1:]:
            sim.step(a)
        torch.cuda.synchronize()
        assert sim.bin_counts[0] == sim.n, sim.bin_counts
        for name, got, want in (("posm", sim.posm, ref[0]), ("mom", sim.mom, ref[1]), ("acc", sim.acc, ref[2])):
            assert np.array_equal(_bits(got), _bits(want)), (max_bins, name)


@pytest.mark.parametrize("kind", ["uniform", "clumps"])
def test_reduces_to_global_step_bitwise(engine, kind):
    """max_bins = 1, and max_bins = 5 with every particle in bin 0 (eta = 1e30): posm, mom and acc bit-equal to the
    global step; 8 192 particles, G = 32, three steps."""
    pos, mom, mass = _set(kind, 8192, 5)
    _check_reduction(engine, pos, mom, mass, np.geomspace(0.3, 0.36, 4), 32, 0.5, 0.01)


def test_reduces_to_global_step_bitwise_production(engine):
    """The same at 2^24 Zel'dovich particles (256^3, z = 49), G = 256, two steps."""
    pos, mom, mass, a0 = b200grav.comoving_zeldovich_dev(engine, grid=256, box=L, z_initial=49.0, seed=3)
    _check_reduction(engine, pos, mom, mass, np.geomspace(a0, 0.025, 3), 256, 0.5, 0.01)


# ---- 2. the sync-point pass against numpy -----------------------------------------------------------------------------

def _pass_inputs(n, max_bins, seed):
    rng = np.random.default_rng(seed)
    scale = lambda: np.exp(rng.normal(0, 2, (n, 1)))
    d = dict(mass=rng.uniform(0.5, 2, n).astype(np.float32), mom=rng.normal(0, 1, (n, 3)).astype(np.float32),
             acc=(rng.normal(0, 1, (n, 3)) * scale()).astype(np.float32),
             acc_long=(rng.normal(0, 1, (n, 3)) * scale()).astype(np.float32),
             acc_short=(rng.normal(0, 1, (n, 3)) * scale()).astype(np.float32),
             bins=rng.integers(0, max_bins, n).astype(np.uint8))
    if n > 8:
        d["acc"][:4] = [[0, 0, 0], [np.inf, 0, 0], [np.nan, 1, 1], [1e30, 1e30, 0]]
        d["acc_short"][4:6] = [[0, 0, 0], [np.nan, 0, 0]]
    fac = np.random.default_rng(seed + 1).uniform(1e-3, 2e-2, 2 * (2 ** max_bins - 1)).astype(np.float32)
    return d, fac


@pytest.mark.parametrize("n", [1, 3, 1023, 1024, 4097, 2 ** 20 + 3])
def test_sync_pass_matches_numpy_bitwise(engine, n):
    """Every k in 0..S for max_bins = 1, 3 and 6 on random bins, with and without the drift: positions, mom, acc,
    bins and the histogram bit-equal to blockstep_np.sync_pass32; rows of zero, infinite and NaN accelerations
    included (NaNs compared as NaNs)."""
    dev = torch.device("cuda")
    for max_bins in (1, 3, 6):
        d, fac = _pass_inputs(n, max_bins, 17 + max_bins)
        pos = np.random.default_rng(n).uniform(0, L, (n, 3)).astype(np.float32)
        dfac = torch.from_numpy(fac).to(dev)
        gl, gs = torch.from_numpy(d["acc_long"]).to(dev), torch.from_numpy(d["acc_short"]).to(dev)
        hist = torch.zeros(16, dtype=torch.int32, device=dev)
        dlna, crit = 0.3, np.float32(0.05)
        for k in range(2 ** (max_bins - 1) + 1):
            posm = torch.from_numpy(np.concatenate([pos, d["mass"][:, None]], 1)).to(dev)
            mom, acc = torch.from_numpy(d["mom"]).to(dev), torch.from_numpy(d["acc"]).to(dev)
            bins = torch.from_numpy(d["bins"]).to(dev)
            drift = np.float32(0.37 if k % 2 == 0 and k < 2 ** (max_bins - 1) else 0.0)      # drifting and not
            engine.block_kick_dev(posm, mom, acc, gl, gs, bins, n, k, max_bins, dfac, crit, dlna, hist, drift, L)
            em, ea, eb, eh, ep = bs.sync_pass32(k, max_bins, d["mass"], d["mom"], d["acc"], d["acc_long"],
                                                d["acc_short"], d["bins"], fac, crit, dlna, pos, drift, L)
            assert np.array_equal(_bits(posm[:, :3]), _bits(ep)), (max_bins, k, "pos")
            assert np.array_equal(_bits(mom), _bits(em)), (max_bins, k, "mom")
            assert np.array_equal(_bits(acc), _bits(ea)), (max_bins, k, "acc")
            assert np.array_equal(bins.cpu().numpy(), eb), (max_bins, k, "bins")
            assert np.array_equal(hist.cpu().numpy(), eh), (max_bins, k, "hist")


def test_sync_pass_errors(engine):
    n = 64
    dev = torch.device("cuda")
    z3 = lambda: torch.zeros((n, 3), dtype=torch.float32, device=dev)
    posm = torch.ones((n, 4), dtype=torch.float32, device=dev)
    mom, acc, gl, gs = z3(), z3(), z3(), z3()
    bins = torch.zeros(n, dtype=torch.uint8, device=dev)
    fac = torch.full((2 * 15,), 1e-3, dtype=torch.float32, device=dev)
    hist = torch.zeros(16, dtype=torch.int32, device=dev)
    p = lambda t: t.data_ptr()
    call = lambda **kw: engine.L.b200_block_kick_dev(
        engine._h, kw.get("posm", p(posm)), kw.get("mom", p(mom)), kw.get("acc", p(acc)), p(gl), p(gs),
        kw.get("bins", p(bins)), n, kw.get("k", 0), kw.get("mb", 4), kw.get("fac", p(fac)), kw.get("crit", 1.0),
        kw.get("dlna", 0.1), kw.get("hist", p(hist)), kw.get("drift", 0.0), L, None)
    assert call() == 0 and call(k=8) == 0
    for kw in (dict(mb=0), dict(mb=17), dict(k=-1), dict(k=9), dict(posm=None), dict(mom=None), dict(acc=None),
               dict(bins=None), dict(fac=None), dict(hist=None), dict(mom=p(mom) + 4), dict(posm=p(posm) + 8),
               dict(crit=-1.0), dict(crit=float("nan")), dict(dlna=float("inf")), dict(dlna=-0.1),
               dict(drift=float("nan")), dict(k=8, drift=0.1)):
        assert call(**kw) == 1, kw
    assert engine.L.b200_block_kick_dev(None, p(posm), p(mom), p(acc), p(gl), p(gs), p(bins), n, 0, 4, p(fac), 1.0,
                                        0.1, p(hist), 0.0, L, None) == 1


# ---- 3. the active short walk ---------------------------------------------------------------------------------------------

def test_active_walk_matches_full_walk(engine):
    """Rows of the active particles equal b200_tree_walk_short_dev over [0, n) bit for bit, inactive rows poisoned
    with NaN stay NaN, n_active equals the numpy filter and the histogram's prediction; empty and full lists."""
    pos, _, mass = _set("clumps", 8192, 23)
    n, G, mb = len(pos), 32, 4
    rs = 1.25 * L / G
    posm = torch.from_numpy(np.concatenate([pos, mass[:, None]], 1)).cuda()
    engine.tree_build_fixed_dev(posm, n, 8, 20, 0.01)
    ref = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
    engine.tree_walk_short_dev(ref, 0, n, 0.5, L, rs, 4.5 * rs)
    ref = ref.cpu().numpy()
    rng = np.random.default_rng(4)
    cases = [(rng.integers(0, mb, n), k) for k in range(9)]
    cases += [(np.zeros(n, np.int64), 3), (np.zeros(n, np.int64), 8), (np.full(n, 3), 5)]    # empty, full, full
    for b, k in cases:
        bins = torch.from_numpy(b.astype(np.uint8)).cuda()
        out = torch.full((n, 3), float("nan"), dtype=torch.float32, device="cuda")
        na = engine.tree_walk_short_active_dev(bins, n, k, mb, 0.5, L, rs, 4.5 * rs, out)
        act = k % (1 << (mb - 1 - b)) == 0
        counts = np.bincount(b, minlength=16)
        predicted = sum(counts[q] for q in range(mb) if k % (1 << (mb - 1 - q)) == 0)
        o = out.cpu().numpy()
        assert na == act.sum() == predicted, (k, na, act.sum(), predicted)
        assert np.array_equal(_bits(o[act]), _bits(ref[act])), k
        assert np.isnan(o[~act]).all(), k
    bins = torch.zeros(n, dtype=torch.uint8, device="cuda")
    out = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
    c = engine.L.b200_tree_walk_short_active_dev
    import ctypes as C
    na = C.c_size_t()
    args = lambda **kw: (engine._h, kw.get("bins", bins.data_ptr()), kw.get("n", n), kw.get("k", 0), kw.get("mb", mb),
                         0.5, L, rs, kw.get("rc", 4.5 * rs), kw.get("out", out.data_ptr()),
                         kw.get("na", C.byref(na)), None)
    assert c(*args()) == 0 and na.value == n
    for kw in (dict(mb=0), dict(mb=17), dict(k=9), dict(k=-1), dict(bins=None), dict(out=None), dict(na=None),
               dict(rc=0.5 * L)):
        assert c(*args(**kw)) == 1, kw
    assert c(*args(n=n - 1)) == 3
    fresh = b200grav.Engine(0)
    assert c(*((fresh._h,) + args()[1:])) == 3
    fresh.close()
    engine.tree_build_dev(posm, n, L, 8, 20)                            # the reference-faithful tree
    assert c(*args()) == 3


# ---- 4. the scheme against the float64 oracle ------------------------------------------------------------------------

def _pairs_set(eps):
    """A 16^3 lattice background (forces nearly cancel: bin 0) and 12 tight pairs at cell centres on near-circular
    orbits, separated so that the criterion puts them mid-way into bins 1, 2 and 3 (dlna^2 / crit = 1/2 below)."""
    g = 16
    q = (np.arange(g) + 0.5) * L / g
    lat = np.stack(np.meshgrid(q, q, q, indexing="ij"), -1).reshape(-1, 3)
    n_pairs = 12
    m = 3 * LCDM[0] * L ** 3 / (8 * np.pi * (len(lat) + 2 * n_pairs))
    rng = np.random.default_rng(8)
    cells = rng.choice(g ** 3, n_pairs, replace=False)
    pos, mom = [lat], [np.zeros_like(lat)]
    a0 = 0.5
    for i, c in enumerate(cells):
        b = 1 + i % 3
        gmag = 2.0 * 4.0 ** (b - 0.5)
        d = np.sqrt(m / gmag)
        centre = lat[c] + 0.5 * L / g
        u = rng.normal(size=3); u /= np.linalg.norm(u)
        w = np.cross(u, rng.normal(size=3)); w /= np.linalg.norm(w)
        v = 0.5 * np.sqrt(2 * a0 * m / d)                   # each member: half the relative circular speed
        pos.append(np.stack([centre + 0.5 * d * u, centre - 0.5 * d * u]))
        mom.append(np.stack([v * w, -v * w]))
    pos = np.concatenate(pos) % L
    return pos, np.concatenate(mom), np.full(len(pos), m), a0


def test_scheme_matches_oracle(engine):
    """theta = 0, max_bins = 4, three PM steps a = 0.5 -> 0.56: the GPU bins equal the oracle's at the end, and
    positions agree to 1e-5, momenta to 1e-3 (measured on a B200: 1.1e-6 and 4.2e-4, DESIGN 3.14).  The oracle's criterion margin (distance of log4(dlna^2 |g| / crit)
    from an integer at every rebinning) is asserted, so no bin can flip under rounding."""
    eps, G = 0.01, 32
    pos, mom, mass, a0 = _pairs_set(eps)
    a_grid = np.geomspace(a0, 0.56, 4)
    dlna = np.log(a_grid[1] / a_grid[0])
    eta = 2 * dlna * dlna / (eps * bs.crit_of(a0, 1.0, 1.0))             # dlna^2 / crit = 1/2 at a0
    rs = 1.25 * L / G
    margins = []

    def rec(k, a, bins, x):
        xf = x[np.isfinite(x) & (x > -0.5)]
        if len(xf):
            margins.append(np.abs(xf - np.round(xf)).min())
    ref = bs.scheme(pos, mom, mass, L, a_grid, 4, bs.treepm_forces(mass, L, G, rs, eps, 4.5 * rs), eta=eta, eps=eps,
                    record=rec)
    sim = b200grav.ComovingSimulation(engine, pos.astype(np.float32), mom, mass, L, a0, force="treepm", pm_grid=G,
                                      theta=0.0, eps=eps, cosmo=LCDM, max_bins=4, eta=eta)
    for a in a_grid[1:]:
        sim.step(a)
    x, p = sim.positions().astype(np.float64), sim.momenta().astype(np.float64)
    dx = x - ref[0]
    dx -= L * np.round(dx / L)
    ex = np.linalg.norm(dx) / np.linalg.norm(ref[0])
    ep = np.linalg.norm(p - ref[1]) / np.linalg.norm(ref[1])
    print(f"block scheme vs oracle: x {ex:.2e}, p {ep:.2e}; bins {np.bincount(ref[2], minlength=4)}, "
          f"smallest criterion margin {min(margins):.3f}")
    assert min(margins) >= 0.05, min(margins)
    assert np.array_equal(sim.bins.cpu().numpy(), ref[2])
    assert set(np.unique(ref[2])) == {0, 1, 2, 3}
    assert ex <= 1e-5 and ep <= 1e-3, (ex, ep)


def test_invalid_settings(engine):
    pos, mom, mass = _set("uniform", 64, 1)
    for kw in (dict(force="pm", max_bins=2), dict(max_bins=0), dict(max_bins=17), dict(eta=0.0), dict(eta=-1.0)):
        with pytest.raises(ValueError):
            b200grav.ComovingSimulation(engine, pos, mom, mass, L, 0.5, **kw)


# ---- 5. efficiency at equal accuracy, 6. Layzer-Irvine ------------------------------------------------------------------

def _evolved(engine, grid, a_end, n_steps, pm_grid, seed=7):
    pos, mom, mass, a0 = b200grav.comoving_zeldovich_dev(engine, grid=grid, box=L, z_initial=49.0, seed=seed)
    sim = b200grav.ComovingSimulation(engine, pos, mom, mass, L, a0, force="treepm", pm_grid=pm_grid, theta=0.5,
                                      eps=0.02, cosmo=LCDM)
    for a in np.geomspace(a0, a_end, n_steps + 1)[1:]:
        sim.step(a)
    return sim.positions(), sim.momenta(), mass


def test_efficiency_at_equal_accuracy(engine):
    """64^3 Zel'dovich particles evolved to a = 0.6; then one PM step of dln a = 0.02 (the criterion puts most
    particles in bins 0 and 1 there; at dln a = 0.1 it put 94 % in bin 3, which saves nothing): block steps
    (max_bins = 4), global steps of that size and of an eighth of it, all against 32 global steps.  The block error
    is at most half the coarse global error, with at most half the short-range target evaluations of the fine
    global run."""
    pos, mom, mass = _evolved(engine, 64, 0.6, 60, 64)
    a0 = 0.6
    a1 = a0 * np.exp(0.02)

    def run(n_steps, max_bins):
        sim = b200grav.ComovingSimulation(engine, pos, mom, mass, L, a0, force="treepm", pm_grid=64, theta=0.5,
                                          eps=0.02, cosmo=LCDM, max_bins=max_bins)
        sim.short_targets = 0
        for a in np.geomspace(a0, a1, n_steps + 1)[1:]:
            sim.step(a)
        return sim.positions().astype(np.float64), sim.short_targets, sim.bin_counts
    xr = run(32, 1)[0]

    def err(x):
        d = x - xr
        d -= L * np.round(d / L)
        return np.sqrt((d * d).sum(1).mean())
    xb, tb, hb = run(1, 4)
    x1, t1, _ = run(1, 1)
    x8, t8, _ = run(8, 1)
    eb, e1, e8 = err(xb), err(x1), err(x8)
    print(f"block (max_bins 4): err {eb:.3e}, short targets {tb}, bins {hb[:4]}; global dlna: err {e1:.3e}, "
          f"{t1}; global dlna/8: err {e8:.3e}, {t8}")
    assert eb <= 0.5 * e1, (eb, e1)
    assert tb <= 0.5 * t8, (tb, t8)


def test_layzer_irvine_block_steps(engine):
    """The 128^3 run of test_gpu_comoving (TreePM, theta = 0.5) taken to a = 1 with a quarter of its late PM steps
    (20 from a = 0.1) and max_bins = 3: I(a) = a (K + W) + int K da stays within 2 % of |W(a = 1)|."""
    pos, mom, mass, a0 = b200grav.comoving_zeldovich_dev(engine, grid=128, box=L, z_initial=49.0, seed=7)
    sim = b200grav.ComovingSimulation(engine, pos, mom, mass, L, a0, force="treepm", pm_grid=128, theta=0.5,
                                      eps=0.02, cosmo=LCDM, max_bins=3)
    del pos, mom
    grid_a = np.concatenate([np.geomspace(a0, 0.1, 25), np.geomspace(0.1, 1.0, 21)[1:]])
    k_, w_ = sim.energies()
    ks, ws, As = [k_], [w_], [a0]
    for a in grid_a[1:]:
        sim.step(a)
        k_, w_ = sim.energies()
        ks.append(k_); ws.append(w_); As.append(a)
    assert not engine.tree_overflowed()
    As, ks, ws = np.array(As), np.array(ks), np.array(ws)
    cumk = np.concatenate([[0.0], np.cumsum(0.5 * (ks[1:] + ks[:-1]) * np.diff(As))])
    I = As * (ks + ws) + cumk
    dev = np.abs(I - I[0]).max() / abs(ws[-1])
    print(f"Layzer-Irvine, max_bins 3, 20 late steps: max |I - I0| / |W(1)| = {dev:.2e}; bins at a = 1 "
          f"{sim.bin_counts[:3]}, short targets {sim.short_targets}")
    assert dev <= 0.02, dev
