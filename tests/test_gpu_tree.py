"""-m gpu parity tests, Barnes-Hut path (rows T1-T6).  Gates: Morton keys, sort
permutation and tree topology BIT-EXACT; forces within 1e-3 relative L2 at equal
theta / leaf capacity (north_star)."""
import numpy as np
import pytest

from conftest import golden
from inputs import clustered_np, masses_np, rel_l2, uniform_mt, uniform_np

pytestmark = pytest.mark.gpu
TOL_TREE = 1e-3
TREE_KEYS = ("level", "center", "size", "first_child", "part_off", "part_idx", "mass", "com")


def _posm(p, m):
    import torch
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([p, m[:, None]], 1), np.float32)).cuda()


def _build_export(engine, p, m, **kw):
    import torch
    posm = _posm(p, m)
    engine.tree_build_dev(posm, p.shape[0], **kw)
    torch.cuda.synchronize()
    return posm, engine.tree_export()


def test_morton_keys_bit_exact(engine, oracle):
    import torch
    g = golden("zeldovich_4096.npz")
    r = golden("random_2048.npz")
    for pos, keys in ((g["pos_box"], g["keys"]), (r["pos"], r["keys"])):
        posm = _posm(pos, np.ones(len(pos), np.float32))
        out = torch.empty(len(pos), dtype=torch.int32, device="cuda")
        engine.morton_keys_dev(posm, len(pos), 100.0, out)
        assert np.array_equal(out.cpu().numpy().view(np.uint32), keys)
    p = uniform_np(200000, seed=31, lo=-80.0, hi=180.0)      # outside the box: wraps
    p[:6] = [[0, 0, 0], [100, 100, 100], [50, 50, 50], [99.99999, 0, 0], [-0.0, 25, 12.5], [100.0, -100.0, 200.0]]
    posm = _posm(p, np.ones(len(p), np.float32))
    out = torch.empty(len(p), dtype=torch.int32, device="cuda")
    engine.morton_keys_dev(posm, len(p), 100.0, out)
    assert np.array_equal(out.cpu().numpy().view(np.uint32), oracle.morton_keys(p, 100.0))


@pytest.mark.parametrize("n,hi", [(1, 10), (2, 1), (255, 4), (4096, 1 << 30), (4097, 7), (100000, 1 << 30), (1 << 20, 1 << 10)])
def test_sort_permutation_bit_exact(engine, oracle, n, hi):
    import torch
    rng = np.random.default_rng(n)
    keys = rng.integers(0, hi, size=n, dtype=np.int64).astype(np.uint32)
    kin = torch.from_numpy(keys.view(np.int32)).cuda()
    kout = torch.empty_like(kin)
    perm = torch.empty(n, dtype=torch.int32, device="cuda")
    engine.sort_pairs_dev(kin, n, kout, perm)
    sk, sp = oracle.sort_pairs(keys)
    assert np.array_equal(kout.cpu().numpy().view(np.uint32), sk)
    assert np.array_equal(perm.cpu().numpy(), sp)
    assert np.array_equal(kin.cpu().numpy().view(np.uint32), keys)      # input untouched


@pytest.mark.parametrize("name", ["tree_centred_4096.npz", "tree_box_3000.npz", "tree_clustered_2500.npz"])
def test_tree_golden_topology_and_forces(engine, name):
    g = golden(name)                      # the reference's own tree, dumped node for node
    kw = dict(box=float(g["box"]), leaf_cap=int(g["leaf_cap"]), max_depth=int(g["max_depth"]))
    posm, t = _build_export(engine, g["pos"], g["mass"], **kw)
    for k in TREE_KEYS:
        assert np.array_equal(t[k], g["t_" + k]), k
    st = engine.tree_stats()
    assert (st["n_nodes"], st["n_leaves"], st["depth"]) == tuple(int(x) for x in g["stats"])
    a = engine.tree_forces_host(g["pos"], g["mass"], theta=float(g["theta"]), **kw)
    assert rel_l2(a, g["acc"]) < TOL_TREE
    assert rel_l2(a, g["acc"]) < 1e-5     # same interaction lists => only round-off differs


def test_tree_stats_kat(engine):
    p = uniform_mt(16384)
    _build_export(engine, p, np.ones(16384, np.float32))
    st = engine.tree_stats()
    assert (st["n_nodes"], st["n_leaves"], st["depth"]) == (4793, 4194, 6)


@pytest.mark.parametrize("cap,depth", [(8, 20), (1, 20), (3, 4), (8, 0), (64, 20), (8, 1)])
def test_tree_edge_cases_bit_exact(engine, oracle, cap, depth):
    p = uniform_np(6000, seed=12)
    p[100:130] = p[0:30]
    p[200:230, 0] = 0.0
    p[230:260] = np.array([12.5, -25.0, 6.25], np.float32)
    p[300:340] *= 1.3
    m = masses_np(6000, seed=13)
    _, t = _build_export(engine, p, m, box=100.0, leaf_cap=cap, max_depth=depth)
    o = oracle.tree_build(p, m, leaf_cap=cap, max_depth=depth)
    for k in TREE_KEYS + ("arrivals",):
        assert np.array_equal(t[k], getattr(o, k)), k


def test_tree_graph_replay_shallow_deep_shallow(engine, oracle):
    """The build graph runs the levels a uniform tree never reaches only through IF nodes armed on the device
    (tree.cu: arm_deep_levels_kernel).  One cached graph (same buffers, sizes, parameters) is replayed on a shallow
    tree, on a 21-level one (the [0, box) convention: an eighth of the particles pile up in one corner chain) and on a
    shallow one again: every build must be the reference's tree, and the forces of the last must not see leftovers
    of the deep build."""
    import torch
    n = 40000
    shallow = uniform_np(n, seed=77)
    deep = uniform_np(n, seed=78, lo=0.0, hi=100.0)
    m = np.ones(n, np.float32)
    posm = _posm(shallow, m)
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    depths = []
    for pos in (shallow, deep, shallow):
        posm[:, :3] = torch.from_numpy(pos).cuda()
        engine.tree_build_dev(posm, n, 100.0, 8, 20)           # same pointer, n, parameters: the cached graph
        torch.cuda.synchronize()
        t = engine.tree_export()
        o = oracle.tree_build(pos, m)
        for k in TREE_KEYS:
            assert np.array_equal(t[k], getattr(o, k)), k
        depths.append(engine.tree_stats()["depth"])
        engine.tree_walk_dev(acc, 0, n, theta=0.5)
        torch.cuda.synchronize()
        ref = oracle.tree_forces(o, pos, 0.5, i0=0, n_targets=2048)
        assert rel_l2(acc[:2048].cpu().numpy(), ref) < TOL_TREE
    assert depths[0] < 12 and depths[1] == 21 and depths[2] == depths[0]


@pytest.mark.parametrize("gen", ["uniform", "box", "clustered"])
def test_tree_forces_and_counters_vs_oracle(engine, oracle, gen):
    import torch
    n = 50000
    if gen == "uniform":
        p = uniform_mt(n, seed=11)
    elif gen == "box":
        p = uniform_np(n, seed=12, lo=0.0, hi=100.0)        # what the reference generators emit
    else:
        p = clustered_np(n, seed=13)
    m = masses_np(n, seed=14)
    posm, t = _build_export(engine, p, m, box=100.0, leaf_cap=8, max_depth=20)
    o = oracle.tree_build(p, m)
    for k in TREE_KEYS:
        assert np.array_equal(t[k], getattr(o, k)), k
    engine.tree_set_counting(True)
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.tree_walk_dev(acc, 0, n, theta=0.5)
    torch.cuda.synchronize()
    cnt = engine.tree_counters()
    engine.tree_set_counting(False)
    want, ocnt = oracle.tree_forces(o, p, 0.5, counters=True)
    assert np.array_equal(cnt, ocnt), (cnt, ocnt)      # identical accept/open decisions
    assert rel_l2(acc.cpu().numpy(), want) < 1e-5
    # sharded walk == rows of the full walk
    part = torch.empty((7000, 3), dtype=torch.float32, device="cuda")
    engine.tree_walk_dev(part, 20000, 7000, theta=0.5)
    torch.cuda.synchronize()
    assert np.array_equal(part.cpu().numpy(), acc[20000:27000].cpu().numpy())


def test_tree_theta_zero_is_leaf_direct(engine, oracle):
    """theta = 0 never accepts a cell: the walk degenerates to unit-mass pair sums
    over the particles that are in leaves (orphans are not sources -- quirk T6)."""
    n = 3000
    p = uniform_mt(n, seed=2)
    m = masses_np(n)
    a = engine.tree_forces_host(p, m, theta=0.0)
    o = oracle.tree_build(p, m)
    assert rel_l2(a, oracle.tree_forces(o, p, 0.0)) < 1e-5
    big = engine.tree_forces_host(p, m, theta=0.5, leaf_cap=n + 1)    # one root leaf = direct sum
    assert rel_l2(big, oracle.direct_f32(p, None)) < 1e-5


def test_tree_full_size(engine, oracle):
    """BASELINE config 3 size: 2^20 particles, theta 0.5, leaf 8; topology bit-exact,
    forces on a target sample, node statistics."""
    import torch
    n = 1 << 20
    p = uniform_mt(n, seed=42)
    m = np.ones(n, np.float32)
    posm, t = _build_export(engine, p, m, box=100.0, leaf_cap=8, max_depth=20)
    o = oracle.tree_build(p, m)
    for k in TREE_KEYS:
        assert np.array_equal(t[k], getattr(o, k)), k
    assert int(t["part_off"][-1]) == n and np.array_equal(np.sort(t["part_idx"]), np.arange(n))
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.tree_walk_dev(acc, 0, n, theta=0.5)
    torch.cuda.synchronize()
    a = acc.cpu().numpy()
    assert np.isfinite(a).all()
    want = oracle.tree_forces(o, p, 0.5, i0=500000, n_targets=20000)
    assert rel_l2(a[500000:520000], want) < TOL_TREE


def test_tree_c4_size_16m(engine, oracle):
    """BASELINE config 4 size: 2^24 particles.  Topology, COM and masses bit-exact against the oracle's build
    (6.7 M nodes), forces on two target samples (one of them the last particles), and one fused kick-kick-drift of
    all 2^24 particles bit-exact against the oracle's leapfrog with the walk's accelerations."""
    import torch
    n = 1 << 24
    p = uniform_mt(n, seed=42)
    m = np.ones(n, np.float32)
    posm, t = _build_export(engine, p, m, box=100.0, leaf_cap=8, max_depth=20)
    o = oracle.tree_build(p, m)
    for k in TREE_KEYS:
        assert np.array_equal(t[k], getattr(o, k)), k
    assert int(t["part_off"][-1]) == n
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.tree_walk_dev(acc, 0, n, theta=0.5)
    torch.cuda.synchronize()
    a = acc.cpu().numpy()
    assert np.isfinite(a).all()
    for i0, cnt in ((5000000, 4096), (n - 2048, 2048)):
        want = oracle.tree_forces(o, p, 0.5, i0=i0, n_targets=cnt)
        assert rel_l2(a[i0:i0 + cnt], want) < TOL_TREE
    vel = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
    dt = np.float32(1e-4)
    engine.leapfrog_dev(posm, vel, acc, n, 2, dt * np.float32(0.5), 1.0, dt, 0.0)
    torch.cuda.synchronize()
    vo, po = np.zeros((n, 3), np.float32), p.copy()
    oracle.kick(vo, a, m, dt * np.float32(0.5), 1.0)
    oracle.kick(vo, a, m, dt * np.float32(0.5), 1.0)
    oracle.drift(po, vo, dt, 0.0)
    assert np.array_equal(vel.cpu().numpy(), vo)
    assert np.array_equal(posm[:, :3].cpu().numpy(), po)


def test_tree_zeldovich_c3(engine, oracle):
    """BASELINE config 3 scale: Zel'dovich initial conditions (grid 128 -> 2^20 particles, seed 12345, z = 49,
    box 100) from the engine's own generator (b200_zeldovich_ics_dev, held to oracle/ics_np.py by
    test_gpu_ics.py), shifted to the centred convention."""
    import torch
    n = 1 << 20
    ics = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    engine.zeldovich_ics_dev(ics, torch.empty((n, 3), dtype=torch.float32, device="cuda"), n_particles=n, grid=128,
                             box=100.0, z_initial=49.0, seed=12345)
    torch.cuda.synchronize()
    zp, zm = np.ascontiguousarray(ics[:, :3].cpu().numpy()), np.ascontiguousarray(ics[:, 3].cpu().numpy())
    del ics
    p = (zp - np.float32(50.0)).astype(np.float32)
    posm, t = _build_export(engine, p, zm, box=100.0, leaf_cap=8, max_depth=20)
    o = oracle.tree_build(p, zm)
    for k in TREE_KEYS:
        assert np.array_equal(t[k], getattr(o, k)), k
    engine.tree_set_counting(True)
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.tree_walk_dev(acc, 0, n, theta=0.5)
    torch.cuda.synchronize()
    engine.tree_set_counting(False)
    want = oracle.tree_forces(o, p, 0.5, i0=300000, n_targets=30000)
    assert rel_l2(acc[300000:330000].cpu().numpy(), want) < TOL_TREE
    # Morton keys of the generator's box-convention output, bit-exact
    keys = torch.empty(n, dtype=torch.int32, device="cuda")
    engine.morton_keys_dev(_posm(zp, zm), n, 100.0, keys)
    assert np.array_equal(keys.cpu().numpy().view(np.uint32), oracle.morton_keys(zp, 100.0))


def test_spatial_order_is_a_local_permutation(engine):
    """b200_spatial_order_dev: a permutation of the particles along a Hilbert curve -- consecutive particles
    are close in space (every step of a Hilbert curve moves to a face-adjacent lattice cell)."""
    import torch
    n = 200000
    pos = uniform_mt(n, seed=77)
    posm = torch.from_numpy(np.concatenate([pos, np.ones((n, 1), np.float32)], 1)).cuda()
    perm = torch.empty(n, dtype=torch.int32, device="cuda")
    engine.spatial_order_dev(posm, n, 100.0, perm)
    torch.cuda.synchronize()
    p = perm.cpu().numpy()
    assert np.array_equal(np.sort(p), np.arange(n))
    step = np.abs(np.diff(pos[p], axis=0)).sum(1)
    rand = np.abs(np.diff(pos, axis=0)).sum(1)
    assert step.mean() < 0.04 * rand.mean()                  # ~2 vs ~100 (L1 distance between neighbours)
    assert np.percentile(step, 99.9) < 15.0                  # no long jumps: a Morton curve would have 50-unit ones
