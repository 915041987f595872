"""-m gpu parity tests, direct sum (rows D1-D3): the CUDA path, called through
the C ABI, against the golden vectors and the CPU oracle.
Gate (BASELINE.json north_star): forces within 1e-5 relative L2."""
import numpy as np
import pytest

from conftest import golden
from inputs import masses_np, rel_l2, uniform_mt, uniform_np

pytestmark = pytest.mark.gpu
TOL = 1e-5


def test_two_body_kat(engine):
    pos = np.array([[0, 0, 0], [1, 0, 0]], np.float32)
    a = engine.direct_forces_host(pos, None, eps=0.01)
    assert abs(a[0, 0] - 0.999850035) < 2e-6 and abs(a[1, 0] + 0.999850035) < 2e-6
    assert np.all(a[:, 1:] == 0)
    # masses scale the partner's pull (the CPU leaf loop honours masses when given)
    b = engine.direct_forces_host(pos, np.array([3, 5], np.float32), eps=0.01)
    assert abs(b[0, 0] - 5 * 0.999850035) < 1e-5 and abs(b[1, 0] + 3 * 0.999850035) < 1e-5


def test_direct_golden(engine):
    g = golden("direct_768.npz")          # reference's own CPU direct sum
    a = engine.direct_forces_host(g["pos"], None, eps=0.01)
    assert rel_l2(a, g["acc"]) < TOL


@pytest.mark.parametrize("n", [1, 2, 31, 511, 512, 513, 1000, 2049, 16384])
def test_direct_vs_oracle_sizes(engine, oracle, n):
    p = uniform_mt(n, seed=100 + n % 7)
    m = masses_np(n, seed=n)
    a = engine.direct_forces_host(p, m, eps=0.01)
    want = oracle.direct_f32(p, m, eps=0.01)
    if n == 1:
        assert np.all(a == 0)
    else:
        assert rel_l2(a, want) < TOL


def test_direct_empty_and_invalid(engine):
    import b200grav
    assert engine.direct_forces_host(np.zeros((0, 3), np.float32)).shape == (0, 3)
    with pytest.raises(b200grav.B200Error):
        engine.direct_forces_host(np.zeros((4, 3), np.float32), eps=0.0)


def test_direct_duplicates_and_eps(engine, oracle):
    p = uniform_np(3000, seed=4)
    p[10:20] = p[0:10]                     # coincident pairs: softening keeps them finite
    m = masses_np(3000)
    for eps in (0.01, 0.1, 1.0):
        a = engine.direct_forces_host(p, m, eps=eps)
        assert np.isfinite(a).all()
        assert rel_l2(a, oracle.direct_f64(p, m, eps=eps)) < TOL


def test_direct_target_shard_dev(engine, oracle):
    """The multi-GPU form: targets [i0, i0+nt) against all sources."""
    import torch
    n, i0, nt = 9000, 2500, 3100
    p = uniform_mt(n, seed=5)
    m = masses_np(n, seed=6)
    posm = torch.from_numpy(np.concatenate([p, m[:, None]], 1)).cuda()
    acc = torch.empty((nt, 3), dtype=torch.float32, device="cuda")
    engine.direct_forces_dev(posm, acc, i0, nt, eps=0.01)
    torch.cuda.synchronize()
    assert rel_l2(acc.cpu().numpy(), oracle.direct_f32(p, m, eps=0.01, i0=i0, n_targets=nt)) < TOL


def test_direct_parts_equals_whole(engine):
    """Sources given as several tile-SoA parts (the peer-memory path) == one buffer."""
    import torch
    n = 5000
    p = uniform_mt(n, seed=8)
    m = masses_np(n, seed=9)
    posm = torch.from_numpy(np.concatenate([p, m[:, None]], 1)).cuda()
    whole = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.direct_forces_dev(posm, whole, 0, n, eps=0.01)
    cuts = [0, 1300, 1300, 3700, n]        # includes an empty part
    parts, lens = [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        t = torch.empty(max(engine.tiles_bytes(b - a), 16) // 4, dtype=torch.float32, device="cuda")
        engine.pack_tiles_dev(posm[a:b], b - a, t)
        parts.append(t)
        lens.append(b - a)
    out = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.direct_forces_parts_dev(parts, lens, posm, n, out, eps=0.01)
    torch.cuda.synchronize()
    assert rel_l2(out.cpu().numpy(), whole.cpu().numpy()) < 2e-6
    # the equal-mass promise: same sources with m = 2.5 everywhere
    posm[:, 3] = 2.5
    engine.direct_forces_dev(posm, whole, 0, n, eps=0.01)
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        t = torch.empty(max(engine.tiles_bytes(b - a), 16) // 4, dtype=torch.float32, device="cuda")
        engine.pack_tiles_dev(posm[a:b], b - a, t)
        parts.append(t)
    engine.direct_forces_parts_dev(parts, lens, posm, n, out, eps=0.01, all_masses_equal=True)
    torch.cuda.synchronize()
    assert rel_l2(out.cpu().numpy(), whole.cpu().numpy()) < 2e-6


def test_direct_periodic_vs_oracle(engine, oracle):
    n, box = 4000, 100.0
    p = uniform_np(n, seed=14, lo=0.0, hi=box)
    m = masses_np(n, seed=15)
    a = engine.direct_forces_host(p, m, eps=0.05, box=box)
    want = oracle.direct_periodic_f32(p, m, 0.05, box)
    # A pair separated by exactly half a box along an axis may take either image
    # (roundf(d/box) in the reference, computed with --use_fast_math there); leave
    # out the targets that have such a borderline partner.
    d = np.abs(p[:, None, :].astype(np.float64) - p[None, :, :].astype(np.float64))
    ok = ~(np.abs(d - 0.5 * box) < 2e-4).any(axis=(1, 2))
    assert ok.sum() > 0.9 * n
    assert rel_l2(a[ok], want[ok]) < TOL


def _fixed_path_n(sm, n_min):
    """The smallest n >= n_min (targets = sources = n) on the fixed-point path: direct_forces takes it when
    ceil(n / 2048) * ceil(n / 512) >= 4 * SMs (and n >= 8192, eps >= 1e-4 box)."""
    n = n_min
    while -(-n // 2048) * -(-n // 512) < 4 * sm:
        n += 1
    return n


@pytest.mark.parametrize("n,unit,eps,box", [(20000, True, 0.05, 100.0), (20000, False, 0.05, 100.0),
                                            (20000, True, 0.05, 64.0), (9000, True, 0.05, 100.0),
                                            (20000, False, 1e-3, 100.0),
                                            ("fixed", True, 0.05, 100.0), ("fixed", False, 0.05, 100.0),
                                            ("fixed", True, 0.05, 64.0), ("fixed", False, 1e-3, 100.0)])
def test_direct_periodic_both_minimum_image_paths(engine, oracle, n, unit, eps, box):
    """With eps >= 1e-4 box and at least 4 (2048-target block x 512-source tile) work units per SM (24577 particles
    on 148 SMs; "fixed" = the smallest such n + 1000) the x and y separations are taken in 32-bit fixed point (the
    wrap is the integer overflow); below either bound (9000 and 20000 particles: 400 units on 148 SMs; eps = 1e-3)
    the FP32 minimum image runs.  Same gate for both; n is never a multiple of the 512-source tile, so the padding slots are exercised too
    (equal and general masses)."""
    if n == "fixed":
        n = _fixed_path_n(engine.sm_count, 8192) + 1000
        assert n % 512
    rng = np.random.default_rng(n + int(box))
    p = rng.uniform(0.0, box, (n, 3)).astype(np.float32)
    m = np.full(n, 1.5, np.float32) if unit else masses_np(n, seed=16)
    a = engine.direct_forces_host(p, m, eps=eps, box=box)
    sel = slice(1234, 1234 + 1024)
    want = oracle.direct_periodic_f32(p, m, eps, box, i0=sel.start, n_targets=1024)
    d = np.abs(p[sel, None, :].astype(np.float64) - p[None, :, :].astype(np.float64))
    ok = ~(np.abs(d - 0.5 * box) < 2e-6 * box).any(axis=(1, 2))    # see test_direct_periodic_vs_oracle
    assert ok.sum() > 0.7 * 1024
    assert rel_l2(a[sel][ok], want[ok]) < TOL


def test_direct_periodic_nan_propagates(engine):
    """A NaN coordinate poisons every force in both minimum-image paths (the fixed-point conversion of x and y
    must not swallow it): 3000 and 20000 particles run the FP32 minimum image, the third size the fixed point."""
    rng = np.random.default_rng(3)
    for n in (3000, 20000, _fixed_path_n(engine.sm_count, 8192) + 1000):
        p = rng.uniform(0.0, 100.0, (n, 3)).astype(np.float32)
        p[n // 2, 0] = np.nan
        a = engine.direct_forces_host(p, None, eps=0.05, box=100.0)
        assert np.isnan(a).all(axis=1).sum() >= n - 1 and np.isnan(a[n // 2]).all()


def test_direct_deterministic(engine):
    p = uniform_mt(20000, seed=3)
    a = engine.direct_forces_host(p, None)
    b = engine.direct_forces_host(p, None)
    assert np.array_equal(a, b)


def test_direct_64k_vs_f64(engine, oracle):
    """Above 64 K sources the FP32 CPU loop is itself ~1e-5 from the truth, so the
    gate is taken against the FP64 oracle (subsampled targets, all sources)."""
    n = 65536
    p = uniform_mt(n, seed=42)
    a = engine.direct_forces_host(p, None)
    sel = slice(30000, 30000 + 2048)
    want = oracle.direct_f64(p, None, i0=sel.start, n_targets=2048)
    assert rel_l2(a[sel], want) < TOL


def test_direct_full_size_properties(engine, oracle):
    """BASELINE config 2 size (2^20): size-independent properties + a target sample."""
    n = 1 << 20
    p = uniform_mt(n, seed=42)
    m = masses_np(n, seed=43)
    a = engine.direct_forces_host(p, m)
    assert np.isfinite(a).all()
    # Newton's third law: sum_i m_i a_i = 0 (cancellation to ~1e-6 of sum |m a|)
    tot = (a.astype(np.float64) * m[:, None]).sum(0)
    scale = np.abs(a.astype(np.float64) * m[:, None]).sum(0)
    assert np.all(np.abs(tot) < 1e-5 * scale)
    sel = slice(777777, 777777 + 256)
    want = oracle.direct_f64(p, m, i0=sel.start, n_targets=256)
    assert rel_l2(a[sel], want) < TOL
    # linearity in the source masses: doubling every mass doubles every acceleration
    b = engine.direct_forces_host(p, 2.0 * m)
    assert rel_l2(b[::4096], 2.0 * a[::4096]) < 1e-6


def test_direct_full_size_unit_mass_sample(engine, oracle):
    """The benchmarked instance itself: 2^20 particles, all masses equal (the 11-op UNIT kernel, R = 8), a
    2048-target block against the FP64 oracle over all sources -- through the host call and through the
    target-sharded device call bench.py times."""
    import torch
    n = 1 << 20
    rng = np.random.default_rng(42)                         # bench.py's make_particles
    p = rng.uniform(-50.0, 50.0, size=(n, 3)).astype(np.float32)
    a = engine.direct_forces_host(p, np.ones(n, np.float32))
    sel = slice(349184, 349184 + 2048)
    want = oracle.direct_f64(p, None, i0=sel.start, n_targets=2048)
    assert rel_l2(a[sel], want) < TOL
    posm = torch.from_numpy(np.concatenate([p, np.ones((n, 1), np.float32)], 1)).cuda()
    acc = torch.empty((n // 8, 3), dtype=torch.float32, device="cuda")
    lo = 2 * (n // 8)                                       # rank 2 of 8
    engine.direct_forces_dev(posm, acc, lo, n // 8, eps=0.01)
    torch.cuda.synchronize()
    assert rel_l2(acc.cpu().numpy(), a[lo:lo + n // 8]) < 1e-7         # the shard of rank 2 of 8 = the same rows
