"""CPU checks of oracle/direct_np.py, the float64 direct sum that tests/test_gpu_direct_edges.py holds the kernels to:
against the C oracle (open float64, periodic float32, energy), Newton's third law, whole-period shifts, the two-body
known answer and the two tie rules."""
import numpy as np
import pytest

from inputs import masses_np, rel_l2, uniform_np
from oracle import direct_np


def _dyadic(n, seed, box, q=1024.0):
    rng = np.random.default_rng(seed)
    return (np.floor(rng.uniform(0.0, box, (n, 3)) * q) / q).astype(np.float32)


def test_open_matches_c_float64(oracle):
    p, m = uniform_np(1500, seed=1), masses_np(1500, seed=2)
    for eps in (0.01, 0.5):
        want = oracle.direct_f64(p, m, eps=float(np.float32(eps)))      # the kernels' eps is a float
        got = direct_np.forces(p, m, eps)
        assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    t = np.array([0, 7, 1499])
    assert np.array_equal(direct_np.forces(p, m, 0.01, targets=t), direct_np.forces(p, m, 0.01)[t])


@pytest.mark.parametrize("box", [100.0, 64.0, 737.5])
def test_periodic_matches_c_float32_tie_free(oracle, box):
    n = 2000
    p = np.random.default_rng(3).uniform(0.0, box, (n, 3)).astype(np.float32)
    p = p[[t.size == 0 for t in direct_np.tie_partners(p, box)]]    # float32 ties do happen (box 64)
    m = masses_np(p.shape[0], seed=4)
    assert p.shape[0] > 0.99 * n and all(t.size == 0 for t in direct_np.tie_partners(p, box))
    got = direct_np.forces(p, m, 0.05, box)
    assert rel_l2(oracle.direct_periodic_f32(p, m, 0.05, box), got) < 1e-5
    # the two tie rules only differ at ties
    assert np.array_equal(got, direct_np.forces(p, m, 0.05, box, ties="flip"))


@pytest.mark.parametrize("box", [0.0, 100.0])
def test_potential_matches_c_energy(oracle, box):
    n = 1500
    p = np.random.default_rng(5).uniform(0.0, 100.0, (n, 3)).astype(np.float32)
    p[20:25] = p[0:5]                                              # coincident pairs count m_j / eps
    m = masses_np(n, seed=6)
    phi = direct_np.potential(p, m, 0.05, box)
    assert np.all(phi > 0)
    _, pe = oracle.energy(p, np.zeros_like(p), m, 0.05, box)
    assert abs(-0.5 * float((m.astype(np.float64) * phi).sum()) - pe) <= 1e-6 * abs(pe)


def test_periodic_newton_third_law_with_ties():
    """sum_i m_i a_i = 0 with every particle a target, planted half-box pairs included (both rules are odd in d)."""
    box, n = 64.0, 600
    p = _dyadic(n, 7, box)
    p[1::2, 0] = np.mod(p[0::2, 0] + np.float32(box / 2), box)      # every other particle ties with its neighbour
    m = masses_np(n, seed=8)
    assert sum(t.size > 0 for t in direct_np.tie_partners(p, box)) >= n
    for ties in ("raw", "flip"):
        a = direct_np.forces(p, m, 0.05, box, ties=ties)
        ma = a * m[:, None]
        assert np.all(np.abs(ma.sum(0)) <= 1e-12 * np.abs(ma).sum(0))


def test_periodic_whole_period_shifts_are_exact():
    box, n = 64.0, 500
    p = _dyadic(n, 9, box)
    p = p[[t.size == 0 for t in direct_np.tie_partners(p, box)]]
    m = masses_np(p.shape[0], seed=10)
    a0, phi0 = direct_np.forces(p, m, 0.05, box), direct_np.potential(p, m, 0.05, box)
    k = np.random.default_rng(11).integers(-3, 4, p.shape)
    q = (p + k * box).astype(np.float32)
    assert np.array_equal(q.astype(np.float64) - k * box, p)       # the shift itself is exact
    assert np.array_equal(direct_np.forces(q, m, 0.05, box), a0)
    assert np.array_equal(direct_np.potential(q, m, 0.05, box), phi0)


def test_two_body_known_answer():
    want = 1.0 / (1.0 + float(np.float32(0.01)) ** 2) ** 1.5      # 0.999850035...
    p = np.array([[0, 0, 0], [1, 0, 0]], np.float32)
    for box, q in ((0.0, p), (100.0, p), (100.0, np.array([[0.5, 3, 3], [99.5, 3, 3]], np.float32))):
        a = direct_np.forces(q, np.array([3.0, 5.0], np.float32), 0.01, box)
        s = -1.0 if q[1, 0] > 50 else 1.0                           # 99.5 is the image of -0.5
        assert np.allclose(a, [[5 * s * want, 0, 0], [-3 * s * want, 0, 0]], rtol=1e-15, atol=0)
        phi = direct_np.potential(q, np.array([3.0, 5.0], np.float32), 0.01, box)
        assert np.allclose(phi, [5 / np.sqrt(1 + float(np.float32(0.01)) ** 2), 3 / np.sqrt(1 + float(np.float32(0.01)) ** 2)],
                           rtol=1e-15)


def test_tie_rules():
    box = 100.0
    d = np.array([50.0, -50.0, 150.0, -150.0, 250.0, 49.999996, 0.0, 100.0])
    assert np.array_equal(direct_np.minimum_image(d, box, "raw"), [50, -50, 50, -50, 50, 49.999996, 0, 0])
    assert np.array_equal(direct_np.minimum_image(d, box, "flip"), [-50, 50, -50, 50, -50, 49.999996, 0, 0])
    p = np.array([[25, 1, 1], [75, 2, 2], [-25, 3, 3], [10, 4, 4]], np.float32)
    t = direct_np.tie_partners(p, box)
    assert [list(x) for x in t] == [[1, 2], [0], [0], []]           # 75 and -25 are one box apart
    # a tie pair: the two rules give opposite x forces of the same size, the other axes agree
    ar, af = (direct_np.forces(p[:2], None, 0.01, box, ties=r) for r in ("raw", "flip"))
    assert ar[0, 0] > 0 and af[0, 0] == -ar[0, 0] and np.array_equal(ar[:, 1:], af[:, 1:])
    with pytest.raises(ValueError):
        direct_np.minimum_image(d, box, "nearest")
