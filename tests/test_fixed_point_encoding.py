"""CPU check of the arithmetic behind the periodic direct sum's fixed-point x and y separations
(direct.cu: fixed_point(), PMODE_FIXED_XY): positions in units of box / 2^32 modulo 2^32, the upper half shifted
down by one unit; the 32-bit difference of two encodings is then the minimum-image separation.  A pair exactly half
a box apart with both positions in [0, box) keeps the sign of its raw separation, like minimum_image
(lambda_cdm_kernels.cu:122-141).  Outside [0, box) the image of a tie follows the wrapped positions and may take
either sign, and the FP32 path keeps the raw sign only when fl(1/box) box / 2 <= 1/2 (box 100 yes, box 1000 no);
test_half_box_ties_outside_the_frame pins these cases.  This restates the device function in numpy; the kernel
itself is held to float64 in tests/test_gpu_direct_edges.py and tests/test_gpu_direct.py."""
import numpy as np


def encode(x, box):
    q = np.rint(x.astype(np.float64) * (4294967296.0 / box)).astype(np.int64)      # __double2ll_rn
    e = (q & 0xFFFFFFFF).astype(np.uint32)
    return (e - (e >> np.uint32(31))).astype(np.uint32)


def separation(ej, ei, box):
    d = (ej.astype(np.int64) - ei.astype(np.int64)) & 0xFFFFFFFF
    d = np.where(d >= 1 << 31, d - (1 << 32), d)                                     # the int32 reinterpretation
    return d.astype(np.float64) * (box / 4294967296.0)


def minimum_image(d, box):                                                           # K2, :122-141
    h = 0.5 * box
    return np.where(d > h, d - box, np.where(d < -h, d + box, d))


def test_wrapped_difference_is_the_minimum_image():
    rng = np.random.default_rng(0)
    for box in (100.0, 64.0, 1.0, 737.5):
        x = rng.uniform(0.0, box, 200000).astype(np.float32)
        xi, xj = x[:100000], x[100000:]
        got = separation(encode(xj, box), encode(xi, box), box)
        want = minimum_image(xj.astype(np.float64) - xi.astype(np.float64), box)
        # one quantum of rounding per position plus the one-unit shift of the upper half
        assert np.abs(got - want).max() <= 2.01 * box / 4294967296.0


def test_half_box_pairs_keep_the_raw_sign():
    box = 100.0
    rng = np.random.default_rng(1)
    lo = rng.uniform(0.0, 50.0, 100000).astype(np.float32)
    hi = (lo + np.float32(50.0)).astype(np.float32)
    exact = hi.astype(np.float64) - lo.astype(np.float64) == 50.0                    # representable ties only
    assert exact.sum() > 10000
    lo, hi = lo[exact], hi[exact]
    up = separation(encode(hi, box), encode(lo, box), box)      # source above the target: +box/2, as K2 leaves it
    down = separation(encode(lo, box), encode(hi, box), box)    # source below: -box/2
    assert np.all(up > 0) and np.all(down < 0)
    assert np.abs(up - 50.0).max() <= 2.01 * box / 4294967296.0 and np.abs(down + 50.0).max() <= 2.01 * box / 4294967296.0


def test_out_of_box_and_self():
    box = 100.0
    x = np.array([-0.25, 0.0, 99.999992, 100.0, 150.0, -1e-6], np.float32)
    e = encode(x, box)
    assert np.all(separation(e, e, box) == 0.0)                                      # the self pair is exactly 0
    # 150 is the image of 50; -0.25 the image of 99.75
    assert abs(separation(encode(np.array([150.0], np.float32), box), encode(np.array([50.0], np.float32), box), box)[0]) < 1e-7
    assert abs(separation(e[:1], encode(np.array([99.75], np.float32), box), box)[0]) < 1e-7


def test_fp32_magic_round_is_the_minimum_image():
    """PMODE_FLOAT (and the z component of PMODE_FIXED_XY, and the tree's periodic pair rows):
    q = (d * (1/box) + 1.5*2^23) - 1.5*2^23 is rint(d / box) for |d| < box, and d - box q (one FMA) is K2's minimum
    image except for separations within a few ulps of half a box, where either image is equally near."""
    F = np.float32
    rng = np.random.default_rng(2)
    for box in (F(100.0), F(64.0), F(1.0), F(737.5)):
        xi = rng.uniform(0.0, float(box), 1_000_000).astype(F)
        xj = rng.uniform(0.0, float(box), 1_000_000).astype(F)
        d = (xj - xi).astype(F)
        ib = (F(1.0) / box).astype(F)
        magic = F(12582912.0)
        t = (d.astype(np.float64) * float(ib) + float(magic)).astype(F)              # fma.rn
        q = (t - magic).astype(F)
        got = (q.astype(np.float64) * -float(box) + d.astype(np.float64)).astype(F)  # fma.rn
        want = minimum_image(d.astype(np.float64), float(box))
        border = np.abs(np.abs(d.astype(np.float64)) - 0.5 * float(box)) < 4e-7 * float(box)
        assert np.all(np.isin(q, (-1.0, 0.0, 1.0)))
        assert np.array_equal(got[~border].astype(np.float64), want[~border].astype(F).astype(np.float64))
        assert np.all(np.abs(got[border]) <= 0.5 * float(box) * (1 + 1e-6))


def _float_path(d, box):
    """PMODE_FLOAT's minimum image of float32 separations d (see test_fp32_magic_round_is_the_minimum_image)."""
    F = np.float32
    ib, magic = (F(1.0) / F(box)).astype(F), F(12582912.0)
    q = ((d.astype(np.float64) * float(ib) + float(magic)).astype(F) - magic).astype(F)
    return (q.astype(np.float64) * -float(box) + d.astype(np.float64)).astype(F)


def test_half_box_ties_outside_the_frame():
    """What the two paths promise at an exact tie: one of the two images.  In frame the fixed-point path keeps the
    raw sign; out of frame it follows the wrapped positions; the FP32 path keeps the raw sign only when
    fl(1/box) box / 2 <= 1/2."""
    box = 100.0
    for xi, xj in ((-25.0, 25.0), (-50.0, 0.0)):
        a, b = np.array([xi], np.float32), np.array([xj], np.float32)
        assert separation(encode(b, box), encode(a, box), box)[0] < 0                   # raw +50, fixed -50
        assert _float_path((b - a).astype(np.float32), box)[0] == 50.0                  # FP32 +50
    for xi, xj in ((25.0, 75.0), (0.0, 50.0), (49.0, 99.0)):                              # in frame: raw sign on both
        a, b = np.array([xi], np.float32), np.array([xj], np.float32)
        assert separation(encode(b, box), encode(a, box), box)[0] > 0
        assert _float_path((b - a).astype(np.float32), box)[0] == 50.0
    for b, keeps in ((64.0, True), (100.0, True), (200.0, True), (3.0, False), (75.0, False), (250.0, False),
                     (500.0, False), (737.5, False), (1000.0, False)):
        h = np.array([b / 2, -b / 2], np.float32)
        got = _float_path(h, b)
        assert np.array_equal(got, h if keeps else -h), b
