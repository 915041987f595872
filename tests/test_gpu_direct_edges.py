"""-m gpu: every direct-sum kernel instance at the edges of its dispatch rule and at production size, against the
float64 restatement oracle/direct_np.py (open forces: the C oracle's float64 loop).

direct_forces / direct_potential (csrc/direct.cu) pick the instance from n_targets, the source tile count, eps, box
and the SM count; _force_instance / _potential_instance below restate that rule, every shape is derived from the
device's SM count, and test_every_instance_is_reached runs this file's case lists through the rule.  Each force
instance exists in an equal-mass (UNIT, chosen on the device) and a general-mass version.

Gates: forces 1e-5 relative L2 against float64, potential 2e-6 max relative (test_gpu_direct.py, test_gpu_energy.py).
Also here: the production periodic configuration's route (bitwise), the half-box tie contract of both periodic
paths, frame and whole-period invariance (bitwise, dyadic input), mass and coordinate edges, non-finite inputs on
every path, shard sums of the energy and the multi-part (peer-memory) source path."""
import numpy as np
import pytest
import torch

from inputs import rel_l2
from oracle import direct_np

pytestmark = pytest.mark.gpu

TOL = 1e-5
POT_TOL = 2e-6
TILE = 512
SM = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
FIXED_ENV = {"B200_DIRECT_VARIANT": "4,512,1"}             # periodic: the fixed-point x/y instance, R4 x 512
FLOAT_ENV = {"B200_DIRECT_PERIODIC_FLOAT": "1"}            # periodic: the FP32 minimum image only


# ---- the dispatch rule, restated -------------------------------------------------------------------------------------

def _tiles(ns):
    return -(-ns // TILE)


def _force_instance(nt, tiles, eps, box, sm=SM, force_float=False):
    units = -(-nt // 2048) * tiles
    small = nt < 4 * 2048 or units < 4 * sm
    if box == 0:
        return "OPEN_R2" if small else "OPEN_R8"
    fixed_ok = np.float32(eps) >= np.float32(np.float32(1e-4) * np.float32(box)) and not small and not force_float
    return "FIXED_R4" if fixed_ok else ("FLOAT_R2" if small else "FLOAT_R4")


def _potential_instance(nt, tiles, box, sm=SM):
    small = nt < 4 * 1536 or -(-nt // 1536) * tiles < 4 * sm
    if box == 0:
        return "OPEN_R2" if small else "OPEN_R6"
    return "PER_R2" if small else "PER_R4"


def _first_not_small(block, sm=SM):
    """Smallest n (targets = sources = n) whose call is not "small"."""
    n = 4 * block
    while -(-n // block) * _tiles(n) < 4 * sm:
        n += 1
    return n


NS_LO, NS_HI = TILE * (SM - 1), TILE * (SM - 1) + 1       # SM - 1 and SM source tiles: 4 x tiles straddles 4 SM
N_F = _first_not_small(2048)                              # 24577 on 148 SMs
N_P = _first_not_small(1536)                              # 21505 on 148 SMs
N_PAD = TILE * (SM + 2)                                   # + 1 / + 511: one or 511 live slots in the last tile


# ---- helpers ---------------------------------------------------------------------------------------------------------

def _posm(pos, mass):
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([pos, np.asarray(mass, np.float32)[:, None]], 1),
                                                 np.float32)).cuda()


def _forces(engine, posm, i0, nt, eps, box):
    acc = torch.empty((nt, 3), dtype=torch.float32, device="cuda")
    engine.direct_forces_dev(posm, acc, i0, nt, eps=eps, box=box)
    torch.cuda.synchronize()
    return acc.cpu().numpy()


def _potential(engine, posm, i0, nt, eps, box):
    phi = torch.empty(nt, dtype=torch.float32, device="cuda")
    engine.direct_potential_dev(posm, phi, i0, nt, eps=eps, box=box)
    torch.cuda.synchronize()
    return phi.cpu().numpy()


def _with_env(monkeypatch, env):
    for k in ("B200_DIRECT_VARIANT", "B200_DIRECT_PERIODIC_FLOAT"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _sample(i0, nt, k, seed=0):
    """Up to k target indices in [i0, i0 + nt): both ends, every block edge of 512 / 1024 / 1536 / 2048, the rest
    random."""
    edges = {i0, i0 + nt - 1}
    for b in (512, 1024, 1536, 2048):
        for e in range(b, nt, b):
            edges.update((i0 + e - 1, i0 + e))
    edges = sorted(edges)
    edges = sorted(set(edges[:: max(1, 2 * len(edges) // k)]) | {i0, i0 + nt - 1})
    rest = np.random.default_rng(seed).choice(np.arange(i0, i0 + nt), min(nt, k) - len(edges), replace=False)
    return np.unique(np.concatenate([edges, rest]).astype(np.int64))


def _want_forces(oracle, pos, mass, eps, box, idx):
    if box == 0:
        return _open_rows(oracle, pos, mass, eps, idx)
    return direct_np.forces(pos, mass, eps, box, targets=idx)


def _open_rows(oracle, pos, mass, eps, idx):
    """Float64 open forces of arbitrary rows, via contiguous runs of the C oracle."""
    out = np.empty((idx.size, 3))
    runs = np.split(np.arange(idx.size), np.nonzero(np.diff(idx) != 1)[0] + 1)
    for r in runs:
        out[r] = oracle.direct_f64(pos, mass, eps=float(np.float32(eps)), i0=int(idx[r[0]]), n_targets=r.size)
    return out


def _cloud(n, box, seed):
    """Open: uniform in [-50, 50).  Periodic: the tie-free dyadic cloud below.  A random float32 cloud has pairs
    within a rounding of half a box, where the FP32 separation may round onto the tie and take the other image
    than float64 does; the dyadic one has exact separations at least 1 / Q away from every tie."""
    if box > 0:
        return _tie_free_cloud(n, box, seed)
    return np.random.default_rng(seed).uniform(-50.0, 50.0, (n, 3)).astype(np.float32)


def _mass(n, unit, seed):
    return np.full(n, 1.5, np.float32) if unit else np.random.default_rng(seed).uniform(0.5, 1.5, n).astype(np.float32)


# ---- 1. every instance against float64 -------------------------------------------------------------------------------
# (name, n_sources, i0, n_targets, eps, box); each runs with equal and with general masses.  Periodic inputs lie in
# [0, box) and are free of half-box ties (_cloud).

FORCE_CASES = [
    ("open_8191_lo", NS_LO, 0, 8191, 0.01, 0.0),
    ("open_8192_lo", NS_LO, 0, 8192, 0.01, 0.0),
    ("open_8191_hi", NS_HI, 0, 8191, 0.01, 0.0),
    ("open_8192_hi", NS_HI, NS_HI - 8192, 8192, 0.01, 0.0),
    ("per_8191_lo", NS_LO, 0, 8191, 0.05, 100.0),
    ("per_8192_lo", NS_LO, 0, 8192, 0.05, 100.0),
    ("per_8191_hi", NS_HI, 0, 8191, 0.05, 100.0),
    ("per_8192_hi", NS_HI, NS_HI - 8192, 8192, 0.05, 100.0),
    ("float_8192_hi", NS_HI, 3, 8192, 1e-3, 100.0),
    ("open_first_not_small_m1", N_F - 1, 0, N_F - 1, 0.01, 0.0),
    ("open_first_not_small", N_F, 0, N_F, 0.01, 0.0),
    ("per_first_not_small_m1", N_F - 1, 0, N_F - 1, 0.05, 100.0),
    ("per_first_not_small", N_F, 0, N_F, 0.05, 100.0),
    ("float_first_not_small", N_F, 0, N_F, 1e-3, 100.0),
    ("open_pad1", N_PAD + 1, 777, 9000, 0.01, 0.0),
    ("open_pad511", N_PAD + 511, 1535, 9000, 0.01, 0.0),
    ("fixed_pad1_box64", N_PAD + 1, 2047, 9000, 0.05, 64.0),
    ("fixed_pad511", N_PAD + 511, 1023, 9000, 0.05, 100.0),
    ("float_pad1_box64", N_PAD + 1, 513, 9000, 1e-3, 64.0),
    ("float_pad511", N_PAD + 511, 1, 9000, 1e-3, 100.0),
    ("float_r2_pad1_box64", N_PAD + 1, 1000, 3000, 0.05, 64.0),
]


@pytest.mark.parametrize("unit", [True, False], ids=["unit", "general"])
@pytest.mark.parametrize("case", FORCE_CASES, ids=[c[0] for c in FORCE_CASES])
def test_force_instance_vs_float64(engine, oracle, monkeypatch, case, unit):
    name, ns, i0, nt, eps, box = case
    _with_env(monkeypatch, {})
    pos, mass = _cloud(ns, box, len(name)), _mass(ns, unit, ns)
    a = _forces(engine, _posm(pos, mass), i0, nt, eps, box)
    idx = _sample(i0, nt, 512 if ns <= 65536 else 384)
    want = _want_forces(oracle, pos, mass, eps, box, idx)
    err = rel_l2(a[idx - i0], want)
    print(f"{name} {'unit' if unit else 'general'} {_force_instance(nt, _tiles(ns), eps, box)}: {err:.2e}")
    assert np.isfinite(a).all() and err < TOL


@pytest.mark.parametrize("box", [0.0, 100.0])
def test_one_target_against_two_to_the_20(engine, oracle, monkeypatch, box):
    """nt = 1: one target block spread over every CTA, the finalize pass adds one record per CTA."""
    _with_env(monkeypatch, {})
    n = 1 << 20
    pos, mass = _cloud(n, box, 5), _mass(n, False, 6)
    posm = _posm(pos, mass)
    i = 654321
    a1 = _forces(engine, posm, i, 1, 0.01, box)
    full = _forces(engine, posm, 0, n, 0.01, box)
    want = _want_forces(oracle, pos, mass, 0.01, box, np.array([i]))
    assert rel_l2(a1, want) < TOL and rel_l2(a1, full[i:i + 1]) < 1e-6


# ---- 2. the production periodic configuration's route ---------------------------------------------------------------

@pytest.fixture(scope="module")
def production():
    n = 1 << 20
    pos = _tie_free_cloud(n, 100.0, 42)
    idx = _sample(0, n, 256, seed=1)
    return pos, idx


def test_production_periodic_route(engine, monkeypatch, production):
    """2^20 particles in [0, 100), eps = 0.01: fl(0.01) == fl(1e-4f * 100), so the fixed-point path is taken on the
    equality; one float below it the FP32 minimum image runs."""
    pos, idx = production
    n = pos.shape[0]
    posm = _posm(pos, np.ones(n, np.float32))
    assert np.float32(0.01) == np.float32(np.float32(1e-4) * np.float32(100.0))
    assert _force_instance(n, _tiles(n), 0.01, 100.0) == "FIXED_R4"
    _with_env(monkeypatch, {})
    dflt = _forces(engine, posm, 0, n, 0.01, 100.0)
    _with_env(monkeypatch, FIXED_ENV)
    fixed = _forces(engine, posm, 0, n, 0.01, 100.0)
    _with_env(monkeypatch, FLOAT_ENV)
    flt = _forces(engine, posm, 0, n, 0.01, 100.0)
    assert np.array_equal(dflt, fixed) and not np.array_equal(dflt, flt)
    want = direct_np.forces(pos, None, 0.01, 100.0, targets=idx)
    e_fixed, e_float = rel_l2(fixed[idx], want), rel_l2(flt[idx], want)
    print(f"production FIXED_R4 {e_fixed:.2e} FLOAT_R4 {e_float:.2e}")
    assert e_fixed < TOL and e_float < TOL
    below = float(np.nextafter(np.float32(0.01), np.float32(0)))
    assert _force_instance(n, _tiles(n), below, 100.0) == "FLOAT_R4"
    _with_env(monkeypatch, {})
    b_dflt = _forces(engine, posm, 0, n, below, 100.0)
    _with_env(monkeypatch, FLOAT_ENV)
    assert np.array_equal(b_dflt, _forces(engine, posm, 0, n, below, 100.0))


def test_production_float_r4_small_eps(engine, monkeypatch, production):
    pos, idx = production
    n = pos.shape[0]
    m = _mass(n, False, 3)
    _with_env(monkeypatch, {})
    assert _force_instance(n, _tiles(n), 1e-3, 100.0) == "FLOAT_R4"
    a = _forces(engine, _posm(pos, m), 0, n, 1e-3, 100.0)
    err = rel_l2(a[idx], direct_np.forces(pos, m, 1e-3, 100.0, targets=idx))
    print(f"production FLOAT_R4 general eps 1e-3: {err:.2e}")
    assert err < TOL


# ---- 3./4. half-box ties and frame invariance ------------------------------------------------------------------------

Q = 1024.0      # positions on a 1 / Q grid
TIE_TOL = 3e-5  # per target, relative


def _tie_free_cloud(n, box, seed):
    """Dyadic positions in [0, box), tie free on every axis and under any whole-period shift: grid indices are even
    in [0, box / 2) and odd in [box / 2, box), while box / 2 is an even number of grid steps."""
    assert (box / 2 * Q) % 2 == 0
    rng = np.random.default_rng(seed)
    k = rng.integers(0, int(box * Q) // 2, (n, 3)) * 2
    k = np.where(k >= box / 2 * Q, k + 1, k)
    return (k / Q).astype(np.float32)


def _centred(pos, box):
    return np.where(pos >= box / 2, pos - np.float32(box), pos).astype(np.float32)


def _planted_ties(n, box, seed, n_pairs=32, heavy=1000.0):
    """A tie-free cloud plus n_pairs light targets, each exactly half a box (on x) from one heavy partner and from
    nothing else.  Returns pos, mass, target indices."""
    pos = _tie_free_cloud(n, box, seed)
    mass = np.ones(n, np.float32)
    rng = np.random.default_rng(seed + 1)
    used = set(np.round(pos[:, 0] * Q).astype(np.int64).tolist())
    free = [k for k in range(0, int(box * Q) // 2, 2) if k not in used and k + int(box / 2 * Q) not in used]
    ks = rng.choice(free, n_pairs, replace=False)
    tgt = np.arange(0, 2 * n_pairs, 2) + 100
    pos[tgt, 0] = ks / Q                                    # light target, in the lower half
    pos[tgt + 1, 0] = ks / Q + box / 2                      # its heavy partner, in the upper half
    mass[tgt + 1] = heavy
    return pos, mass, tgt


@pytest.mark.parametrize("box", [64.0, 100.0, 1000.0])
def test_half_box_ties_take_one_of_the_two_images(engine, oracle, monkeypatch, box):
    """A tie resolves to one of the two images on both periodic paths, in frame and in the origin-centred frame; in
    frame at box 64 and 100 it keeps the raw sign on both (fixed point: in-frame encoding; FP32: fl(1/box) box / 2
    <= 1/2 there)."""
    n = N_F
    pos, mass, tgt = _planted_ties(n, box, int(box))
    partners = direct_np.tie_partners(pos, box, tgt)
    assert all(list(p) == [t + 1] for p, t in zip(partners, tgt))
    for frame in ("in", "centred"):
        p = pos if frame == "in" else _centred(pos, box)
        raw = direct_np.forces(p, mass, 0.05, box, targets=tgt, ties="raw")
        flip = direct_np.forces(p, mass, 0.05, box, targets=tgt, ties="flip")
        gap = np.linalg.norm(raw - flip, axis=1) / np.linalg.norm(raw, axis=1)
        assert gap.min() > 100 * TIE_TOL
        for path, env in (("fixed", FIXED_ENV), ("float", FLOAT_ENV)):
            _with_env(monkeypatch, env)
            a = _forces(engine, _posm(p, mass), 0, n, 0.05, box)[tgt].astype(np.float64)
            e_raw = np.linalg.norm(a - raw, axis=1) / np.linalg.norm(raw, axis=1)
            e_flip = np.linalg.norm(a - flip, axis=1) / np.linalg.norm(flip, axis=1)
            assert np.all(np.minimum(e_raw, e_flip) < TIE_TOL), (frame, path)
            if frame == "in" and box in (64.0, 100.0):
                assert np.all(e_raw < TIE_TOL), (frame, path)
            print(f"ties box {box} {frame} {path}: raw sign kept for {int((e_raw < TIE_TOL).sum())}/{tgt.size}, "
                  f"max error {np.minimum(e_raw, e_flip).max():.2e}")


def test_frame_and_period_invariance_bitwise(engine, monkeypatch):
    """Tie-free dyadic input at box 64: FP32 separations and the fixed-point encoding (taken modulo 2^32) are exact,
    so shifting any particle by whole periods, or writing the origin-centred frame, changes no bit."""
    box, n = 64.0, N_F
    pos = _tie_free_cloud(n, box, 7)
    mass = _mass(n, False, 8)
    k = np.random.default_rng(9).integers(-3, 4, (n, 3)).astype(np.float32)
    shifted = (pos + k * np.float32(box)).astype(np.float32)
    assert np.array_equal(shifted - k * np.float32(box), pos)
    for env in (FIXED_ENV, FLOAT_ENV):
        _with_env(monkeypatch, env)
        a0 = _forces(engine, _posm(pos, mass), 0, n, 0.05, box)
        for q in (shifted, _centred(pos, box)):
            assert np.array_equal(_forces(engine, _posm(q, mass), 0, n, 0.05, box), a0), env


# ---- 5. masses -------------------------------------------------------------------------------------------------------

N_MASS = TILE * (SM - 1) + 300                            # SM tiles, the last holding 300 sources


def _mass_case(kind, n):
    m = np.full(n, 1.5, np.float32)
    if kind == "differs_first":
        m[0] = 2.0
    elif kind == "differs_last":
        m[-1] = 2.0
    elif kind == "differs_in_last_tile":
        m[n - 150] = 0.5
    elif kind == "negative_equal":
        m[:] = -1.5
    elif kind == "signed_zero_total":
        m[0::2], m[1::2] = 1.0, -1.0
        m[-1] = 0.0 if n % 2 else m[-1]
    elif kind == "ratio_1e4":
        m = np.where(np.random.default_rng(1).random(n) < 0.5, 1.0, 1e4).astype(np.float32)
    return m


@pytest.mark.parametrize("box", [0.0, 100.0], ids=["open_r8", "fixed_r4"])
@pytest.mark.parametrize("kind", ["differs_first", "differs_last", "differs_in_last_tile", "negative_equal",
                                  "signed_zero_total", "ratio_1e4"])
def test_masses_vs_float64(engine, oracle, monkeypatch, kind, box):
    _with_env(monkeypatch, {})
    n, nt = N_MASS, 8192
    assert _force_instance(nt, _tiles(n), 0.05, box) == ("OPEN_R8" if box == 0 else "FIXED_R4")
    pos, m = _cloud(n, box, 11), _mass_case(kind, N_MASS)
    if kind == "signed_zero_total":
        assert m.astype(np.float64).sum() == 0.0
    a = _forces(engine, _posm(pos, m), n - nt, nt, 0.05, box)
    idx = _sample(n - nt, nt, 512)
    err = rel_l2(a[idx - (n - nt)], _want_forces(oracle, pos, m, 0.05, box, idx))
    print(f"masses {kind} {'open' if box == 0 else 'fixed'}: {err:.2e}")
    assert err < TOL


@pytest.mark.parametrize("box", [0.0, 100.0], ids=["open_r8", "fixed_r4"])
def test_zero_masses_give_exact_zero(engine, monkeypatch, box):
    """All zero, and +0.0 mixed with -0.0 (equal under ==, so the equal-mass instance runs with m0 = +-0)."""
    _with_env(monkeypatch, {})
    n = N_MASS
    pos = _cloud(n, box, 12)
    signs = np.where(np.random.default_rng(2).random(n) < 0.5, np.float32(0.0), np.float32(-0.0)).astype(np.float32)
    assert np.signbit(signs).any() and not np.signbit(signs).all()
    for m in (np.zeros(n, np.float32), signs):
        assert np.all(_forces(engine, _posm(pos, m), 0, n, 0.05, box) == 0)


# ---- 6. coordinates --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("env", [{}, FLOAT_ENV], ids=["fixed_r4", "float_r4"])
def test_periodic_coordinate_edges(engine, oracle, monkeypatch, env):
    """Coincident pairs (r^2 = eps^2 on the fixed path), particles at 0, -0, box and the floats just below box, and
    particles several boxes out of frame.

    Rows 45-49 sit at (0, 0, 0), (-0, -0, -0), (box, box, box) -- one point of the torus -- and at the two floats
    below box on every axis, 7.6e-6 and 1.5e-5 from it: pairs far closer than eps.  The FP32 path gets their
    separations exactly; the fixed-point path quantises each x and y to box / 2^32 (up to 2 units per separation
    with the upper-half shift), so there a pair's force m d / eps^3 may be off by m 2 box 2^-32 / eps^3 per
    component: 1e-3 of these targets' forces, the documented price of that path (DESIGN 3.1), bounded here."""
    _with_env(monkeypatch, env)
    box, n, eps = 100.0, N_F, 0.05
    pos = _cloud(n, box, 13)
    pos[10:20] = pos[0:10]
    below = np.nextafter(np.float32(box), np.float32(0))
    edge = np.array([0.0, -0.0, box, below, np.nextafter(below, np.float32(0))], np.float32)
    pos[30:35, 0], pos[35:40, 1], pos[40:45, 2] = edge, edge, edge
    pos[45:50] = edge[:, None]
    k = np.random.default_rng(14).integers(-3, 4, (2000, 3)).astype(np.float32)
    pos[1000:3000] = pos[1000:3000] + k * np.float32(box)
    m = _mass(n, False, 15)
    a = _forces(engine, _posm(pos, m), 0, n, eps, box)
    idx = np.unique(np.concatenate([np.arange(0, 60), _sample(0, n, 400)]))
    assert all(t.size == 0 for t in direct_np.tie_partners(pos, box, idx))
    want = direct_np.forces(pos, m, eps, box, targets=idx)
    assert np.isfinite(a).all()
    close = np.isin(idx, np.arange(45, 50))
    err = rel_l2(a[idx], want) if env else rel_l2(a[idx[~close]], want[~close])
    near = np.abs(a[idx[close]] - want[close]).max()
    bound = 4 * float(m.max()) * 2 * (box / 2 ** 32) / float(np.float32(eps)) ** 3      # 4 close partners each
    print(f"coordinates {'float' if env else 'fixed'}: {err:.2e}, rows 45-49 off by {near:.2e} (bound {bound:.2e})")
    assert err < TOL and near <= bound


def test_open_offset_1e4(engine, oracle, monkeypatch):
    _with_env(monkeypatch, {})
    n = NS_HI
    pos = (_cloud(n, 0.0, 16) + np.float32(1e4)).astype(np.float32)
    m = _mass(n, False, 17)
    a = _forces(engine, _posm(pos, m), 0, 8192, 0.05, 0.0)
    idx = _sample(0, 8192, 512)
    assert rel_l2(a[idx], _open_rows(oracle, pos, m, 0.05, idx)) < TOL


# ---- 7. non-finite inputs --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("path", ["open", "float", "fixed"])
@pytest.mark.parametrize("axis", [0, 1, 2], ids=["x", "y", "z"])
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf], ids=["nan", "inf", "-inf"])
def test_non_finite_coordinate_poisons(engine, monkeypatch, path, axis, bad):
    """One non-finite coordinate makes every force NaN (periodic: all three components; open: at least the
    component of the bad axis, where an infinite separation meets a zero 1/r^3), the particle's own row included.
    The fixed-point conversion of x and y saturates on +-inf: the guard must catch infinities as well as NaN."""
    _with_env(monkeypatch, FLOAT_ENV if path == "float" else {})
    n, box = 32768, (0.0 if path == "open" else 100.0)
    assert _force_instance(n, _tiles(n), 0.05, box, force_float=path == "float") == \
        {"open": "OPEN_R8", "float": "FLOAT_R4", "fixed": "FIXED_R4"}[path]
    pos = _cloud(n, 100.0, 18)
    k = n // 2
    pos[k, axis] = bad
    a = _forces(engine, _posm(pos, np.ones(n, np.float32)), 0, n, 0.05, box)
    rows = np.isnan(a).any(1) if path == "open" else np.isnan(a).all(1)
    assert rows.sum() >= n - 1 and rows[k]


# ---- 8. potential and energy -----------------------------------------------------------------------------------------

POT_CASES = [
    ("open_small", N_P - 1, 0.0, True), ("open_small", N_P - 1, 0.0, False),
    ("open_first_not_small", N_P, 0.0, True), ("open_first_not_small", N_P, 0.0, False),
    ("per_small", N_P - 1, 100.0, False),
    ("per_first_not_small", N_P, 100.0, False),
    ("per_box64_pad", 30001, 64.0, True),
]


@pytest.mark.parametrize("case", POT_CASES, ids=[f"{c[0]}_{c[1]}_{'unit' if c[3] else 'general'}" for c in POT_CASES])
def test_potential_instance_vs_float64(engine, monkeypatch, case):
    name, n, box, unit = case
    _with_env(monkeypatch, {})
    pos, m = _cloud(n, box, n), _mass(n, unit, 19)
    posm = _posm(pos, m)
    phi = _potential(engine, posm, 0, n, 0.05, box)
    idx = _sample(0, n, 512)
    want = direct_np.potential(pos, m, 0.05, box, targets=idx)
    err = float(np.max(np.abs(phi[idx] - want) / want))
    print(f"potential {name} {_potential_instance(n, _tiles(n), box)} {'unit' if unit else 'general'}: {err:.2e}")
    assert err < POT_TOL
    # target shards whose bounds cross the 512 / 1536 blocks give the same rows
    for lo, hi in ((0, 1537), (1537, 9001), (9001, n)):
        assert rel_l2(_potential(engine, posm, lo, hi - lo, 0.05, box), phi[lo:hi]) < 1e-7


@pytest.mark.parametrize("box", [0.0, 100.0])
def test_energy_shards_add_up(engine, oracle, box):
    n = N_P + 1000
    pos, m = _cloud(n, box, 20), _mass(n, False, 21)
    vel = np.random.default_rng(22).normal(0.0, 10.0, (n, 3)).astype(np.float32)
    posm = _posm(pos, m)
    ke, pe = engine.energy_dev(posm, torch.from_numpy(vel).cuda(), eps=0.05, box=box)
    ks = ps = 0.0
    for lo, hi in ((0, 1537), (1537, 1538), (1538, 12289), (12289, n)):
        k_, p_ = engine.energy_dev(posm, torch.from_numpy(vel[lo:hi].copy()).cuda(), i0=lo, n_targets=hi - lo,
                                   eps=0.05, box=box)
        ks += k_
        ps += p_
    assert abs(ks - ke) <= 1e-12 * abs(ke) and abs(ps - pe) <= 1e-9 * abs(pe)
    _, pe0 = oracle.energy(pos, vel, m, 0.05, box)
    assert abs(pe - pe0) <= POT_TOL * abs(pe0)


# ---- 9. the multi-part source path, periodic -------------------------------------------------------------------------

PART_CUTS = [0, 0, 1, 1000, 1001, 7000, N_F + 777]        # empty first part, one-source parts, odd sizes


def _part_tiles():
    return sum(_tiles(b - a) for a, b in zip(PART_CUTS[:-1], PART_CUTS[1:]))


@pytest.mark.parametrize("unit", [True, False], ids=["unit", "general"])
@pytest.mark.parametrize("env", [{}, FLOAT_ENV], ids=["fixed_r4", "float_r4"])
def test_parts_periodic(engine, oracle, monkeypatch, env, unit):
    _with_env(monkeypatch, env)
    n, box = PART_CUTS[-1], 100.0
    pos, m = _cloud(n, box, 23), _mass(n, unit, 24)
    posm = _posm(pos, m)
    whole = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    engine.direct_forces_dev(posm, whole, 0, n, eps=0.05, box=box)
    parts, lens = [], []
    for a, b in zip(PART_CUTS[:-1], PART_CUTS[1:]):
        t = torch.empty(max(engine.tiles_bytes(b - a), 16) // 4, dtype=torch.float32, device="cuda")
        if b > a:
            engine.pack_tiles_dev(posm[a:b], b - a, t)
        parts.append(t)
        lens.append(b - a)
    idx = _sample(0, n, 512)
    want = direct_np.forces(pos, m, 0.05, box, targets=idx)
    for equal_flag in ([True, False] if unit else [False]):
        out = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        engine.direct_forces_parts_dev(parts, lens, posm, n, out, eps=0.05, box=box, all_masses_equal=equal_flag)
        torch.cuda.synchronize()
        o, w = out.cpu().numpy(), whole.cpu().numpy()
        e_whole, e_64 = rel_l2(o, w), rel_l2(o[idx], want)
        print(f"parts {env or 'fixed'} {'unit' if unit else 'general'} flag={equal_flag}: {e_whole:.2e} {e_64:.2e}")
        assert e_whole < 2e-6 and e_64 < TOL


# ---- coverage --------------------------------------------------------------------------------------------------------

def test_every_instance_is_reached():
    """Runs this file's case lists through the restated rule: every force instance in both mass versions and every
    potential instance must be reached (periodic potentials always run the general version)."""
    forces = set()
    for _, ns, i0, nt, eps, box in FORCE_CASES:
        for unit in (True, False):
            forces.add((_force_instance(nt, _tiles(ns), eps, box), unit))
    for box in (0.0, 100.0):                                # masses
        forces.add((_force_instance(8192, _tiles(N_MASS), 0.05, box), False))
    for unit in (True, False):                              # parts
        forces.add((_force_instance(N_F + 777, _part_tiles(), 0.05, 100.0), unit))
        forces.add((_force_instance(N_F + 777, _part_tiles(), 0.05, 100.0, force_float=True), unit))
    want = {(f, u) for f in ("OPEN_R2", "OPEN_R8", "FLOAT_R2", "FLOAT_R4", "FIXED_R4") for u in (True, False)}
    assert want <= forces, sorted(want - forces)
    pots = {(_potential_instance(n, _tiles(n), box), unit) for _, n, box, unit in POT_CASES}
    assert {("OPEN_R2", True), ("OPEN_R2", False), ("OPEN_R6", True), ("OPEN_R6", False), ("PER_R2", False),
            ("PER_R4", False)} <= pots
    # the thresholds themselves: both sides of each are in the list
    assert _force_instance(8191, _tiles(NS_HI), 0.01, 0.0) == "OPEN_R2"
    assert _force_instance(8192, _tiles(NS_LO), 0.01, 0.0) == "OPEN_R2"
    assert _force_instance(8192, _tiles(NS_HI), 0.01, 0.0) == "OPEN_R8"
    assert _force_instance(N_F - 1, _tiles(N_F - 1), 0.05, 100.0) == "FLOAT_R2"
    assert _force_instance(N_F, _tiles(N_F), 0.05, 100.0) == "FIXED_R4"
    if SM == 148:
        assert (NS_LO, NS_HI, N_F, N_P) == (75264, 75265, 24577, 21505)
