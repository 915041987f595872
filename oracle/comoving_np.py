"""comoving_np.py -- float64 numpy/scipy restatement of the comoving LambdaCDM integration (DESIGN 3.13): the KDK
factors, the exact linear growing mode, the 1-D Zel'dovich plane wave, a numpy comoving KDK driven by the exact
planar force, the Ewald potential and the TreePM short-range potential at theta = 0.

TEST INFRASTRUCTURE ONLY (imported by tests/).  Units: H0 = 1, G = 1, comoving lengths in the box's unit;
cosmo = (Om, Ok, OL), E(a)^2 = Om a^-3 + Ok a^-2 + OL.  Canonical momentum p = a^2 dx/dt; the mean comoving
density is 3 Om / (8 pi), so the peculiar acceleration of a plane-wave displacement s is g = 4 pi rho s = 1.5 Om s.
"""
import numpy as np
from scipy.integrate import quad
from scipy.special import erfc

from oracle.pm_np import _min_image

LCDM = (0.31, 0.0, 0.69)


def E(a, cosmo=LCDM):
    om, ok, ol = cosmo
    a = np.asarray(a, np.float64)
    return np.sqrt(om / a ** 3 + ok / a ** 2 + ol)


def kdk_factors(a0, a1, cosmo=LCDM):
    """(drift, kick) = (int da / (a^3 E), int da / (a^2 E)) from a0 to a1."""
    q = dict(epsabs=0.0, epsrel=1e-13, limit=200)
    return (quad(lambda a: 1.0 / (a ** 3 * E(a, cosmo)), a0, a1, **q)[0],
            quad(lambda a: 1.0 / (a ** 2 * E(a, cosmo)), a0, a1, **q)[0])


def _growth_integral(a, cosmo):
    return quad(lambda x: 1.0 / (x * E(x, cosmo)) ** 3, 0.0, a, epsabs=0.0, epsrel=1e-13, limit=200)[0]


def growth(a, cosmo=LCDM):
    """Linear growing mode D(a) = 5/2 Om E(a) int_0^a da' / (a' E)^3 (Heath 1977; exact for matter, curvature and
    Lambda), normalised to D -> a as a -> 0."""
    return 2.5 * cosmo[0] * float(E(a, cosmo)) * _growth_integral(a, cosmo)


def growth_rate(a, cosmo=LCDM):
    """f = dln D / dln a = dln E / dln a + 1 / (a^2 E^3 I), I = int_0^a da' / (a' E)^3."""
    om, ok, _ = cosmo
    e2 = float(E(a, cosmo)) ** 2
    return (-1.5 * om / a ** 3 - ok / a ** 2) / e2 + 1.0 / (a ** 2 * e2 ** 1.5 * _growth_integral(a, cosmo))


def plane_wave(q, a, amplitude, box, cosmo=LCDM):
    """Exact 1-D Zel'dovich solution before shell crossing for s(q) = amplitude sin(2 pi q / box):
    x = q + D(a) s(q), p = a^3 E D'(a) s(q), D' = f D / a.  Returns (x, p), x not wrapped."""
    s = amplitude * np.sin(2 * np.pi * np.asarray(q, np.float64) / box)
    d = growth(a, cosmo)
    return q + d * s, a ** 3 * float(E(a, cosmo)) * growth_rate(a, cosmo) * d / a * s


def kdk_plane(disp, p, a_grid, cosmo=LCDM):
    """The comoving KDK of ComovingSimulation on displacements disp = x - q under the exact planar force
    g = 1.5 Om disp (valid before shell crossing), through the scale factors a_grid[0] -> a_grid[-1]."""
    disp = np.array(disp, np.float64)
    p = np.array(p, np.float64)
    acc = 1.5 * cosmo[0] * disp
    for a0, a1 in zip(a_grid[:-1], a_grid[1:]):
        am = np.sqrt(a0 * a1)
        p += acc * kdk_factors(a0, am, cosmo)[1]
        disp += p * kdk_factors(a0, a1, cosmo)[0]
        acc = 1.5 * cosmo[0] * disp
        p += acc * kdk_factors(am, a1, cosmo)[1]
    return disp, p


def ewald_potential(tgt_pos, src_pos, src_mass, box, alpha=None, n_real=2, n_k=6):
    """Periodic potential (positive convention, G = 1) at the targets with a uniform neutralising background:
    phi_i = sum_j m_j psi(x_i - x_j), psi the zero-mean periodic Green's function; a target that is also a source
    (zero separation) drops its own 1/r term and keeps its images.  Targets must be sources or not: the self test
    is a zero minimum-image separation."""
    alpha = 3.0 / box if alpha is None else alpha
    t = np.asarray(tgt_pos, np.float64)
    s = np.asarray(src_pos, np.float64)
    m = np.asarray(src_mass, np.float64)
    out = np.zeros(len(t))
    rng = np.arange(-n_real, n_real + 1)
    for i0 in range(0, len(t), 128):
        d0 = _min_image(s[None, :, :] - t[i0:i0 + 128, None, :], box)
        self_pair = (d0 * d0).sum(-1) == 0
        phi = np.zeros(d0.shape[0])
        for nx in rng:
            for ny in rng:
                for nz in rng:
                    d = d0 + box * np.array([nx, ny, nz], np.float64)
                    r = np.sqrt((d * d).sum(-1))
                    skip = self_pair & (nx == 0) & (ny == 0) & (nz == 0)
                    rr = np.where(skip, 1.0, r)
                    phi += np.where(skip, 0.0, m[None, :] * erfc(alpha * rr) / rr).sum(1)
        # the n = 0 image of the particle itself: its erf(alpha r) / r -> 2 alpha / sqrt(pi) belongs to the k-sum
        phi -= (self_pair * m[None, :]).sum(1) * 2 * alpha / np.sqrt(np.pi)
        out[i0:i0 + 128] = phi
    mk = np.arange(-n_k, n_k + 1)
    kv = 2 * np.pi / box * np.stack(np.meshgrid(mk, mk, mk, indexing="ij"), -1).reshape(-1, 3)
    kv = kv[(kv * kv).sum(1) > 0]
    k2 = (kv * kv).sum(1)
    coef = 4 * np.pi / box ** 3 * np.exp(-k2 / (4 * alpha * alpha)) / k2
    sk = (m[None, :] * np.exp(-1j * (kv @ s.T))).sum(1)                   # sum_j m_j e^{-i k x_j}
    out += (np.real(np.exp(1j * (t @ kv.T)) * sk[None, :]) * coef[None, :]).sum(1)
    return out - np.pi / (alpha * alpha * box ** 3) * m.sum()


def short_potential(tgt_idx, src_pos, src_mass, box, r_split, eps, r_cut):
    """b200_tree_potential_short_dev at theta = 0 for the targets src_pos[tgt_idx]:
    sum_{0 < r < r_cut} m_j erfc(r / 2 r_s) / sqrt(r^2 + eps^2) - m_i / (sqrt(pi) r_s) - 4 pi r_s^2 M / box^3."""
    s = np.asarray(src_pos, np.float64)
    m = np.asarray(src_mass, np.float64)
    idx = np.asarray(tgt_idx)
    out = np.zeros(len(idx))
    for i0 in range(0, len(idx), 256):
        d = _min_image(s[None, :, :] - s[idx[i0:i0 + 256], None, :], box)
        r = np.sqrt((d * d).sum(-1))
        ok = (r > 0) & (r < r_cut)
        rr = np.where(ok, r, 1.0)
        out[i0:i0 + 256] = np.where(ok, m[None, :] * erfc(rr / (2 * r_split)) / np.sqrt(rr * rr + eps * eps), 0.0).sum(1)
    return out - m[idx] / (np.sqrt(np.pi) * r_split) - 4 * np.pi * r_split ** 2 * m.sum() / box ** 3
