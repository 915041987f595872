"""pm_np.py -- float64 numpy restatement of the periodic particle-mesh force (b200_pm_forces_dev), an Ewald sum
for the periodic acceleration with a neutralising background, and the TreePM short-range remainder.

TEST INFRASTRUCTURE ONLY (imported by tests/ and tools/pm_time.py).  G = 1 throughout.  Box L, mesh G^3,
h = L / G, split radius r_s:
  wrap     x -> x - L floor(x / L); mesh point i at i h; cell floor(x / h) mod G, fraction x / h - floor(x / h)
  deposit  rho = sum m W_CIC / h^3 minus its mean (k = 0 mode zero: uniform neutralising background)
  phi_k    = -4 pi rho_k exp(-k^2 r_s^2) / (k^2 W(k)^2),  W(k) = prod_a sinc^2(k_a h / 2)
  a_k      = -i k_a phi_k, zero on the Nyquist plane of axis a; inverse FFT; CIC interpolation at the targets
  phi out  = -(interpolated mesh potential), the positive convention of b200_direct_potential_dev
The Ewald real-space part with alpha = 1 / (2 r_s) is the short-range remainder, its k-space part is the
Gaussian-filtered long-range force above without the mesh: PM + short range -> Ewald as the mesh resolves r_s.
"""
import numpy as np
from scipy.special import erfc


def wrap(x, box):
    x = np.asarray(x, np.float64)
    return x - box * np.floor(x / box)


def _cic(pos, grid, box):
    """Yields (corner cell indices (3 arrays), weights) of the 8 CIC corners of each position."""
    u = wrap(pos, box) * (grid / box)
    fl = np.floor(u)
    f = u - fl
    i = fl.astype(np.int64) % grid
    for dx in (0, 1):
        for dy in (0, 1):
            for dz in (0, 1):
                w = ((f[:, 0] if dx else 1 - f[:, 0]) * (f[:, 1] if dy else 1 - f[:, 1]) *
                     (f[:, 2] if dz else 1 - f[:, 2]))
                yield ((i[:, 0] + dx) % grid, (i[:, 1] + dy) % grid, (i[:, 2] + dz) % grid), w


def deposit(pos, mass, grid, box):
    """Mean-subtracted CIC density rho - rho_bar on the grid^3 mesh."""
    rho = np.zeros(grid ** 3, np.float64)
    m = np.asarray(mass, np.float64)
    for idx, w in _cic(pos, grid, box):
        rho += np.bincount(np.ravel_multi_index(idx, (grid,) * 3), weights=m * w, minlength=grid ** 3)
    rho = rho.reshape((grid,) * 3) / (box / grid) ** 3
    return rho - rho.mean()


def mesh_fields(rho, box, r_split):
    """(mesh potential, [a_x, a_y, a_z] meshes) of the mean-subtracted density."""
    G = rho.shape[0]
    h = box / G
    n = np.fft.fftfreq(G, 1.0 / G)
    nz = np.arange(G // 2 + 1, dtype=np.float64)
    kx = (2 * np.pi / box * n)[:, None, None]
    ky = (2 * np.pi / box * n)[None, :, None]
    kz = (2 * np.pi / box * nz)[None, None, :]
    k2 = kx * kx + ky * ky + kz * kz
    wk = (np.sinc(n / G)[:, None, None] * np.sinc(n / G)[None, :, None] * np.sinc(nz / G)[None, None, :]) ** 2
    k2[0, 0, 0] = 1.0
    green = -4 * np.pi * np.exp(-k2 * r_split * r_split) / (k2 * wk * wk)
    green[0, 0, 0] = 0.0
    phik = green * np.fft.rfftn(rho)
    acc = []
    for a, k in enumerate((kx, ky, kz)):
        ak = -1j * k * phik
        sl = [slice(None)] * 3
        sl[a] = G // 2
        ak[tuple(sl)] = 0.0                      # derivative along a is zero on a's Nyquist plane
        acc.append(np.fft.irfftn(ak, s=(G, G, G), axes=(0, 1, 2)))
    return np.fft.irfftn(phik, s=(G, G, G), axes=(0, 1, 2)), acc


def interpolate(mesh, pos, box):
    G = mesh.shape[0]
    out = np.zeros(len(pos), np.float64)
    for idx, w in _cic(pos, G, box):
        out += w * mesh[idx]
    return out


def pm_forces(src_pos, src_mass, tgt_pos, grid, box, r_split, potential=False):
    """Long-range PM acceleration (n_t, 3) at tgt_pos from the sources; with potential=True also the positive
    potential (n_t,) -- long range only, the target's own smoothed self term included."""
    phi, acc = mesh_fields(deposit(src_pos, src_mass, grid, box), box, r_split)
    a = np.stack([interpolate(m, tgt_pos, box) for m in acc], 1)
    if potential:
        return a, -interpolate(phi, tgt_pos, box)
    return a


def _min_image(d, box):
    return d - box * np.round(d / box)


def short_range(tgt_pos, src_pos, src_mass, box, r_split):
    """sum_j m_j d / r^3 [erfc(r / 2 r_s) + r / (r_s sqrt(pi)) exp(-r^2 / 4 r_s^2)], d = x_j - x_i minimum image,
    r = 0 pairs (self) skipped."""
    t = np.asarray(tgt_pos, np.float64)
    s = np.asarray(src_pos, np.float64)
    m = np.asarray(src_mass, np.float64)
    out = np.zeros((len(t), 3))
    for i0 in range(0, len(t), 256):
        d = _min_image(s[None, :, :] - t[i0:i0 + 256, None, :], box)
        r = np.sqrt((d * d).sum(-1))
        ok = r > 0
        rr = np.where(ok, r, 1.0)
        f = (erfc(rr / (2 * r_split)) + rr / (r_split * np.sqrt(np.pi)) * np.exp(-rr * rr / (4 * r_split * r_split)))
        f = np.where(ok, m[None, :] * f / rr ** 3, 0.0)
        out[i0:i0 + 256] = (f[:, :, None] * d).sum(1)
    return out


def ewald(tgt_pos, src_pos, src_mass, box, alpha=None, n_real=2, n_k=6):
    """Periodic acceleration with a uniform neutralising background (G = 1): real-space images |n_a| <= n_real,
    k-space vectors |m_a| <= n_k; zero-separation pairs (self) are skipped in the real-space sum."""
    alpha = 3.0 / box if alpha is None else alpha
    t = np.asarray(tgt_pos, np.float64)
    s = np.asarray(src_pos, np.float64)
    m = np.asarray(src_mass, np.float64)
    out = np.zeros((len(t), 3))
    rng = np.arange(-n_real, n_real + 1)
    for i0 in range(0, len(t), 256):
        d0 = _min_image(s[None, :, :] - t[i0:i0 + 256, None, :], box)      # x_j - x_i
        self_pair = (d0 * d0).sum(-1) == 0
        acc = np.zeros((d0.shape[0], 3))
        for nx in rng:
            for ny in rng:
                for nz in rng:
                    d = d0 + box * np.array([nx, ny, nz], np.float64)
                    r = np.sqrt((d * d).sum(-1))
                    skip = self_pair & (nx == 0) & (ny == 0) & (nz == 0)
                    rr = np.where(skip, 1.0, r)
                    f = erfc(alpha * rr) + 2 * alpha * rr / np.sqrt(np.pi) * np.exp(-alpha * alpha * rr * rr)
                    f = np.where(skip, 0.0, m[None, :] * f / rr ** 3)
                    acc += (f[:, :, None] * d).sum(1)
        out[i0:i0 + 256] = acc
    mk = np.arange(-n_k, n_k + 1)
    kv = 2 * np.pi / box * np.stack(np.meshgrid(mk, mk, mk, indexing="ij"), -1).reshape(-1, 3)
    kv = kv[(kv * kv).sum(1) > 0]
    k2 = (kv * kv).sum(1)
    coef = 4 * np.pi / box ** 3 * np.exp(-k2 / (4 * alpha * alpha)) / k2
    sk = (m[None, :] * np.exp(-1j * (kv @ s.T))).sum(1)                   # sum_j m_j e^{-i k x_j}
    # a_i = -(4 pi / L^3) sum_k k e^{-k^2/4a^2} / k^2 Im(e^{i k x_i} S_k)
    im = np.imag(np.exp(1j * (t @ kv.T)) * sk[None, :])
    out -= (im * coef[None, :]) @ kv
    return out
