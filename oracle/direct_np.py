"""direct_np.py -- float64 numpy restatement of the softened direct sum, open or periodic.

TEST INFRASTRUCTURE ONLY (imported by tests/).  For a set of targets (indices into the particle list) against every
particle as a source:
  acceleration  a_i   = sum_j m_j d_ij / (|d_ij|^2 + eps^2)^(3/2)          (G = 1; the j == i term is 0)
  potential     phi_i = sum_{j != i} m_j / sqrt(|d_ij|^2 + eps^2)         (positive, as direct_potential)
with d_ij = x_j - x_i taken in float64 from the float32 inputs.  With box > 0 each component is the minimum image,
as the reference's minimum_image (src/physics/lambda_cdm_kernels.cu:122-141) compares it: |d| <= box / 2 after the
wrap.  That compare keeps a separation of exactly +-box/2 as it is ("raw" ties); ties="flip" sends it to the other
image instead.  Unlike the single compare of the reference, the wrap here holds for positions any number of boxes
out of frame; a tie is then an exact odd multiple of box / 2, and "raw" keeps the sign of the raw separation.
"""
import numpy as np


def minimum_image(d, box, ties="raw"):
    """d (float64) reduced to [-box/2, box/2]; a separation exactly half a box from its image keeps the sign of d
    (ties="raw") or takes the opposite one (ties="flip")."""
    if ties not in ("raw", "flip"):
        raise ValueError(ties)
    d = np.asarray(d, np.float64)
    h = 0.5 * box
    r = d - box * np.rint(d / box)             # exact: box * k and the difference are representable
    tie = np.abs(r) == h
    s = np.sign(d) if ties == "raw" else -np.sign(d)
    return np.where(tie, s * h, r)


def _chunks(n_targets, n_sources, budget=1 << 22):
    c = max(1, budget // max(n_sources, 1))
    return range(0, n_targets, c), c


def _separations(pos, idx, box, ties):
    d = pos[None, :, :] - pos[idx][:, None, :]              # [target, source, 3]
    return minimum_image(d, box, ties) if box > 0 else d


def forces(pos, mass=None, eps=0.01, box=0.0, targets=None, ties="raw"):
    """Acceleration (n_targets, 3) float64 of `targets` (indices, default all) against every particle."""
    pos = np.asarray(pos, np.float32).astype(np.float64)
    n = pos.shape[0]
    m = np.ones(n) if mass is None else np.asarray(mass, np.float32).astype(np.float64)
    idx = np.arange(n) if targets is None else np.asarray(targets, np.int64)
    eps2 = float(np.float32(eps)) ** 2
    out = np.empty((idx.size, 3))
    starts, c = _chunks(idx.size, n)
    for s in starts:
        d = _separations(pos, idx[s:s + c], box, ties)
        r2 = (d * d).sum(-1) + eps2
        w = m[None, :] / (r2 * np.sqrt(r2))
        out[s:s + c] = np.einsum("ts,tsk->tk", w, d)
    return out


def potential(pos, mass=None, eps=0.01, box=0.0, targets=None):
    """Potential (n_targets,) float64, the j == i term left out (a coincident j != i still counts m_j / eps)."""
    pos = np.asarray(pos, np.float32).astype(np.float64)
    n = pos.shape[0]
    m = np.ones(n) if mass is None else np.asarray(mass, np.float32).astype(np.float64)
    idx = np.arange(n) if targets is None else np.asarray(targets, np.int64)
    eps2 = float(np.float32(eps)) ** 2
    out = np.empty(idx.size)
    starts, c = _chunks(idx.size, n)
    for s in starts:
        t = idx[s:s + c]
        d = _separations(pos, t, box, "raw")                # |d| is the same for either image of a tie
        w = m[None, :] / np.sqrt((d * d).sum(-1) + eps2)
        w[np.arange(t.size), t] = 0.0
        out[s:s + c] = w.sum(1)
    return out


def tie_partners(pos, box, targets=None):
    """Per target, the sources j whose separation on some axis is exactly half a box from its other image."""
    pos = np.asarray(pos, np.float32).astype(np.float64)
    idx = np.arange(pos.shape[0]) if targets is None else np.asarray(targets, np.int64)
    res = []
    starts, c = _chunks(idx.size, pos.shape[0])
    for s in starts:
        d = pos[None, :, :] - pos[idx[s:s + c]][:, None, :]
        r = d - box * np.rint(d / box)
        tie = (np.abs(r) == 0.5 * box).any(-1)
        res.extend(np.nonzero(row)[0] for row in tie)
    return res
