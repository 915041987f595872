"""treepm_np.py -- float64 numpy restatement of the TreePM short-range force (b200_tree_walk_short_dev at theta = 0).

TEST INFRASTRUCTURE ONLY (imported by tests/).  G = 1.  With pm_np.pm_forces(..., r_split = r_s) as the long range,
pm_forces + short_range is TreePM:
  d = minimum image of x_j - x_i, r = |d|, g(r) = erfc(r / 2 r_s) + r / (r_s sqrt(pi)) exp(-r^2 / 4 r_s^2)
  a_i = sum_j m_j g(r) d / (r^2 + eps^2)^(3/2) over the pairs with 0 < r (< r_cut when a cut-off is given)
With eps = 0 and no cut-off this is pm_np.short_range.
"""
import numpy as np
from scipy.special import erfc

from oracle.pm_np import _min_image, wrap


def _terms(d, m, r_split, eps, r_cut):
    """m g(r) / (r^2 + eps^2)^(3/2) of separations d (..., 3); 0 for r = 0 and for r >= r_cut."""
    r = np.sqrt((d * d).sum(-1))
    ok = r > 0
    if r_cut is not None:
        ok &= r < r_cut
    rr = np.where(ok, r, 1.0)
    g = erfc(rr / (2 * r_split)) + rr / (r_split * np.sqrt(np.pi)) * np.exp(-rr * rr / (4 * r_split * r_split))
    return np.where(ok, m * g / (rr ** 3 if eps == 0 else (rr * rr + eps * eps) ** 1.5), 0.0)


def short_range(tgt_pos, src_pos, src_mass, box, r_split, eps=0.0, r_cut=None, neighbours=False):
    """Short-range acceleration (n_t, 3) at tgt_pos.  neighbours=True (needs 0 < r_cut < box / 2) sums only over the
    sources a periodic k-d tree finds within r_cut of each target, which keeps 2^24 sources cheap; otherwise every
    target meets every source."""
    t = np.asarray(tgt_pos, np.float64)
    s = np.asarray(src_pos, np.float64)
    m = np.asarray(src_mass, np.float64)
    out = np.zeros((len(t), 3))
    if not neighbours:
        for i0 in range(0, len(t), 256):
            d = _min_image(s[None, :, :] - t[i0:i0 + 256, None, :], box)
            f = _terms(d, m[None, :], r_split, eps, r_cut)
            out[i0:i0 + 256] = (f[:, :, None] * d).sum(1)
        return out
    from scipy.spatial import cKDTree
    if r_cut is None or not 0 < r_cut < box / 2:
        raise ValueError("the neighbour-list sum needs 0 < r_cut < box / 2")
    # a slightly larger radius: membership is decided by the same r < r_cut test as the brute-force sum
    lists = cKDTree(wrap(s, box), boxsize=box).query_ball_point(wrap(t, box), r_cut * (1 + 1e-9))
    for i0 in range(0, len(t), 256):
        js = lists[i0:i0 + 256]
        j = np.concatenate([np.asarray(x, np.int64) for x in js])
        i = np.repeat(np.arange(len(js)), [len(x) for x in js])
        d = _min_image(s[j] - t[i0 + i], box)
        f = _terms(d, m[j], r_split, eps, r_cut)
        for a in range(3):
            out[i0:i0 + len(js), a] = np.bincount(i, weights=f * d[:, a], minlength=len(js))
    return out
