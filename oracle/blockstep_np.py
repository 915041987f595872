"""blockstep_np.py -- numpy restatement of the block (hierarchical) time steps of the comoving KDK (DESIGN 3.14):
the factor table, the binning rule and the sync-point pass of b200_block_kick_dev in float32 with its exact operation
order, and the whole scheme in float64 with a pluggable force (e.g. pm_np.pm_forces + treepm_np.short_range).

TEST INFRASTRUCTURE ONLY (imported by tests/).  Units and conventions as oracle/comoving_np.py.  A PM step from a0 to
a1 has S = 2^L sub-steps (L = max_bins - 1) uniform in ln a; bin b steps w_b = 2^(L - b) of them.
"""
import numpy as np

from oracle import comoving_np

f32 = np.float32


def factor_table(a0, a1, max_bins, cosmo=comoving_np.LCDM, kdk=comoving_np.kdk_factors):
    """(kicks, nodes) in float64, the layout of b200grav.block_factor_table: nodes[k] = a0 exp(k Delta / S) (ends
    exact), kicks[(2^b - 1) + j] = K(a_s, m), kicks[(2^max_bins - 1) + (2^b - 1) + j] = K(m, a_e).  kdk(a0, a1, cosmo)
    -> (drift, kick)."""
    L = max_bins - 1
    S = 1 << L
    d = np.log(a1 / a0)
    nodes = np.array([a0] + [a0 * np.exp(k * d / S) for k in range(1, S)] + [a1], np.float64)
    nb = (1 << max_bins) - 1
    kicks = np.empty(2 * nb)
    for b in range(max_bins):
        w = S >> b
        for j in range(1 << b):
            s, e = nodes[j * w], nodes[(j + 1) * w]
            m = np.sqrt(s * e)
            kicks[(1 << b) - 1 + j] = kdk(s, m, cosmo)[1]
            kicks[nb + (1 << b) - 1 + j] = kdk(m, e, cosmo)[1]
    return kicks, nodes


def ko_index(b, j):
    return (1 << b) - 1 + j


def kc_index(b, j, max_bins):
    return (1 << max_bins) - 1 + (1 << b) - 1 + j


def crit_of(a, eta, eps, cosmo=comoving_np.LCDM):
    """2 eta eps a^3 E(a)^2 (double): the criterion is dln a <= sqrt(crit / |g|)."""
    om, ok, ol = cosmo
    return 2.0 * eta * eps * a ** 3 * (om / a ** 3 + ok / a ** 2 + ol)


def next_sync_point(k, counts, max_bins):
    L = max_bins - 1
    return min((((k >> (L - b)) + 1) << (L - b)) for b in range(max_bins) if counts[b] > 0)


def lowest_bin(k, L):
    """L - ctz(k): the longest step that starts on its own grid at sync point 0 < k < 2^L."""
    return L - ((k & -k).bit_length() - 1)


# ---- float32: the device pass, bit for bit ---------------------------------------------------------------------------

def gnorm32(g):
    g = np.asarray(g, f32)
    with np.errstate(over="ignore", invalid="ignore"):
        return np.sqrt((g[:, 0] * g[:, 0] + g[:, 1] * g[:, 1]) + g[:, 2] * g[:, 2])


def desired_bin32(g, dlna, crit, L):
    """The smallest b < L with float(dlna^2 / 4^b) |g| <= crit (float32, one rounding per operation), else L."""
    gn = gnorm32(g)
    out = np.full(len(gn), L, np.int64)
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(L - 1, -1, -1):
            out[f32(dlna * dlna / 4.0 ** b) * gn <= f32(crit)] = b
    return out


def sync_pass32(k, max_bins, mass, mom, acc, acc_long, acc_short, bins, fac, crit, dlna, pos=None, drift=0.0,
                box=0.0):
    """b200_block_kick_dev at sync point k in float32: returns (mom, acc, bins, hist, pos) after the pass; pos
    (float32 (n, 3)) drifts by drift (0: none), wrapped into [0, box) when box > 0."""
    L = max_bins - 1
    S = 1 << L
    mass = np.asarray(mass, f32)
    minv = f32(1.0) / mass
    mom, acc = np.array(mom, f32), np.array(acc, f32)
    gl, gs = np.asarray(acc_long, f32), np.asarray(acc_short, f32)
    fac = np.asarray(fac, f32)
    b = np.minimum(np.asarray(bins, np.int64), L)
    opening = np.zeros(len(b), bool)
    if k == 0:
        b = desired_bin32(acc, dlna, crit, L)
        opening[:] = True
    else:
        w = 1 << (L - b)
        closing = k % w == 0
        kc = fac[kc_index(b, k // w - 1, max_bins)]
        if k == S:                                                   # every step ends
            acc = gl + gs
            z = b == 0
            mom[z] = _kick_rows(mom[z], acc[z], mass[z], minv[z], kc[z])
            nz = ~z
            mom[nz] = _kick_rows(mom[nz], gl[nz], mass[nz], minv[nz], np.full(nz.sum(), fac[kc_index(0, 0, max_bins)]))
            mom[nz] = _kick_rows(mom[nz], gs[nz], mass[nz], minv[nz], kc[nz])
        else:
            c = closing
            mom[c] = _kick_rows(mom[c], gs[c], mass[c], minv[c], kc[c])
            want = desired_bin32(gl[c] + gs[c], dlna, crit, L)
            b = b.copy()
            b[c] = np.maximum(want, lowest_bin(k, L))
            opening = c
    if k < S:
        o = opening
        w = 1 << (L - b[o])
        ko = fac[ko_index(b[o], k // w)]
        mo, mass_o, minv_o = mom[o], mass[o], minv[o]
        if k == 0:
            z = b[o] == 0
            mo[z] = _kick_rows(mo[z], acc[o][z], mass_o[z], minv_o[z], ko[z])
            nz = ~z
            mo[nz] = _kick_rows(mo[nz], gl[o][nz], mass_o[nz], minv_o[nz], np.full(nz.sum(), fac[0], f32))
            mo[nz] = _kick_rows(mo[nz], gs[o][nz], mass_o[nz], minv_o[nz], ko[nz])
        else:
            mo = _kick_rows(mo, gs[o], mass_o, minv_o, ko)
        mom[o] = mo
    hist = np.bincount(b, minlength=16)[:16]
    if pos is not None and f32(drift) != 0:
        pos = np.asarray(pos, f32) + mom * f32(drift)
        if box > 0:
            with np.errstate(invalid="ignore"):                 # rows with a NaN momentum stay NaN
                pos = np.fmod(pos + f32(box), f32(box))
    return mom, acc, b.astype(np.uint8), hist, pos


def _kick_rows(v, a, m, minv, dt):
    """kick1 with a per-row factor dt (float32): v + (((a m) minv) dt) 1."""
    f = a * m[:, None]
    f = f * minv[:, None]
    f = f * np.asarray(dt, f32)[:, None]
    f = f * f32(1.0)
    return v + f


# ---- float64: the whole scheme ---------------------------------------------------------------------------------------

def desired_bin64(g, dlna, crit, L):
    """The binning rule in float64; also returns log4(dlna^2 |g| / crit), whose distance from the integers is the
    margin by which a bin could flip under rounding."""
    gn = np.sqrt((np.asarray(g, np.float64) ** 2).sum(1))
    with np.errstate(divide="ignore"):
        x = np.log(dlna * dlna * gn / crit) / np.log(4.0)
    return np.clip(np.ceil(x), 0, L).astype(np.int64), x


def scheme(pos, mom, mass, box, a_grid, max_bins, forces, eta=0.025, eps=0.01, cosmo=comoving_np.LCDM,
           kdk=comoving_np.kdk_factors, fixed_bins=None, record=None):
    """The block-step KDK in float64 through the PM steps a_grid[0] -> a_grid[1] -> ...  forces(pos, idx, with_long)
    -> (acc_long (n, 3) or None, acc_short rows of the particles idx).  fixed_bins: keep these bins (no rebinning).
    record(k, a_k, bins, margin_x): called after every rebinning.  Returns (pos, mom, bins)."""
    pos = np.array(pos, np.float64)
    mom = np.array(mom, np.float64)
    n = len(pos)
    L = max_bins - 1
    S = 1 << L
    allidx = np.arange(n)
    gl, gs = forces(pos, allidx, True)
    bins = np.zeros(n, np.int64)
    for a0, a1 in zip(a_grid[:-1], a_grid[1:]):
        kicks, nodes = factor_table(a0, a1, max_bins, cosmo, kdk)
        dlna = np.log(a1 / a0)
        ko = lambda b, j: kicks[ko_index(b, j)]
        kc = lambda b, j: kicks[kc_index(b, j, max_bins)]
        # k = 0
        acc = gl + gs
        if fixed_bins is None:
            bins, x = desired_bin64(acc, dlna, crit_of(a0, eta, eps, cosmo), L)
            if record:
                record(0, a0, bins, x)
        else:
            bins = np.asarray(fixed_bins, np.int64).copy()
        z = bins == 0
        mom[z] += acc[z] * ko(0, 0)
        mom[~z] += gl[~z] * ko(0, 0) + gs[~z] * np.array([ko(b, 0) for b in bins[~z]])[:, None]
        k = 0
        while k < S:
            k1 = next_sync_point(k, np.bincount(bins, minlength=max_bins), max_bins)
            pos = pos + mom * kdk(nodes[k], nodes[k1], cosmo)[0]
            pos -= box * np.floor(pos / box)
            k = k1
            w = 1 << (L - bins)
            act = np.flatnonzero(k % w == 0)
            gl_new, gs_act = forces(pos, act, k == S)
            gs = gs.copy()
            gs[act] = gs_act
            kcs = np.array([kc(b, k // (1 << (L - b)) - 1) for b in bins[act]])
            if k == S:
                gl = gl_new
                acc = gl + gs
                z = bins == 0
                mom[z] += acc[z] * kc(0, 0)
                nz = ~z
                mom[nz] += gl[nz] * kc(0, 0) + gs[nz] * kcs[nz][:, None]
                break
            mom[act] += gs[act] * kcs[:, None]
            if fixed_bins is None:
                want, x = desired_bin64(gl[act] + gs[act], dlna, crit_of(nodes[k], eta, eps, cosmo), L)
                bins = bins.copy()
                bins[act] = np.maximum(want, lowest_bin(k, L))
                if record:
                    record(k, nodes[k], bins[act], x)
            kos = np.array([ko(b, k // (1 << (L - b))) for b in bins[act]])
            mom[act] += gs[act] * kos[:, None]
    return pos, mom, bins


def treepm_forces(mass, box, grid, r_split, eps, r_cut):
    """forces() of scheme(): the float64 PM long range (pm_np.pm_forces) and the softened, cut-off short range
    (treepm_np.short_range) of all particles."""
    from oracle import pm_np, treepm_np

    def f(pos, idx, with_long):
        gl = pm_np.pm_forces(pos, mass, pos, grid, box, r_split) if with_long else None
        gs = treepm_np.short_range(pos[idx], pos, mass, box, r_split, eps=eps, r_cut=r_cut) if len(idx) else \
            np.zeros((0, 3))
        return gl, gs
    return f
