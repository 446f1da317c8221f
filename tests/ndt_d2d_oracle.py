"""numpy binary64 restatement of gndt_register_d2d (include/gndt.h): distribution-to-distribution
NDT of the scan's own Gaussians against the map's, at the map level and at the levels.  It takes
two VOXEL_DTYPE tables, the map's and the scan's (a build of the scan in its own frame at the map's
origin), and reuses tests/ndt_oracle.py (transform, keys, pair search, LM) and
tests/ndt_levels_oracle.py (merged moments, coarse pair search, level settings) unchanged.

The derivatives follow the header's formulas term by term with explicit 3 x 3 matrices (B_a, B_ab,
A = B^-1 from numpy), so they check the kernel's compacted form rather than repeat it."""
import numpy as np

from tests import ndt_levels_oracle as NL
from tests import ndt_oracle as N

_II, _JJ = [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]
K = np.array([[[0, 0, 0], [0, 0, -1], [0, 1, 0]],
              [[0, 0, 1], [0, 0, 0], [-1, 0, 0]],
              [[0, -1, 0], [1, 0, 0], [0, 0, 0]]], np.float64)  # K[l] = [e_l]x


def floored(sig6, usable):
    """(Sigma' [m, 3, 3], usable): eigenvalues raised to >= 0.01 lambda_max, unusable when
    lambda_max is not positive and finite (Sigma' = 0 there)."""
    sig = np.zeros((len(sig6), 3, 3))
    for k in range(6):
        sig[:, _II[k], _JJ[k]] = sig6[:, k]
        sig[:, _JJ[k], _II[k]] = sig6[:, k]
    sig[~usable] = np.eye(3)
    w, V = np.linalg.eigh(sig)
    lmax = w[:, 2]
    usable = usable & (lmax > 0) & np.isfinite(lmax)
    out = np.einsum("vik,vk,vjk->vij", V, np.maximum(w, 0.01 * lmax[:, None]), V)
    out[~usable] = 0.0
    return out, usable


class Dists:
    """mu, Sigma', usable count and packed key of every cell of a table at factor k (k = 1: the
    records; k > 1: the level's Chan merges), keyed like ndt_oracle.Gaussians so that its pair
    searches apply.  count 0: not usable."""

    def __init__(self, vox, k=1, normalize_cov=0):
        if k == 1:
            n = vox["count"].astype(np.float64)
            usable = ((vox["flags"] & 1) != 0) & (vox["count"] >= 3)
            s = vox["scatter"].astype(np.float64)
            nm1 = np.where(usable, n - 1.0, 1.0)
            sig6 = (s * n[:, None]) / nm1[:, None] if normalize_cov else s / nm1[:, None]
            self.mu = vox["mean"].astype(np.float64)
            self.key = N._pack(N.contiguous(vox["sx"]), N.contiguous(vox["sy"]), N.contiguous(vox["sz"]))
        else:
            self.key, n, self.mu, S = NL.merged_moments(vox, k, normalize_cov)
            usable = n >= 3
            sig6 = S / np.where(usable, n - 1.0, 1.0)[:, None]
        self.sig, usable = floored(sig6, usable)
        self.count = np.where(usable, n, 0).astype(np.int64)


def derivatives(Gm, sig_s, x, c, R, pi, vi, d1, d2, with_abs=False):
    """S, g[6], H[6, 6] over the pairs (scan Gaussian pi, map Gaussian vi); x = R mu_s + t (binary64),
    sig_s the scan's Sigma' (and the sums of |contribution| per entry when with_abs)."""
    S, g, H = 0.0, np.zeros(6), np.zeros((6, 6))
    aS, ag, aH = 0.0, np.zeros(6), np.zeros((6, 6))
    for lo in range(0, len(pi), 1 << 16):
        p, v = pi[lo:lo + (1 << 16)], vi[lo:lo + (1 << 16)]
        P = len(p)
        Sig = R @ sig_s[p] @ R.T
        B = Sig + Gm.sig[v]
        A = np.linalg.inv(B)
        m = x[p] - Gm.mu[v]
        y = x[p] - c
        a = np.einsum("pij,pj->pi", A, m)
        q = np.einsum("pi,pi->p", m, a)
        e = np.exp(-0.5 * d2 * q)
        ma = np.zeros((P, 6, 3))   # m_a
        Ba = np.zeros((P, 6, 3, 3))  # B_a
        ma[:, [0, 1, 2], [0, 1, 2]] = 1.0
        for l in range(3):
            ma[:, 3 + l] = y @ K[l].T
            Ba[:, 3 + l] = K[l] @ Sig - Sig @ K[l]
        mab = np.zeros((P, 6, 6, 3))
        Bab = np.zeros((P, 6, 6, 3, 3))
        for k in range(3):
            for l in range(3):
                E = 0.5 * (K[k] @ K[l] + K[l] @ K[k])
                mab[:, 3 + k, 3 + l] = y @ E.T
                Bab[:, 3 + k, 3 + l] = E @ Sig + Sig @ E + K[k] @ Sig @ K[l].T + K[l] @ Sig @ K[k].T
        Baa = np.einsum("paij,pj->pai", Ba, a)                      # B_a a
        qa = 2.0 * np.einsum("pai,pi->pa", ma, a) - np.einsum("pi,pai->pa", a, Baa)
        AmA = np.einsum("pij,pbj->pbi", A, ma)                      # A m_b
        ABa = np.einsum("pij,pbj->pbi", A, Baa)                     # A B_b a
        qab = (2.0 * np.einsum("pabi,pi->pab", mab, a) + 2.0 * np.einsum("pai,pbi->pab", ma, AmA)
               - 2.0 * np.einsum("pai,pbi->pab", ma, ABa) - 2.0 * np.einsum("pbi,pai->pab", ma, ABa)
               + 2.0 * np.einsum("pai,pbi->pab", Baa, ABa) - np.einsum("pi,pabij,pj->pab", a, Bab, a))
        w = 0.5 * d1 * d2 * e
        s = -d1 * e
        gc = w[:, None] * qa
        hc = w[:, None, None] * (qab - 0.5 * d2 * qa[:, :, None] * qa[:, None, :])
        S += s.sum(); g += gc.sum(0); H += hc.sum(0)
        if with_abs:
            aS += np.abs(s).sum(); ag += np.abs(gc).sum(0); aH += np.abs(hc).sum(0)
    return (S, g, H, (aS, ag, aH)) if with_abs else (S, g, H)


class Problem(N.Problem):
    """One scan against one level (k = 1: the map level) of one map: map_vox and scan_vox in
    VOXEL_DTYPE, the map's origin / cell lengths / normalize_cov, and the scan's points (for the
    centre).  register() is ndt_oracle's LM (the level's settings of ndt_levels_oracle when k > 1)."""

    def __init__(self, map_vox, scan_vox, origin, grid_len, z_len, scan, k=1, normalize_cov=0, **ndt):
        self.k = int(k)
        self.G = Dists(map_vox, self.k, normalize_cov)
        self.S = Dists(scan_vox, self.k, normalize_cov)
        self.origin, self.grid_len, self.z_len = np.asarray(origin, np.float32), np.float32(grid_len), np.float32(z_len)
        self.p = N.finite_points(scan)
        self.pbar = self.p.astype(np.float64).mean(0) if len(self.p) else np.zeros(3)
        self.np = dict(N.DEFAULTS, **ndt)
        self.d1, self.d2 = NL.constants(self.k, grid_len, z_len, self.np["outlier_ratio"])
        if self.k > 1:
            self.np.update(NL.LEVEL_DEFAULTS)

    def scan_gaussians(self):
        """Indices of the usable scan Gaussians (count >= min_voxel_points)."""
        return np.nonzero(self.S.count >= self.np["min_voxel_points"])[0]

    def pairs(self, x):
        mp = self.np["min_voxel_points"]
        if self.k == 1:
            return N.pairs(self.G, x, self.origin, self.grid_len, self.z_len, mp)
        return NL.coarse_pairs(self.G, x, self.origin, self.grid_len, self.z_len, self.k, mp)

    def evaluate(self, T, with_abs=False, sig_s=None):
        """sig_s: the scan's Sigma' in place of its own (the Sigma'_i = 0 reduction)."""
        T = np.asarray(T, np.float64)
        idx = self.scan_gaussians()
        x = N.transform(T, self.S.mu[idx])
        pi, vi = self.pairs(x)
        c = self.center(T)
        sig = (self.S.sig if sig_s is None else sig_s)[idx]
        r = derivatives(self.G, sig, x, c, T[:3, :3], pi, vi, self.d1, self.d2, with_abs)
        out = dict(score=r[0], gradient=r[1], hessian=r[2], center=c, n_points=len(idx),
                   n_matched=len(np.unique(pi)), n_pairs=len(pi), pi=pi, vi=vi, x=x, idx=idx)
        if with_abs:
            out["abs"] = r[3]
        return out

    def frozen_score(self, T, pi, vi, xi):
        """S at the increment xi = (rho, phi) about c(T), pairs frozen: x' -> E (x' - c) + c + rho and
        R Sigma'_i R^T -> E R Sigma'_i R^T E^T (finite-difference checks)."""
        T = np.asarray(T, np.float64)
        idx = self.scan_gaussians()
        x = N.transform(T, self.S.mu[idx])
        c = self.center(T)
        E = N.so3_exp(xi[3:])
        xn = (x - c) @ E.T + c + xi[:3]
        return derivatives(self.G, self.S.sig[idx], xn, c, E @ T[:3, :3], pi, vi, self.d1, self.d2)[0]


class Pyramid(NL.Pyramid):
    """The map level and the levels of `factors` of one map and scan, D2D; register() is
    ndt_levels_oracle's: levels coarsest first, each from the previous pose, then the map level."""

    def __init__(self, map_vox, scan_vox, origin, grid_len, z_len, scan, factors, normalize_cov=0, **ndt):
        self.map = Problem(map_vox, scan_vox, origin, grid_len, z_len, scan, 1, normalize_cov, **ndt)
        self.levels = {k: Problem(map_vox, scan_vox, origin, grid_len, z_len, scan, k, normalize_cov, **ndt) for k in factors}


def scan_params(m_params, origin):
    """gndt_params of the scan build: the map's, with origin = the map's origin, every point binned,
    no strip filter, max_voxels = 0."""
    from grid_ndt_b200 import _abi
    p = _abi.Params.from_buffer_copy(bytes(m_params))
    p.origin_is_first_point = 0
    for i in range(3):
        p.origin[i] = np.float32(origin[i])
    p.tile_lo = p.tile_hi = 0
    p.max_voxels = 0
    return p


# ---- the D2D instances: EVERY held-out point inside a disc (a random subset leaves about one
# point per cell, so hardly any scan Gaussian exists) ---------------------------------------

def dense_disc(points, centre, radius):
    return points[np.hypot(points[:, 0] - centre[0], points[:, 1] - centre[1]) < radius]


def d2d_instance(cloud, radius=10.0):
    """(map cloud, scan in the scan frame): convergence_instance's 600 k-point map and every one of
    the other points within `radius` of the piers, moved by T_TRUE^-1."""
    perm = 1 + np.random.default_rng(5).permutation(len(cloud) - 1)
    mp = cloud[np.concatenate([[0], np.sort(perm[:599_999])])]
    rest = cloud[np.sort(perm[599_999:]), :3]
    return mp, N.apply(np.linalg.inv(N.T_TRUE), dense_disc(rest, N.PIER_CENTRE, radius))
