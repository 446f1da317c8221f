"""numpy binary64 restatement of the coarse levels of gndt_register_levels (include/gndt.h): the
coarse cell of a map cell and of a scan point (floor division of contiguous indices), the Gaussian
of a coarse cell (sequential Chan merge of its fitted records in table order), the candidates and
score constants of a level, and the per-level Levenberg-Marquardt loop.  The transform, the
derivatives and the LM itself are tests/ndt_oracle.py's.  Works from any VOXEL_DTYPE table."""
import numpy as np

from tests import ndt_oracle as N

LEVEL_DEFAULTS = dict(max_iterations=50, translation_epsilon=1e-3, rotation_epsilon=1e-3)
_II, _JJ = [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]


def floor_div(c, k):
    return np.floor_divide(np.asarray(c, np.int64), int(k))


def coarse_keys(vox, k):
    """(X, Y, Z) of every record of a voxel table at factor k."""
    return tuple(floor_div(N.contiguous(vox[f]), k) for f in ("sx", "sy", "sz"))


def merged_moments(vox, k, normalize_cov=0):
    """(packed key, n, mean [m, 3], un-normalised scatter [m, 6]) of every coarse cell that holds a
    record: the Chan merge, record by record in ascending table index, of its GNDT_F_FITTED records
    (cells without one have n = 0)."""
    key = N._pack(*coarse_keys(vox, k))
    order = np.argsort(key, kind="stable")  # stable: table order inside a cell
    ks = key[order]
    u, start = np.unique(ks, return_index=True)
    cell = np.repeat(np.arange(len(u)), np.diff(np.append(start, len(ks))))
    rank = np.arange(len(ks)) - start[cell]
    v = vox[order]
    fitted = (v["flags"] & 1) != 0
    nb_all = v["count"].astype(np.float64)
    mb_all = v["mean"].astype(np.float64)
    sb_all = v["scatter"].astype(np.float64)
    if normalize_cov:
        sb_all = sb_all * nb_all[:, None]
    n, mu, S = np.zeros(len(u)), np.zeros((len(u), 3)), np.zeros((len(u), 6))
    by_rank = np.argsort(rank, kind="stable")
    bounds = np.searchsorted(rank[by_rank], np.arange(rank.max() + 2 if len(rank) else 1))
    for r in range(len(bounds) - 1):
        sel = by_rank[bounds[r]:bounds[r + 1]]
        sel = sel[fitted[sel]]
        c = cell[sel]
        nb, nc = nb_all[sel], n[c]
        nn = nc + nb
        f, w = nb / nn, nc * nb / nn
        d = mb_all[sel] - mu[c]
        S[c] += sb_all[sel] + d[:, _II] * d[:, _JJ] * w[:, None]
        mu[c] += d * f[:, None]
        n[c] = nn
    return u, n, mu, S


class CoarseGaussians:
    """mu, C and the usable count of every coarse cell of a level (count 0: not usable), keyed
    like ndt_oracle.Gaussians so that its pair search and derivatives apply."""

    def __init__(self, vox, k, normalize_cov=0):
        self.key, n, self.mu, S = merged_moments(vox, k, normalize_cov)
        usable = n >= 3
        sig6 = S / np.where(usable, n - 1.0, 1.0)[:, None]
        sig = np.zeros((len(n), 3, 3))
        for j in range(6):
            sig[:, _II[j], _JJ[j]] = sig6[:, j]
            sig[:, _JJ[j], _II[j]] = sig6[:, j]
        sig[~usable] = np.eye(3)
        w, V = np.linalg.eigh(sig)
        lmax = w[:, 2]
        usable &= (lmax > 0) & np.isfinite(lmax)
        wr = np.maximum(w, 0.01 * lmax[:, None])
        with np.errstate(divide="ignore", invalid="ignore"):
            self.C = np.einsum("vik,vk,vjk->vij", V, 1.0 / wr, V)
        self.C[~usable] = 0.0
        self.count = np.where(usable, n, 0).astype(np.int64)


def constants(k, grid_len, z_len, outlier_ratio):
    """d1, d2 of a level: V = (k grid_len)^2 (k z_len) in binary64."""
    p_o = float(np.float32(outlier_ratio))
    kg, kz = k * float(np.float32(grid_len)), k * float(np.float32(z_len))
    V = kg * kg * kz
    c1, c2 = 10.0 * (1.0 - p_o), p_o / V
    d3 = -np.log(c2)
    d1 = -np.log(c1 + c2) - d3
    d2 = -2.0 * np.log((-np.log(c1 * np.exp(-0.5) + c2) - d3) / d1)
    return d1, d2


def coarse_pairs(G, x, origin, grid_len, z_len, k, min_points):
    """(point index, coarse cell index) of every candidate pair: the point's map cell (binning of
    x rounded to binary32), floor-divided by k, then the 15 candidates on coarse indices."""
    cx, cy, cz, ok = N.keys(x.astype(np.float32), origin, grid_len, z_len)
    X, Y, Z = floor_div(cx, k), floor_div(cy, k), floor_div(cz, k)
    pi, vi = [], []
    idx = np.nonzero(ok)[0]
    for dx, dy, dz in N.OFFSETS:
        key = N._pack(X[idx] + dx, Y[idx] + dy, Z[idx] + dz)
        j = np.minimum(np.searchsorted(G.key, key), len(G.key) - 1)
        hit = (G.key[j] == key) & (G.count[j] >= min_points)
        pi.append(idx[hit]); vi.append(j[hit])
    return np.concatenate(pi), np.concatenate(vi)


class Level(N.Problem):
    """One scan against the level of factor k of one map; register() is ndt_oracle's LM with the
    level's max_iterations and epsilons (ndt_oracle.DEFAULTS' outlier_ratio / min_voxel_points)."""

    def __init__(self, vox, origin, grid_len, z_len, scan, k, normalize_cov=0, **ndt):
        super().__init__(vox, origin, grid_len, z_len, scan, normalize_cov, **ndt)
        self.k = int(k)
        self.G = CoarseGaussians(vox, self.k, normalize_cov)
        self.d1, self.d2 = constants(self.k, grid_len, z_len, self.np["outlier_ratio"])
        self.np.update(LEVEL_DEFAULTS)

    def evaluate(self, T, with_abs=False):
        x = N.transform(T, self.p)
        pi, vi = coarse_pairs(self.G, x, self.origin, self.grid_len, self.z_len, self.k, self.np["min_voxel_points"])
        c = self.center(T)
        r = N.derivatives(self.G, x, c, pi, vi, self.d1, self.d2, with_abs)
        out = dict(score=r[0], gradient=r[1], hessian=r[2], center=c, n_points=len(self.p),
                   n_matched=len(np.unique(pi)), n_pairs=len(pi), pi=pi, vi=vi)
        if with_abs:
            out["abs"] = r[3]
        return out


def level_settings(level):
    """A factor or a dict with "factor" and any gndt_ndt_level field -> full dict."""
    d = dict(level) if isinstance(level, dict) else dict(factor=int(level))
    return dict(LEVEL_DEFAULTS, **d)


class Pyramid:
    """The map level and the levels of `factors` of one map and scan; register() runs the levels
    coarsest first, each from the pose the previous one returned, then the map level."""

    def __init__(self, vox, origin, grid_len, z_len, scan, factors, normalize_cov=0, **ndt):
        self.map = N.Problem(vox, origin, grid_len, z_len, scan, normalize_cov, **ndt)
        self.levels = {k: Level(vox, origin, grid_len, z_len, scan, k, normalize_cov, **ndt) for k in factors}

    def register(self, guess, levels):
        T, out = np.array(guess, np.float64), []
        for lv in map(level_settings, levels):
            pr = self.levels[lv["factor"]]
            pr.np.update({k: lv[k] for k in LEVEL_DEFAULTS})
            r = pr.register(T)
            out.append(r)
            T = r["pose"]
        return self.map.register(T), out
