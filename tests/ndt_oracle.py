"""numpy binary64 restatement of gndt_register (include/gndt.h): the cell key of a transformed
point, its candidate voxels, the regularised inverse covariances, the NDT score with its
gradient and Hessian, and the same Levenberg-Marquardt loop.  Works from any voxel table in
VOXEL_DTYPE: a GPU copy (gndt_copy_voxels) or a C-oracle build (oracle.oracle_build)."""
import numpy as np

MAX_INDEX = 32767
BIAS = 32768
CONVERGED, STALLED, MAX_ITER, NO_MATCH = 0, 1, 2, 3
DEFAULTS = dict(outlier_ratio=0.55, min_voxel_points=6, max_iterations=100, translation_epsilon=1e-4, rotation_epsilon=1e-4)
# the 5 candidate columns (own + 4 edge neighbours) x 3 layers
OFFSETS = [(dx, dy, dz) for dx, dy in ((-1, 0), (0, -1), (0, 0), (0, 1), (1, 0)) for dz in (-1, 0, 1)]


def axis_index(p, p0, length):
    """Contiguous signed index of binning (float32 IEEE divide and ceil) and its validity."""
    p = np.asarray(p, np.float32)
    d = np.abs(p - np.float32(p0))
    with np.errstate(invalid="ignore", over="ignore"):
        c = np.ceil(d / np.float32(length))
        ok = c <= np.float32(MAX_INDEX)
    n = np.where(ok, c, 1).astype(np.int64)
    n[n == 0] = 1
    return np.where(p > np.float32(p0), n - 1, -n), ok


def keys(x32, origin, grid_len, z_len):
    """(cx, cy, cz, valid) of float32 positions [n, 3]."""
    cx, ox = axis_index(x32[:, 0], origin[0], grid_len)
    cy, oy = axis_index(x32[:, 1], origin[1], grid_len)
    cz, oz = axis_index(x32[:, 2], origin[2], z_len)
    return cx, cy, cz, ox & oy & oz


def contiguous(s):
    s = np.asarray(s, np.int64)
    return np.where(s > 0, s - 1, s)


def _pack(cx, cy, cz):
    return ((cx + BIAS) << 32) | ((cy + BIAS) << 16) | (cz + BIAS)


class Gaussians:
    """mu, C and the usable count of every voxel of a table (count 0: not usable)."""

    def __init__(self, vox, normalize_cov=0):
        n = vox["count"].astype(np.float64)
        usable = ((vox["flags"] & 1) != 0) & (vox["count"] >= 3)
        s = vox["scatter"].astype(np.float64)
        nm1 = np.where(usable, n - 1.0, 1.0)
        sig6 = (s * n[:, None]) / nm1[:, None] if normalize_cov else s / nm1[:, None]
        ii, jj = [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]
        sig = np.zeros((len(vox), 3, 3))
        for k in range(6):
            sig[:, ii[k], jj[k]] = sig6[:, k]
            sig[:, jj[k], ii[k]] = sig6[:, k]
        sig[~usable] = np.eye(3)
        w, V = np.linalg.eigh(sig)
        lmax = w[:, 2]
        usable &= (lmax > 0) & np.isfinite(lmax)
        wr = np.maximum(w, 0.01 * lmax[:, None])
        with np.errstate(divide="ignore", invalid="ignore"):
            self.C = np.einsum("vik,vk,vjk->vij", V, 1.0 / wr, V)
        self.C[~usable] = 0.0
        self.mu = vox["mean"].astype(np.float64)
        self.count = np.where(usable, vox["count"], 0).astype(np.int64)
        self.key = _pack(contiguous(vox["sx"]), contiguous(vox["sy"]), contiguous(vox["sz"]))
        assert np.all(np.diff(self.key) > 0), "voxel table not in (cx, cy, cz) order"


def constants(grid_len, z_len, outlier_ratio):
    p_o = float(np.float32(outlier_ratio))
    V = float(np.float32(grid_len)) * float(np.float32(grid_len)) * float(np.float32(z_len))
    c1, c2 = 10.0 * (1.0 - p_o), p_o / V
    d3 = -np.log(c2)
    d1 = -np.log(c1 + c2) - d3
    d2 = -2.0 * np.log((-np.log(c1 * np.exp(-0.5) + c2) - d3) / d1)
    return d1, d2


def transform(T, p):
    """x' = R p + t in binary64, ((R_i0 p0 + R_i1 p1) + R_i2 p2) + t_i, each op rounded."""
    p = p.astype(np.float64)
    return np.stack([((T[i, 0] * p[:, 0] + T[i, 1] * p[:, 1]) + T[i, 2] * p[:, 2]) + T[i, 3] for i in range(3)], 1)


def finite_points(scan):
    p = np.asarray(scan, np.float32)[:, :3]
    return p[np.all(np.isfinite(p), axis=1)]


def pairs(G, x, origin, grid_len, z_len, min_points):
    """(point index, voxel index) of every candidate pair of positions x [n, 3] (binary64)."""
    cx, cy, cz, ok = keys(x.astype(np.float32), origin, grid_len, z_len)
    pi, vi = [], []
    idx = np.nonzero(ok)[0]
    for dx, dy, dz in OFFSETS:
        k = _pack(cx[idx] + dx, cy[idx] + dy, cz[idx] + dz)
        j = np.searchsorted(G.key, k)
        j = np.minimum(j, len(G.key) - 1)
        hit = (G.key[j] == k) & (G.count[j] >= min_points)
        pi.append(idx[hit]); vi.append(j[hit])
    return np.concatenate(pi), np.concatenate(vi)


def derivatives(G, x, c, pi, vi, d1, d2, with_abs=False):
    """S, g[6], H[6,6] summed over the pairs (and the sums of |contribution| per entry)."""
    S, g, H = 0.0, np.zeros(6), np.zeros((6, 6))
    aS, ag, aH = 0.0, np.zeros(6), np.zeros((6, 6))
    for lo in range(0, len(pi), 1 << 18):
        p, v = pi[lo:lo + (1 << 18)], vi[lo:lo + (1 << 18)]
        d = x[p] - G.mu[v]
        y = x[p] - c
        C = G.C[v]
        a = np.einsum("pij,pj->pi", C, d)
        q = np.einsum("pi,pi->p", d, a)
        e = np.exp(-0.5 * d2 * q)
        w = d1 * d2 * e
        J = np.zeros((len(p), 3, 6))
        J[:, [0, 1, 2], [0, 1, 2]] = 1.0
        # columns e_l x y
        J[:, 1, 3], J[:, 2, 3] = -y[:, 2], y[:, 1]
        J[:, 0, 4], J[:, 2, 4] = y[:, 2], -y[:, 0]
        J[:, 0, 5], J[:, 1, 5] = -y[:, 1], y[:, 0]
        ga = np.einsum("pi,pik->pk", a, J)
        jcj = np.einsum("pik,pij,pjl->pkl", J, C, J)
        dch = np.zeros_like(jcj)
        ay = np.einsum("pi,pi->p", a, y)
        for k in range(3):
            for l in range(3):
                dch[:, 3 + k, 3 + l] = 0.5 * (a[:, l] * y[:, k] + a[:, k] * y[:, l]) - (ay if k == l else 0.0)
        s = -d1 * e
        gc = w[:, None] * ga
        hc = w[:, None, None] * (-d2 * ga[:, :, None] * ga[:, None, :] + jcj + dch)
        S += s.sum(); g += gc.sum(0); H += hc.sum(0)
        if with_abs:
            aS += np.abs(s).sum(); ag += np.abs(gc).sum(0); aH += np.abs(hc).sum(0)
    return (S, g, H, (aS, ag, aH)) if with_abs else (S, g, H)


class Problem:
    """One scan against one map: vox (VOXEL_DTYPE), the map's origin / cell lengths / normalize_cov."""

    def __init__(self, vox, origin, grid_len, z_len, scan, normalize_cov=0, **ndt):
        self.G = Gaussians(vox, normalize_cov)
        self.origin, self.grid_len, self.z_len = np.asarray(origin, np.float32), np.float32(grid_len), np.float32(z_len)
        self.p = finite_points(scan)
        self.pbar = self.p.astype(np.float64).mean(0) if len(self.p) else np.zeros(3)
        self.np = dict(DEFAULTS, **ndt)
        self.d1, self.d2 = constants(grid_len, z_len, self.np["outlier_ratio"])

    def center(self, T):
        return np.array([T[i, 0] * self.pbar[0] + T[i, 1] * self.pbar[1] + T[i, 2] * self.pbar[2] + T[i, 3] for i in range(3)])

    def evaluate(self, T, with_abs=False):
        x = transform(T, self.p)
        pi, vi = pairs(self.G, x, self.origin, self.grid_len, self.z_len, self.np["min_voxel_points"])
        c = self.center(T)
        r = derivatives(self.G, x, c, pi, vi, self.d1, self.d2, with_abs)
        out = dict(score=r[0], gradient=r[1], hessian=r[2], center=c, n_points=len(self.p),
                   n_matched=len(np.unique(pi)), n_pairs=len(pi), pi=pi, vi=vi)
        if with_abs:
            out["abs"] = r[3]
        return out

    def frozen_score(self, T, pi, vi, xi):
        """S at the increment xi = (rho, phi) about c(T), pairs frozen (finite-difference checks)."""
        x = transform(T, self.p)
        c = self.center(T)
        E = so3_exp(xi[3:])
        xn = (x - c) @ E.T + c + xi[:3]
        return derivatives(self.G, xn, c, pi, vi, self.d1, self.d2)[0]

    def register(self, guess):
        T = np.array(guess, np.float64)
        cur = self.evaluate(T)
        it, term = 0, MAX_ITER
        if cur["n_pairs"] == 0:
            return dict(cur, pose=T, score=0.0, gradient=np.zeros(6), hessian=np.zeros((6, 6)), iterations=0, termination=NO_MATCH)
        lam = 1e-3
        while it < self.np["max_iterations"]:
            H, g = cur["hessian"], cur["gradient"]
            tiny = max(1e-6 * np.abs(np.diag(H)).max(), 1e-300)
            A = -H + lam * np.diag(np.maximum(-np.diag(H), tiny))
            try:
                L = np.linalg.cholesky(A)
            except np.linalg.LinAlgError:
                lam *= 10.0
                if lam > 1e12:
                    term = STALLED
                    break
                continue
            delta = np.linalg.solve(L.T, np.linalg.solve(L, g))
            if lam < 1.0 and np.linalg.norm(delta[:3]) < self.np["translation_epsilon"] and np.linalg.norm(delta[3:]) < self.np["rotation_epsilon"]:
                term = CONVERGED
                break
            E = so3_exp(delta[3:])
            c = cur["center"]
            Tn = np.eye(4)
            Tn[:3, :3] = E @ T[:3, :3]
            Tn[:3, 3] = c + delta[:3] + E @ (T[:3, 3] - c)
            cand = self.evaluate(Tn)
            it += 1
            if cand["score"] > cur["score"]:
                T, cur = Tn, cand
                lam = max(lam / 10.0, 1e-12)
            else:
                lam *= 10.0
                if lam > 1e12:
                    term = STALLED
                    break
        return dict(cur, pose=T, iterations=it, termination=term)


def so3_exp(phi):
    phi = np.asarray(phi, np.float64)
    th2 = float(phi @ phi)
    th = np.sqrt(th2)
    a = 1.0 - th2 / 6.0 if th2 < 1e-24 else np.sin(th) / th
    b = 0.5 - th2 / 24.0 if th2 < 1e-24 else (1.0 - np.cos(th)) / th2
    K = np.array([[0.0, -phi[2], phi[1]], [phi[2], 0.0, -phi[0]], [-phi[1], phi[0], 0.0]])
    return np.eye(3) + a * K + b * (K @ K)


def pose(rot_deg=(0.0, 0.0, 0.0), trans=(0.0, 0.0, 0.0)):
    """4x4 from roll/pitch/yaw in degrees (R = Rz Ry Rx) and a translation."""
    r, p, y = np.radians(rot_deg)
    Rx = np.array([[1, 0, 0], [0, np.cos(r), -np.sin(r)], [0, np.sin(r), np.cos(r)]])
    Ry = np.array([[np.cos(p), 0, np.sin(p)], [0, 1, 0], [-np.sin(p), 0, np.cos(p)]])
    Rz = np.array([[np.cos(y), -np.sin(y), 0], [np.sin(y), np.cos(y), 0], [0, 0, 1]])
    T = np.eye(4)
    T[:3, :3] = Rz @ Ry @ Rx
    T[:3, 3] = trans
    return T


def pose_error(A, B, at):
    """(distance in m between the images of the scan-frame point `at`, rotation angle in degrees)
    between two poses; `at` is the scan's centroid, so a rotation error is not counted twice."""
    dR = A[:3, :3].T @ B[:3, :3]
    ang = np.degrees(np.arccos(np.clip((np.trace(dR) - 1.0) / 2.0, -1.0, 1.0)))
    at = np.asarray(at, np.float64)
    return float(np.linalg.norm((A[:3, :3] - B[:3, :3]) @ at + A[:3, 3] - B[:3, 3])), float(ang)


def apply(T, scan):
    """Points of a scan [n, >=3] moved by T, as float32 [n, 4] (x, y, z, 1)."""
    x = transform(np.asarray(T, np.float64), np.asarray(scan, np.float32)[:, :3])
    out = np.ones((len(x), 4), np.float32)
    out[:, :3] = x
    return out


# ---- the convergence instances (shared by the CPU and GPU tests) --------------------------

PIER_CENTRE = (18.0, 12.0)  # centre of the bridge of cfg2(scale=0.3): deck, pier walls, ramps
T_TRUE = pose((0.8, -0.6, 2.5), (0.35, -0.25, 0.06))


def disc(points, centre, radius, n, rng):
    """n points drawn at random among those within `radius` (x-y) of `centre`.  Not the first n:
    the clouds are sorted by y, so a prefix of the disc is a thin strip across it."""
    near = np.nonzero(np.hypot(points[:, 0] - centre[0], points[:, 1] - centre[1]) < radius)[0]
    return points[np.sort(rng.choice(near, min(n, len(near)), replace=False))]


def convergence_instance(cloud, n_scan=30_000):
    """(map cloud, scan in the scan frame) from cfg2(900_000, scale=0.3): 600k points drawn at
    random for the map (point 0, the origin, first) and, from the remaining points, n_scan within
    10 m of the piers for the scan, moved by T_TRUE^-1.  The cloud is sorted by y before its
    64k-window shuffle, so a prefix split would give map and scan disjoint halves."""
    perm = 1 + np.random.default_rng(5).permutation(len(cloud) - 1)
    mp = cloud[np.concatenate([[0], np.sort(perm[:599_999])])]
    rest = cloud[np.sort(perm[599_999:]), :3]
    return mp, apply(np.linalg.inv(T_TRUE), disc(rest, PIER_CENTRE, 10.0, n_scan, np.random.default_rng(6)))


WORKFLOW_CENTRES = ((16.0, 8.0), (20.0, 8.0), (18.0, 12.0), (16.0, 16.0), (20.0, 16.0))


def workflow_instance(cloud):
    """(initial map cloud, [(scan in its own frame, T_true, odometry guess)] * 5) for the register ->
    transform -> update loop: 500k random points of cfg2(900_000, scale=0.3) for the map, scans of
    20k of the other points in 8 m discs around the bridge, each moved by its own T_true^-1 of up to
    2 deg / 0.3 m per axis, guesses off by GUESS_OFFSETS."""
    perm = 1 + np.random.default_rng(9).permutation(len(cloud) - 1)
    mp = cloud[np.concatenate([[0], np.sort(perm[:500_000])])]
    rest = cloud[np.sort(perm[500_000:]), :3]
    rng = np.random.default_rng(21)
    scans = []
    for c in WORKFLOW_CENTRES:
        pts = disc(rest, c, 8.0, 20_000, rng)
        T = pose(rng.uniform(-2, 2, 3), rng.uniform(-0.3, 0.3, 3))
        scan = apply(np.linalg.inv(T), pts)
        pbar = scan[:, :3].astype(np.float64).mean(0)
        guess = guesses(T, transform(T, pbar[None])[0], n=1, seed=int(rng.integers(1 << 30)), **GUESS_OFFSETS)[0]
        scans.append((scan, T, guess))
    return mp, scans


def guesses(T_true, centre, n=8, seed=11, max_t=0.1, max_deg=1.5):
    """n seeded guesses: T_true followed by offsets of up to max_t per axis and max_deg per axis,
    rotating about `centre` (where the scan lies in the map frame)."""
    rng = np.random.default_rng(seed)
    centre = np.asarray(centre, np.float64)
    out = []
    for _ in range(n):
        off = pose(rng.uniform(-max_deg, max_deg, 3), rng.uniform(-max_t, max_t, 3))
        off[:3, 3] += centre - off[:3, :3] @ centre
        out.append(off @ T_true)
    return out

# Offsets of the convergence guesses.  With 0.2 m cells, 4 mm surface noise and eigenvalues
# floored at 1 % of the largest, a ground Gaussian is ~6 mm thick: a point a few cm above it
# contributes nothing, so 0.1 m / 1.5 deg offsets lie outside the basin even of this oracle.
GUESS_OFFSETS = dict(max_t=0.01, max_deg=0.1)
