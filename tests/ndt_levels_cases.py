"""Hand-made maps and scans for the boundaries of the NDT levels (tests/test_ndt_levels.py checks
each construction on the oracle, tests/test_gpu_ndt_levels.py runs it on the GPU).

Every map has its origin at (0, 0, 0), cells of GRID x GRID x ZLEN metres (powers of two) and points
at eighth-cell offsets, so every coordinate, mean and scatter is exact in binary32 and the map
cell of a point is known in closed form: cell c of an axis holds (c + f) * len for 0 < f < 1."""
import numpy as np

GRID, ZLEN = 0.25, 0.125
# eighth-cell offsets of the points of one voxel: 4 points span all three axes, and no symmetry
# between the axes, so merged Gaussians have distinct eigenvalues (a double eigenvalue costs the
# closed-form 3x3 solver about half the binary64 digits, at the map level as at the levels)
PATTERN = np.array([(1, 2, 1), (7, 1, 5), (3, 6, 7), (5, 7, 2)], np.float64) / 8.0


def cloud_of(cells, n_points=4):
    """float32 [n, 4] cloud (origin first) with n_points (1..4, or a per-cell sequence) points in
    each cell (cx, cy, cz) of `cells` (contiguous indices)."""
    cells = np.asarray(cells, np.int64).reshape(-1, 3)
    n_points = np.broadcast_to(np.asarray(n_points), len(cells))
    pts = [np.zeros(3)]
    for c, m in zip(cells, n_points):
        pts.extend((c + PATTERN[:m]) * (GRID, GRID, ZLEN))
    out = np.ones((len(pts), 4), np.float32)
    out[:, :3] = np.array(pts)
    assert np.array_equal(out[:, :3].astype(np.float64), np.array(pts))
    return out


def block(x, y, z):
    """Every cell of the box x x y x z (three (lo, hi) ranges, hi exclusive)."""
    g = np.meshgrid(np.arange(*x), np.arange(*y), np.arange(*z), indexing="ij")
    return np.stack([a.ravel() for a in g], 1)


def edge_values(v):
    """v, and one binary32 ulp below and above it."""
    v = np.float32(v)
    return [np.nextafter(v, np.float32(-np.inf)), v, np.nextafter(v, np.float32(np.inf))]


def edge_scan(k, axis, coarse=True, around=(-3, -1, 0, 1, 2)):
    """Scan points on the cell edges of one axis (and one ulp either side): coarse edges
    X * k * len when `coarse`, else the map-cell edges (k X + j) len, 0 < j < k, in between.  The
    other two coordinates sit inside cell 0."""
    L = (GRID, GRID, ZLEN)[axis]
    cells = [X * k for X in around] if coarse else [X * k + j for X in around for j in range(1, k)]
    pts = []
    for c in cells:
        for v in edge_values(c * L):
            p = np.array([0.375 * GRID, 0.625 * GRID, 0.5 * ZLEN], np.float32)
            p[axis] = v
            pts.append(p)
    out = np.ones((len(pts), 4), np.float32)
    out[:, :3] = pts
    return out


# the map around the edge scans: all cells of [-3k, 3k) x [-k, k) x [-k, k), full
def edge_map(k):
    return cloud_of(block((-3 * k, 3 * k), (-k, k), (-k, k)))


def slab_maps(k):
    """{name: (cloud, scan)} of hand-made slab layouts at factor k, X = 0 and 1, Y = -1 .. 1.
    The scan is the map's own points."""
    out = {}
    xs, ys = range(0, 2 * k), range(-k, 2 * k)

    def cols(sel):
        c = np.array([(x, y, z) for x in xs for y in ys for z in (0, 1) if sel(x, y)], np.int64)
        return cloud_of(c)

    out["first_row"] = cols(lambda x, y: x % k == 0)
    out["last_row"] = cols(lambda x, y: x % k == k - 1)
    out["all_columns"] = cols(lambda x, y: True)
    out["missing_rows"] = cols(lambda x, y: x % k in (0, k - 1))  # rows 1 .. k-2 of each slab absent
    out["single_column"] = cols(lambda x, y: (x, y) == (k + 1, 2))
    return {n: (c, c[1:]) for n, c in out.items()}


def mixed_map(k):
    """Coarse cells mixing fitted voxels (4 points) and unfitted ones (1 or 2 points)."""
    cells = block((-k, k), (-k, k), (0, 2))
    n = np.where((cells[:, 0] + 2 * cells[:, 1] + cells[:, 2]) % 3 == 0, 4, 1 + (cells[:, 0] & 1))
    return cloud_of(cells, n)


def count_map(k):
    """Coarse cell (0, 0, 0) = two fitted voxels of 4 points (merged count 8); nothing else."""
    return cloud_of([(0, 0, 0), (k - 1, k - 1, k - 1)])


def extreme_map():
    """Map cells at contiguous index +-32766 / -32767 (signed +-32767) on x, y and z, with their
    neighbours towards the origin."""
    cells = []
    for ax in range(3):
        for c in (32765, 32766, -32766, -32767):
            p = [1, 2, 0]
            p[ax] = c
            cells.append(p)
    return cloud_of(np.array(cells))
