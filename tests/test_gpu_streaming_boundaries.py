"""Parity of the streaming path (gndt_update / gndt_remove: fuse_scan in gndt_api.cu and the kernels
of gndt_update.cuh) at its own boundaries: where the match (U1) finds new or dead voxels, the three
exclusive scans (kScanTile = 1024 items, look-back groups of 32 tiles), placement of resident and new
voxels in the merged table (U5 / U6), removal down to an empty map, error paths, sequences of
updates and removes, and the numerics of the inverse merge.

Every cloud is built on purpose, as in tests/test_gpu_boundaries.py.  The tests without the gpu
marker check on the oracle alone that each construction puts its edge where it claims; the gpu tests
hold the streamed map to the full parity bar (tests/parity.py) of the BATCH build: the oracle's build
of every cloud fused so far, less the removed ones.

The resident map's origin is point 0 of its first cloud, at (0, 0, 0).  Scans have no origin point:
every point of a scan is binned against the resident origin."""
import json

import numpy as np
import pytest

from grid_ndt_b200 import _abi, synthetic
from grid_ndt_b200._abi import default_params
from tests.test_gpu_boundaries import FIN_BLOCK, GL, SI, ZL, _cloud, _edge, _gpu, _map, _oracle, _signed, _voxel
from tests.test_gpu_update import _touched_columns

SCAN_TILE, SCAN_GROUP = 1024, 32
TILE_COUNTS = [SCAN_TILE - 1, SCAN_TILE, SCAN_TILE + 1, SCAN_GROUP * SCAN_TILE, SCAN_GROUP * SCAN_TILE + 1]
LENS = np.array([GL, GL, ZL])


# ---- construction helpers ----------------------------------------------------------------

def _pts(rng, cells, counts, lo=0.1, hi=0.9):
    """counts[i] points strictly inside contiguous cell cells[i], (lo, hi) of a cell from its lower faces."""
    cells = np.asarray(cells, np.float64).reshape(-1, 3)
    counts = np.broadcast_to(np.asarray(counts, np.int64), (len(cells),))
    rep = np.repeat(cells, counts, axis=0)
    xyz = (rep + rng.uniform(lo, hi, rep.shape)) * LENS
    return np.concatenate([xyz, np.ones((len(xyz), 1))], 1).astype(np.float32)


def _shuffle(rng, *parts):
    pts = np.concatenate(parts)
    return pts[rng.permutation(len(pts))]


def _scan_params():
    return default_params(GL, ZL, SI, origin=(0, 0, 0), origin_is_first_point=0)


def _key(c):
    c = np.asarray(c, np.int64).reshape(-1, 3) + 32768
    return (c[:, 0] << 32) | (c[:, 1] << 16) | c[:, 2]


def _okeys(o):
    v = o.voxels
    c = lambda s: np.where(s > 0, s - 1, s).astype(np.int64)
    return _key(np.stack([c(v["sx"]), c(v["sy"]), c(v["sz"])], 1))


def _grid(nx, ny, nz, x0=0, y0=0, z0=0):
    """Cells of a box in table order (x, then y, then z ascending)."""
    return [(x, y, z) for x in range(x0, x0 + nx) for y in range(y0, y0 + ny) for z in range(z0, z0 + nz)]


# ---- GPU helpers ----------------------------------------------------------------------------

def _compare(m, cloud, p, exact_first=True):
    """The full parity bar against the oracle's batch build of `cloud`.  exact_first=False: first_index
    values (and so morton_list order) are taken from the oracle after the cells were found identical;
    everything else is held to the bar."""
    from oracle import oracle as O
    from tests import parity
    o32, o64 = O.oracle_build(cloud, p, "faithful32"), O.oracle_build(cloud, p, "truth64")
    v, c = m.voxels, m.columns
    if not exact_first:
        assert len(v) == len(o32.voxels) and len(c) == len(o32.columns)
        for f in ("sx", "sy", "sz", "count"):
            assert np.array_equal(v[f], o32.voxels[f]), f
        v, c = v.copy(), c.copy()
        v["first_index"] = o32.voxels["first_index"]
        c["first_index"] = o32.columns["first_index"]
    rep = parity.compare(v, c, m.slopes, m.counts(), o32, o64, p)
    assert rep["ok"], json.dumps(rep, default=str)
    return rep, o32, o64


def _check_changed(m, scan, removed=False):
    """changed_columns against the reference's change list of the scan; after a remove, the cells that
    vanished with the scan are not listed."""
    got = [(int(c["sx"]), int(c["sy"])) for c in m.columns[m.changed_columns]]
    want = _touched_columns(scan, m.origin(), GL)
    if removed:
        live = {(int(c["sx"]), int(c["sy"])) for c in m.columns}
        want = [k for k in want if k in live]
    assert got == want, (len(got), len(want))


def _tables(m):
    return m.voxels.tobytes(), m.slopes.tobytes(), m.columns.tobytes(), m.counts()


def _check_edges(m, o, p):
    from oracle import oracle as O
    from tests.test_gpu_graph import _rows
    off, tgt = m.edges()
    ooff, otgt = O.oracle_edges(o, p)
    assert _rows(off, tgt) == _rows(ooff, otgt)


# ---- 1. U1 match / U3 new keys --------------------------------------------------------------

MATCH_KINDS = ("below", "above", "interleaved", "identical", "only_new")


def match_clouds(kind, seed=0):
    """(A, B): resident cloud A (origin + 3 points in each of its cells), scan B.
      below / above: B's cells are all new, every key below / above every resident key;
      interleaved:   B holds every resident cell and one new cell between each two, so the merged
                     table alternates resident / new one by one;
      identical:     B's cells are exactly A's (n_new = 0);
      only_new:      B's cells are all new and alternate with A's in the merged table."""
    rng = np.random.default_rng(100 + MATCH_KINDS.index(kind) + seed)
    res = _grid(4, 4, 6, z0=0)
    res_cells = [c for c in res if c[2] % 2 == 0]
    new_cells = {"below": _grid(2, 4, 3, x0=-3), "above": _grid(2, 3, 4, x0=5),
                 "interleaved": [c for c in res if c[2] % 2 == 1] + res_cells, "identical": res_cells,
                 "only_new": [c for c in res if c[2] % 2 == 1]}[kind]
    a = _cloud([_pts(rng, res_cells, 3)], rng)
    b = _shuffle(rng, _pts(rng, new_cells, rng.integers(1, 5, len(new_cells))))
    return a, b


def _n_new(kind):
    return {"below": 24, "above": 24, "interleaved": 48, "identical": 0, "only_new": 48}[kind]


@pytest.mark.parametrize("kind", MATCH_KINDS)
def test_match_construction(kind):
    a, b = match_clouds(kind)
    p = default_params(GL, ZL, SI)
    ka, kb = _okeys(_oracle(a, p)), _okeys(_oracle(b, _scan_params()))
    merged = np.union1d(ka, kb)
    new = np.setdiff1d(kb, ka)
    assert len(new) == _n_new(kind)
    if kind == "below":
        assert kb.max() < ka.min()
    elif kind == "above":
        assert kb.min() > ka.max()
    elif kind == "identical":
        assert np.array_equal(ka, kb)
    else:
        is_res = np.isin(merged, ka)
        assert np.all(is_res[::2]) and not np.any(is_res[1::2]) and len(merged) == 2 * len(ka)
        assert np.array_equal(np.isin(ka, kb), np.full(len(ka), kind == "interleaved"))


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
@pytest.mark.parametrize("kind", MATCH_KINDS)
def test_match_update_and_remove(kind, demand):
    _gpu()
    a, b = match_clouds(kind)
    p = default_params(GL, ZL, SI, demand)
    m = _map()
    m.chatterCallback(a, demand)
    m.change2DMap(b)
    _compare(m, np.concatenate([a, b]), p)
    _check_changed(m, b)
    m.del2DMap(b)
    _compare(m, a, p)
    _check_changed(m, b, removed=True)
    m.close()


def invalid_scan(seed=0):
    """NaN rows and points beyond index 32767 on each axis: 0 scan voxels."""
    rng = np.random.default_rng(900 + seed)
    nan = np.full((40, 4), np.nan, np.float32)
    nan[20:, 1:] = 1.0  # NaN in x only
    far = np.ones((60, 4), np.float32)
    for k in range(3):
        far[20 * k:20 * k + 20, k] = rng.uniform(1e5, 2e5, 20) * rng.choice([-1, 1], 20)
    return _shuffle(rng, nan, far)


def test_invalid_scan_construction():
    o = _oracle(invalid_scan(), _scan_params())
    assert o.counts["n_binned"] == 0 and o.counts["n_voxels"] == 0 and o.counts["n_dropped"] == 100


@pytest.mark.gpu
def test_invalid_scan_moves_counters_not_tables():
    """A scan with no binned point: n_input and n_dropped grow, the tables stay byte-identical, the
    change list is empty, and the cloud indices of a later scan still count the dropped points."""
    _gpu()
    a, _ = match_clouds("interleaved")
    bad = invalid_scan()
    c = _shuffle(np.random.default_rng(5), _pts(np.random.default_rng(6), _grid(3, 3, 2, x0=2), 2))
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    vb, sb, cb, n0 = _tables(m)
    m.change2DMap(bad)
    v1, s1, c1, n1 = _tables(m)
    assert (v1, s1, c1) == (vb, sb, cb)
    assert n1["n_input"] == n0["n_input"] + len(bad) and n1["n_dropped"] == n0["n_dropped"] + len(bad)
    assert {k: n1[k] for k in n1 if k not in ("n_input", "n_dropped")} == {k: n0[k] for k in n0 if k not in ("n_input", "n_dropped")}
    assert len(m.changed_columns) == 0
    m.del2DMap(bad)
    assert _tables(m) == (vb, sb, cb, n0)
    m.change2DMap(bad)
    m.change2DMap(c)
    _compare(m, np.concatenate([a, bad, c]), p)
    m.close()


def disjoint_clouds(passes):
    """A small resident map around the origin; a scan whose bounding box lies elsewhere and spans the
    whole x index range, with points on index +-32767 (and the next float outward, dropped):
      5 passes: z cells 10..50 (above A's), y cells 0..8192  -> bz 6, column id 30 bits;
      6 passes: y cells 10..4106 (beside A's), z over the whole index range -> bz 16, 29 bits."""
    rng = np.random.default_rng(50 + passes)
    a = _cloud([_pts(rng, _grid(6, 6, 4, -3, -3, 0), 3)], rng)
    if passes == 5:
        lo, hi = np.array([-32767, 0, 10]), np.array([32766, 8192, 50])
    else:
        lo, hi = np.array([-32767, 10, -32767]), np.array([32766, 4106, 32766])
    corners = np.array([[(lo if (k >> i) & 1 else hi)[i] for i in range(3)] for k in range(8)])
    cells = np.concatenate([corners, rng.integers(lo, hi + 1, (3000, 3))])
    body = _pts(rng, cells, rng.integers(1, 4, len(cells)))
    extra, n_out = [], 0
    for ax in range(3):
        if hi[ax] - lo[ax] + 1 != 65534:
            continue
        inside, outside = _edge(LENS[ax], ax)
        for v in (inside, -inside, outside, -outside):
            q = _pts(rng, [(lo + hi) // 2], 1)
            q[0, ax] = v
            extra.append(q)
        n_out += 2
    return a, _shuffle(rng, body, *extra), n_out, (lo, hi)


def _planned(o):
    """(passes, bz, bcol) plan_kernel derives for an oracle map's bounding box (test_gpu_boundaries)."""
    c = lambda s: np.where(s > 0, s - 1, s)
    nx, ny, nz = (int(c(o.voxels[f]).max() - c(o.voxels[f]).min() + 1) for f in ("sx", "sy", "sz"))
    bz, bcol = max(1, int(nz - 1).bit_length()), max(1, int(nx * ny - 1).bit_length())
    B = bz + bcol
    P = max(2, -(-B // 9))
    while (B - min(bz, 8, -(-B // P)) + P - 2) // (P - 1) > 9:
        P += 1
    return P, bz, bcol


@pytest.mark.parametrize("passes", [5, 6])
def test_disjoint_scan_construction(passes):
    a, b, n_out, (lo, hi) = disjoint_clouds(passes)
    ob = _oracle(b, _scan_params())
    assert ob.counts["n_dropped"] == n_out and ob.counts["n_binned"] == len(b) - n_out
    assert _planned(ob)[0] == passes and _planned(_oracle(a, default_params(GL, ZL, SI)))[0] == 2
    assert np.abs(ob.voxels["sx"]).max() == _abi.GNDT_MAX_INDEX
    assert len(np.intersect1d(_okeys(ob), _okeys(_oracle(a, default_params(GL, ZL, SI))))) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("passes", [5, 6])
def test_disjoint_scan_update_and_remove(passes):
    """The scan's sort key is planned over the scan alone; the match runs on the absolute 48-bit key."""
    _gpu()
    a, b, n_out, _ = disjoint_clouds(passes)
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    rep, _, _ = _compare(m, np.concatenate([a, b]), p)
    assert rep["n_voxels"][0] > 3000
    m.del2DMap(b)
    _compare(m, a, p)
    m.close()


# ---- 2. the three exclusive scans at kScanTile and look-back group edges ----------------------

BIG = _grid(60, 60, 10, -30, -30, 0)  # 36000 cells in table order


def new_scan_clouds(n_scan, seed=0):
    """The scan holds exactly n_scan voxels (the items of the is_new scan): BIG[:n_scan], 1..3 points
    each.  The resident map holds the odd ones of them plus 50 cells beyond, so new and matched scan
    voxels alternate and every new voxel's slot depends on the scan's prefix."""
    rng = np.random.default_rng(n_scan + seed)
    res = BIG[1:n_scan:2] + BIG[n_scan:n_scan + 50]
    a = _cloud([_pts(rng, res, 3)], rng)
    b = _shuffle(rng, _pts(rng, BIG[:n_scan], rng.integers(1, 4, n_scan)))
    return a, b


@pytest.mark.parametrize("n_scan", TILE_COUNTS)
def test_new_scan_construction(n_scan):
    a, b = new_scan_clouds(n_scan)
    ob = _oracle(b, _scan_params())
    assert ob.counts["n_voxels"] == n_scan
    oab = _oracle(np.concatenate([a, b]), default_params(GL, ZL, SI))
    assert oab.counts["n_voxels"] == n_scan + 50
    assert len(np.setdiff1d(_okeys(ob), _okeys(_oracle(a, default_params(GL, ZL, SI))))) == (n_scan + 1) // 2


@pytest.mark.gpu
@pytest.mark.parametrize("n_scan", TILE_COUNTS)
def test_new_scan_tiles(n_scan):
    _gpu()
    a, b = new_scan_clouds(n_scan)
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    _compare(m, np.concatenate([a, b]), p)
    _check_changed(m, b)
    m.close()


def _dead_set(n_res):
    return sorted({0, 1, SCAN_TILE - 2, SCAN_TILE - 1, SCAN_TILE, SCAN_TILE + 1, 2 * SCAN_TILE - 1, 2 * SCAN_TILE,
                   SCAN_GROUP * SCAN_TILE - 1, SCAN_GROUP * SCAN_TILE, n_res - 1} & set(range(n_res)))


def dead_scan_clouds(n_res, seed=0):
    """build(A) + update(B) holds exactly n_res voxels (BIG[:n_res]); B holds every point of the voxels
    at the table indices _dead_set(n_res) (dead on both sides of the dead scan's tile and group edges)
    and one point of every third other voxel."""
    rng = np.random.default_rng(7 * n_res + seed)
    dead = _dead_set(n_res)
    live = [BIG[i] for i in range(n_res) if i not in set(dead)]
    a = _cloud([_pts(rng, live, 3)], rng)
    b = _shuffle(rng, _pts(rng, [BIG[i] for i in dead], 2), _pts(rng, live[::3], 1))
    return a, b, dead


@pytest.mark.parametrize("n_res", TILE_COUNTS)
def test_dead_scan_construction(n_res):
    a, b, dead = dead_scan_clouds(n_res)
    p = default_params(GL, ZL, SI)
    o = _oracle(np.concatenate([a, b]), p)
    assert o.counts["n_voxels"] == n_res
    for i in dead:
        assert _voxel(o, *BIG[i]) == i
    edges = (SCAN_TILE - 1, SCAN_TILE, SCAN_GROUP * SCAN_TILE - 1, SCAN_GROUP * SCAN_TILE, n_res - 1)
    assert all(i in dead for i in edges if i < n_res)
    assert _oracle(a, p).counts["n_voxels"] == n_res - len(dead)


@pytest.mark.gpu
@pytest.mark.parametrize("n_res", TILE_COUNTS)
def test_dead_scan_tiles(n_res):
    _gpu()
    a, b, dead = dead_scan_clouds(n_res)
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    assert m.counts()["n_voxels"] == n_res
    m.del2DMap(b)
    _compare(m, a, p)
    assert m.counts()["n_voxels"] == n_res - len(dead)
    _check_changed(m, b, removed=True)
    m.close()


def _markers(n_pts):
    return sorted({SCAN_TILE - 2, SCAN_TILE - 1, SCAN_TILE, SCAN_GROUP * SCAN_TILE - 1, SCAN_GROUP * SCAN_TILE, n_pts - 1}
                  & set(range(n_pts)))


def changed_scan_clouds(n_pts, seed=0):
    """A scan of exactly n_pts points (the items of the change-list scan).  Each marker position
    (_markers) holds the first and only point of a new column, so its slot in the change list comes
    straight from the scan of that position; the other points fall in resident columns."""
    rng = np.random.default_rng(3 * n_pts + seed)
    res = _grid(10, 10, 3, -5, -5, 0)
    a = _cloud([_pts(rng, res, 3)], rng)
    marks = _markers(n_pts)
    body = _pts(rng, [res[i] for i in rng.integers(0, len(res), n_pts - len(marks))], 1)
    b = np.empty((n_pts, 4), np.float32)
    is_mark = np.zeros(n_pts, bool)
    is_mark[marks] = True
    b[~is_mark] = body
    b[is_mark] = _pts(rng, [(20, k, 1) for k in range(len(marks))], 1)
    return a, b, marks


@pytest.mark.parametrize("n_pts", TILE_COUNTS)
def test_changed_scan_construction(n_pts):
    a, b, marks = changed_scan_clouds(n_pts)
    assert len(b) == n_pts
    touched = _touched_columns(b, (0.0, 0.0, 0.0), GL)
    cols = [(_signed(20), _signed(k)) for k in range(len(marks))]
    sxy = [_touched_columns(b[k:k + 1], (0.0, 0.0, 0.0), GL)[0] for k in range(n_pts)]
    pos = {}
    for k, c in enumerate(sxy):
        pos.setdefault(c, k)
    assert [pos[c] for c in cols] == marks and all(c in touched for c in cols)
    assert _oracle(b, _scan_params()).counts["n_binned"] == n_pts


@pytest.mark.gpu
@pytest.mark.parametrize("n_pts", TILE_COUNTS)
def test_changed_scan_tiles(n_pts):
    _gpu()
    a, b, _ = changed_scan_clouds(n_pts)
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    _compare(m, np.concatenate([a, b]), p)
    _check_changed(m, b)
    m.del2DMap(b)
    _compare(m, a, p)
    _check_changed(m, b, removed=True)
    m.close()


# ---- 3. U5 / U6: placement in the merged table and relabelling ---------------------------------

PLACED = {"first": (-1, -1, 0), "last": (4, 4, 9), "col_below": (1, 1, 0), "col_above": (1, 1, 8),
          "mid_below": (2, 2, 1), "mid_above": (2, 2, 7)}


def placement_clouds(seed=0):
    """Resident cells (0..3, 0..3, 2..5); the scan adds the new cells PLACED: merged index 0, the last
    index, and below / above every voxel of columns (1, 1) and (2, 2); it also adds a point to every
    second resident cell."""
    rng = np.random.default_rng(60 + seed)
    res = _grid(4, 4, 4, 0, 0, 2)
    a = _cloud([_pts(rng, res, 3)], rng)
    b = _shuffle(rng, _pts(rng, list(PLACED.values()), 3), _pts(rng, res[::2], 1))
    return a, b


def test_placement_construction():
    a, b = placement_clouds()
    o = _oracle(np.concatenate([a, b]), default_params(GL, ZL, SI))
    V = o.counts["n_voxels"]
    assert V == 64 + len(PLACED)
    assert _voxel(o, *PLACED["first"]) == 0 and _voxel(o, *PLACED["last"]) == V - 1
    for col, lo, hi in (((1, 1), "col_below", "col_above"), ((2, 2), "mid_below", "mid_above")):
        c = o.columns[(o.columns["sx"] == _signed(col[0])) & (o.columns["sy"] == _signed(col[1]))][0]
        assert _voxel(o, *PLACED[lo]) == c["voxel_begin"] and _voxel(o, *PLACED[hi]) == c["voxel_begin"] + c["voxel_count"] - 1


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_placement(demand):
    _gpu()
    a, b = placement_clouds()
    p = default_params(GL, ZL, SI, demand)
    m = _map()
    m.chatterCallback(a, demand)
    m.change2DMap(b)
    _compare(m, np.concatenate([a, b]), p)
    m.del2DMap(b)
    _compare(m, a, p)
    m.close()


def block_shift_clouds(upper_first):
    """One resident column of layers 0..299 without layer 10: layers 255 / 256 are records 254 / 255,
    both in finalize block 0.  The scan adds layer 10, which moves them to records 255 / 256, across
    the block edge: each becomes the other's halo record.  Layer 255 sits near the top of its cell,
    256 near the bottom; which of the two comes first in the cloud decides up(255) and down(256)
    (see tall_column_cloud in test_gpu_boundaries)."""
    rng = np.random.default_rng(255 + upper_first)
    layers = {k: _pts(rng, [(0, 0, k)], 3, *((0.88, 0.92) if k == 255 else (0.08, 0.12) if k == 256 else (0.4, 0.6)))
              for k in range(300) if k != 10}
    first = [256, 255] if upper_first else [255, 256]
    body = _shuffle(rng, *[layers[k] for k in layers if k not in first])
    a = _cloud([layers[first[0]], layers[first[1]], body], rng, shuffle=False)
    b = _pts(rng, [(0, 0, 10)], 3)
    return a, b


@pytest.mark.parametrize("upper_first", [True, False])
def test_block_shift_construction(upper_first):
    a, b = block_shift_clouds(upper_first)
    p = default_params(GL, ZL, SI)
    oa, o = _oracle(a, p), _oracle(np.concatenate([a, b]), p)
    assert _voxel(oa, 0, 0, 255) == FIN_BLOCK - 2 and _voxel(oa, 0, 0, 256) == FIN_BLOCK - 1
    assert _voxel(o, 0, 0, 255) == FIN_BLOCK - 1 and _voxel(o, 0, 0, 256) == FIN_BLOCK
    v = o.voxels
    up255, down256 = bool(v["flags"][FIN_BLOCK - 1] & _abi.F_UP), bool(v["flags"][FIN_BLOCK] & _abi.F_DOWN)
    assert (up255, down256) == ((False, True) if upper_first else (True, False))


@pytest.mark.gpu
@pytest.mark.parametrize("upper_first", [True, False])
def test_block_shift(upper_first):
    _gpu()
    a, b = block_shift_clouds(upper_first)
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    rep, _, _ = _compare(m, np.concatenate([a, b]), p)
    assert rep["label_mismatch"] == 0
    m.del2DMap(b)
    rep, _, _ = _compare(m, a, p)
    assert rep["label_mismatch"] == 0
    m.close()


def new_column_row_clouds(seed=0):
    """Flat resident cells in rows x = 0 and x = 2, columns y = 0, 2, 3, at two heights; the scan adds
    column (0, 1) between two resident columns of row 0, and the whole row x = 1 between two rows."""
    rng = np.random.default_rng(70 + seed)
    res = [(x, y, z) for x in (0, 2) for y in (0, 2, 3) for z in (0, 5)]
    new = [(0, 1, 0), (0, 1, 5)] + [(1, y, z) for y in (0, 1, 2, 3) for z in (0, 5)]
    a = _cloud([_flat(rng, res)], rng)
    b = _shuffle(rng, _flat(rng, new))
    return a, b


def _flat(rng, cells):
    """8 points per cell spread over its x-y extent and 1 mm in z: a near-horizontal Slope."""
    pts = _pts(rng, cells, 8)
    pts[:, 2] = ((np.repeat(np.asarray(cells)[:, 2], 8) + 0.5 + rng.uniform(-0.005, 0.005, len(pts))) * ZL).astype(np.float32)
    return pts


def test_new_column_row_construction():
    a, b = new_column_row_clouds()
    p = default_params(GL, ZL, SI)
    oa, o = _oracle(a, p), _oracle(np.concatenate([a, b]), p)
    assert len(o.columns) == len(oa.columns) + 5
    # the resident slopes next to the new cells gain reach bits towards them
    reach = lambda om, c: int(om.voxels["flags"][_voxel(om, *c)] & _abi.F_REACH_ALL)
    for c in ((0, 0, 0), (0, 2, 0), (2, 0, 0), (2, 3, 0)):
        assert reach(o, c) != reach(oa, c), c


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_new_column_and_row(demand):
    _gpu()
    a, b = new_column_row_clouds()
    p = default_params(GL, ZL, SI, demand)
    m = _map()
    m.chatterCallback(a, demand)
    m.change2DMap(b)
    rep, o, _ = _compare(m, np.concatenate([a, b]), p)
    assert rep["reach_mismatch"] == 0
    _check_edges(m, o, p)
    m.del2DMap(b)
    rep, o, _ = _compare(m, a, p)
    assert rep["reach_mismatch"] == 0
    _check_edges(m, o, p)
    m.close()


# ---- 4. remove --------------------------------------------------------------------------------

REM = _grid(6, 10, 10)  # 600 cells, 10 per column, 100 per x row
REM_DEAD = sorted({0, len(REM) - 1} | set(range(FIN_BLOCK, 2 * FIN_BLOCK)) | set(range(550, 560)))
FALL = (5, 4, 4)  # fitted with 4 points, 2 of them removed
FALL_BELOW = (5, 4, 3)
SURV = {(5, 6, 2): 1, (5, 6, 6): 2}  # survivors of 1 and 2 points under 5 removed points each


def remove_clouds(seed=0):
    """build(A) + update(B) holds the 600 cells REM.  Removing B kills the voxels at table indices
    REM_DEAD: index 0, the last index, every record of finalize block 1 (256..511: whole columns and
    the whole x row 3) and column (5, 5).  FALL drops from 4 points to 2 (below min_points): its Slope
    disappears and FALL_BELOW, which saw it as fitted before itself, gains UP.  SURV keeps 1 and 2
    points.  B also holds one point of every third other voxel."""
    rng = np.random.default_rng(80 + seed)
    dead = set(REM_DEAD)
    special = {FALL, FALL_BELOW, *SURV}
    live = [c for i, c in enumerate(REM) if i not in dead and c not in special]
    first = [_pts(rng, [FALL], 2, 0.1, 0.15), _pts(rng, [FALL_BELOW], 3, 0.85, 0.9)]
    a = _cloud(first + [_shuffle(rng, _pts(rng, live, 3), *[_pts(rng, [c], k) for c, k in SURV.items()])], rng, shuffle=False)
    b = _shuffle(rng, _pts(rng, [REM[i] for i in REM_DEAD], 2), _pts(rng, live[::3], 1), _pts(rng, [FALL], 2, 0.1, 0.15),
                 _pts(rng, list(SURV), 5))
    return a, b


def test_remove_construction():
    a, b = remove_clouds()
    p = default_params(GL, ZL, SI)
    o, oa = _oracle(np.concatenate([a, b]), p), _oracle(a, p)
    assert o.counts["n_voxels"] == len(REM) and oa.counts["n_voxels"] == len(REM) - len(REM_DEAD)
    for i in (0, FIN_BLOCK - 1, FIN_BLOCK, 2 * FIN_BLOCK - 1, 2 * FIN_BLOCK, 550, len(REM) - 1):
        assert _voxel(o, *REM[i]) == i
    assert not np.any(oa.voxels["sx"] == _signed(3))  # the whole x row 3 is gone
    f = lambda om, c: int(om.voxels["flags"][_voxel(om, *c)])
    assert f(o, FALL) & _abi.F_FITTED and not f(oa, FALL) & _abi.F_FITTED
    assert not f(o, FALL_BELOW) & _abi.F_UP and f(oa, FALL_BELOW) & _abi.F_UP
    for c, k in SURV.items():
        assert int(oa.voxels["count"][_voxel(oa, *c)]) == k


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_remove(demand):
    _gpu()
    a, b = remove_clouds()
    p = default_params(GL, ZL, SI, demand)
    m = _map()
    m.chatterCallback(a, demand)
    m.change2DMap(b)
    _compare(m, np.concatenate([a, b]), p)
    m.del2DMap(b)
    _, o, _ = _compare(m, a, p)
    _check_changed(m, b, removed=True)
    _check_edges(m, o, p)
    m.close()


@pytest.mark.gpu
def test_remove_in_two_halves():
    _gpu()
    a, b = remove_clouds(seed=1)
    p = default_params(GL, ZL, SI, "true")
    h = len(b) // 2
    m = _map()
    m.chatterCallback(a, "true")
    m.change2DMap(b)
    m.del2DMap(b[:h])
    _compare(m, np.concatenate([a, b[h:]]), p, exact_first=False)
    _check_changed(m, b[:h], removed=True)
    m.del2DMap(b[h:])
    _compare(m, a, p)
    _check_changed(m, b[h:], removed=True)
    m.close()


@pytest.mark.gpu
def test_remove_everything_then_update():
    """The map empties; an update then equals the batch build of the origin and the new scan, cloud
    indices included."""
    _gpu()
    a, _ = remove_clouds(seed=2)
    c, _ = match_clouds("above", seed=3)
    c = c[1:]
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.del2DMap(a[1:])
    n = m.counts()
    assert n["n_voxels"] == n["n_columns"] == n["n_slopes"] == n["n_binned"] == 0 and n["n_input"] == 1
    assert len(m.voxels) == len(m.columns) == len(m.slopes) == 0
    m.change2DMap(c)
    _compare(m, np.concatenate([a[:1], c]), p)
    _check_changed(m, c)
    m.close()


@pytest.mark.gpu
def test_remove_errors_leave_the_map_unchanged():
    """GNDT_ERR_STATE when a scan voxel holds one point more than the resident voxel, and when a scan
    key is absent from the map; tables and counters stay byte-identical."""
    _gpu()
    from grid_ndt_b200 import GndtError
    a, b = remove_clouds(seed=3)
    rng = np.random.default_rng(4)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    before = _tables(m)
    o = _oracle(np.concatenate([a, b]), default_params(GL, ZL, SI))
    k = int(o.voxels["count"][_voxel(o, *REM[300])])
    for bad in (_shuffle(rng, b[:100], _pts(rng, [REM[300]], k + 1)), _shuffle(rng, b[:100], _pts(rng, [(9, 9, 9)], 1))):
        m.del2DMap(bad)
        with pytest.raises(GndtError) as e:
            m.counts()
        assert e.value.status == _abi.GNDT_ERR_STATE
        assert _tables(m) == before
    m.del2DMap(b)  # a valid remove still works afterwards
    _compare(m, a, default_params(GL, ZL, SI))
    m.close()


# ---- 5. sequences -------------------------------------------------------------------------------

def sequence_clouds():
    cloud = synthetic.cfg2(360_000, scale=0.2)
    return cloud[:200_000], cloud[200_000:240_000], cloud[240_000:280_000], cloud[280_000:320_000], cloud[320_000:]


def test_sequence_construction():
    a, b1, b2, c, d = sequence_clouds()
    p = default_params(GL, ZL, SI)
    assert _oracle(a, p).counts["n_binned"] == len(a) - 1
    for s in (b1, b2, c, d):
        o = _oracle(s, _scan_params())
        assert o.counts["n_binned"] == len(s) and o.counts["n_voxels"] > 1000


@pytest.mark.gpu
def test_update_remove_update():
    """build(A) + update(B) + remove(B) + update(C) == build(A ++ C), first_index and morton_list
    order included: removing the most recent scan gives its cloud indices back."""
    _gpu()
    a, b, _, c, _ = sequence_clouds()
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    _check_changed(m, b)
    m.del2DMap(b)
    _check_changed(m, b, removed=True)
    assert m.counts()["n_input"] == len(a)
    m.change2DMap(c)
    _check_changed(m, c)
    _compare(m, np.concatenate([a, c]), p)
    assert int(m.voxels["first_index"].max()) < m.counts()["n_input"]
    m.close()


@pytest.mark.gpu
def test_two_updates_remove_last_update():
    """build(A) + update(B1) + update(B2) + remove(B2) + update(C) == build(A ++ B1 ++ C)."""
    _gpu()
    a, b1, b2, c, _ = sequence_clouds()
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    for s in (b1, b2):
        m.change2DMap(s)
        _check_changed(m, s)
    m.del2DMap(b2)
    _check_changed(m, b2, removed=True)
    _compare(m, np.concatenate([a, b1]), p)
    m.change2DMap(c)
    _check_changed(m, c)
    _compare(m, np.concatenate([a, b1, c]), p)
    m.close()


@pytest.mark.gpu
def test_remove_older_scan():
    """Removing a scan that is not the most recent: the map equals the batch build without it except
    for first_index values (voxels the removed scan touched first keep its indices, and a later update
    reuses indices).  demand "true" labels do not depend on first-seen order."""
    _gpu()
    a, b, c, d, _ = sequence_clouds()
    p = default_params(GL, ZL, SI, "true")
    m = _map()
    m.chatterCallback(a, "true")
    m.change2DMap(b)
    m.change2DMap(c)
    m.del2DMap(b)
    _check_changed(m, b, removed=True)
    _compare(m, np.concatenate([a, c]), p, exact_first=False)
    assert m.counts()["n_input"] == len(a) + len(c)
    m.change2DMap(d)
    _check_changed(m, d)
    _compare(m, np.concatenate([a, c, d]), p, exact_first=False)
    m.close()


# ---- 6. numerics of the inverse merge -------------------------------------------------------

# (survivor points, survivor spread in m, removed points in the same voxel)
SURVIVORS = [(3, 1e-3, 1_000_000), (4, 1e-3, 200_000), (5, 1e-3, 100_000), (3, 1e-3, 100_000),
             (3, 1e-2, 500_000), (4, 1e-2, 100_000), (5, 1e-2, 100_000), (3, 1e-2, 100_000)]
DEGENERATE = [("identical", 100_000), ("collinear", 100_000)]


def survivor_clouds(X, seed=0):
    """A = origin + a few tightly clustered points in each survivor cell near (X, X, X); B = a large
    removed mass spread uniformly over each of those cells.  The cells lie two columns apart.
    Returns (A, B, survivor cells, degenerate cells)."""
    rng = np.random.default_rng(int(X) + seed)
    base = np.array([int(X / GL), int(X / GL), int(X / ZL)])
    cells = [tuple(base + [2 * k, 0, 0]) for k in range(len(SURVIVORS) + len(DEGENERATE))]
    surv, mass = [], []
    for (n, spread, nb), c in zip(SURVIVORS, cells):
        centre = (np.array(c) + rng.uniform(0.3, 0.7, 3)) * LENS
        xyz = centre + rng.uniform(-spread / 2, spread / 2, (n, 3))
        surv.append(np.concatenate([xyz, np.ones((n, 1))], 1).astype(np.float32))
        mass.append(_pts(rng, [c], nb, 0.001, 0.999))
    for (kind, nb), c in zip(DEGENERATE, cells[len(SURVIVORS):]):
        q = _pts(rng, [c], 1, 0.3, 0.7)
        q = np.repeat(q, 3, 0)
        if kind == "collinear":
            q[:, 0] = q[0, 0] + np.array([0.0, 3e-3, 7e-3], np.float32)
        surv.append(q.astype(np.float32))
        mass.append(_pts(rng, [c], nb, 0.001, 0.999))
    a = _cloud(surv, rng, shuffle=False)
    return a, _shuffle(rng, *mass), cells[:len(SURVIVORS)], cells[len(SURVIVORS):]


XS = [10.0, 100.0, 1000.0]


@pytest.mark.parametrize("X", XS)
def test_survivor_construction(X):
    a, b, cells, degen = survivor_clouds(X)
    p = default_params(GL, ZL, SI)
    o, oa = _oracle(np.concatenate([a, b]), p), _oracle(a, p)
    assert o.counts["n_voxels"] == oa.counts["n_voxels"] == len(cells) + len(degen)
    for (n, _, nb), c in zip(SURVIVORS, cells):
        assert int(o.voxels["count"][_voxel(o, *c)]) == n + nb and int(oa.voxels["count"][_voxel(oa, *c)]) == n
    assert len(a) + len(b) < 4_000_000
    # the batch build of a degenerate survivor has an exactly zero / rank-1 scatter
    from oracle import oracle as O
    t = O.oracle_build(a, p, "truth64").voxels
    s = t["scatter"][_voxel(oa, *degen[0])]
    assert np.all(s == 0)
    s = t["scatter"][_voxel(oa, *degen[1])]
    assert s[0] > 0 and np.all(s[1:] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("X", XS)
def test_survivor_scatter(X):
    """A scan adds 1e5..1e6 points to voxels far from the origin that hold a few tightly clustered
    points, and is removed again: the survivors' mean and scatter must come back at the 1e-5 bar
    against truth64, which is the bar at 1000 m, where the binary32 oracle's own scatter is noise."""
    _gpu()
    from oracle import oracle as O
    from tests import parity
    a, b, cells, degen = survivor_clouds(X)
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    m.del2DMap(b)
    o32, o64 = O.oracle_build(a, p, "faithful32"), O.oracle_build(a, p, "truth64")
    v = m.voxels
    idx = [_voxel(o32, *c) for c in cells]
    g, t = v["scatter"][idx].astype(np.float64), o64.voxels["scatter"][idx].astype(np.float64)
    err = np.abs(g - t).max(axis=1) / np.abs(t).max(axis=1)
    gm, tm = v["mean"][idx].astype(np.float64), o64.voxels["mean"][idx].astype(np.float64)
    merr = np.abs(gm - tm).max(axis=1) / np.maximum(1.0, np.abs(tm).max(axis=1))
    dg = {k: v["scatter"][_voxel(o32, *c)].tolist() for (k, _), c in zip(DEGENERATE, degen)}
    print(json.dumps({"X": X, "scatter_rel_err_vs_truth64": err.tolist(), "mean_rel_err_vs_truth64": merr.tolist(),
                      "degenerate_scatter": dg}))
    assert err.max() <= parity.REL_TOL, err.tolist()
    assert merr.max() <= parity.REL_TOL, merr.tolist()
    rep = parity.compare(v, m.columns, m.slopes, m.counts(), o32, o64, p)
    assert rep["ok"], json.dumps(rep, default=str)
    m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("X", XS)
def test_degenerate_survivors(X):
    """Three identical points and three points on an x line survive a removed mass: the batch build
    gives an exactly zero and a rank-1 scatter (only xx non-zero), and so must the inverse merge."""
    _gpu()
    a, b, _, degen = survivor_clouds(X)
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    m.del2DMap(b)
    o = _oracle(a, default_params(GL, ZL, SI))
    v = m.voxels
    ident, line = v[_voxel(o, *degen[0])], v[_voxel(o, *degen[1])]
    assert np.all(ident["scatter"] == 0), ident["scatter"].tolist()
    assert ident["rough"] == np.float32(0.01) and ident["evals"].tolist() == [0.0, 0.0, 0.0]
    assert line["scatter"][0] > 0 and np.all(line["scatter"][1:] == 0), line["scatter"].tolist()
    assert line["rough"] == np.float32(0.01)
    for r, w in ((ident, o.voxels[_voxel(o, *degen[0])]), (line, o.voxels[_voxel(o, *degen[1])])):
        assert np.array_equal(r["normal"], w["normal"]) and r["flags"] == w["flags"]
    m.close()
