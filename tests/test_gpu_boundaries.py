"""Parity at the kernels' own boundaries: reduce tiles and the carry chain (gndt_reduce.cuh), the
key layout and index range the planner derives (plan_kernel, gndt_sort.cuh), finalize blocks and
their halo records (finalize_label_kernel, gndt_label.cuh), parameters the defaults never set,
capacity at the exact edge and a handle reused across builds.

Every cloud is built on purpose.  The tests without the gpu marker check, on the oracle alone,
that each construction really puts the edge it claims where it claims it; the gpu tests then hold
the GPU build to the full parity bar (tests/parity.py) on the same clouds.

Positions in the sorted stream: in the oracle's table order, voxel i holds sorted-stream
positions [cumsum(count)[i] - count[i], cumsum(count)[i]).  Reduce tiles are 2048 of them, sort
tiles 4096, finalize blocks 256 voxel records.

Clouds are built in contiguous index space (cell c >= 0 is signed index c + 1, c < 0 is c) about
an origin at (0, 0, 0), which is point 0 of every cloud and so is not binned itself."""
import ctypes as C
import json

import numpy as np
import pytest

from grid_ndt_b200 import _abi, synthetic
from grid_ndt_b200._abi import default_params

GL, ZL, SI = 0.2, 0.1, 0.08
RED_TILE, SORT_TILE, FIN_BLOCK = 2048, 4096, 256
LONG_RUN = 64  # runs longer than this are reduced by a whole warp (kLongRun)


# ---- construction helpers ----------------------------------------------------------------

def _signed(c):
    return c + 1 if c >= 0 else c


def _cell_points(rng, n, cx, cy, cz, gl=GL, zl=ZL, z_frac=(0.1, 0.9)):
    """n points strictly inside contiguous cell (cx, cy, cz), a tenth of a cell away from its faces."""
    x = (cx + rng.uniform(0.1, 0.9, n)) * gl
    y = (cy + rng.uniform(0.1, 0.9, n)) * gl
    z = (cz + rng.uniform(z_frac[0], z_frac[1], n)) * zl
    return np.stack([x, y, z, np.ones(n)], 1).astype(np.float32)


def _cloud(parts, rng, shuffle=True):
    """Point 0 is the origin; the parts follow in cloud order (shuffled unless told otherwise)."""
    pts = np.concatenate(parts) if parts else np.zeros((0, 4), np.float32)
    if shuffle:
        pts = pts[rng.permutation(len(pts))]
    return np.concatenate([np.array([[0, 0, 0, 1]], np.float32), pts])


def _oracle(cloud, p):
    from oracle import oracle as O
    return O.oracle_build(cloud, p, "faithful32")


def _voxel(o, cx, cy, cz):
    """Table index of contiguous cell (cx, cy, cz) in an oracle map."""
    v = o.voxels
    i = np.nonzero((v["sx"] == _signed(cx)) & (v["sy"] == _signed(cy)) & (v["sz"] == _signed(cz)))[0]
    assert len(i) == 1, f"cell {(cx, cy, cz)} holds no voxel"
    return int(i[0])


def _stream(o):
    """(start, end) sorted-stream positions of every voxel of an oracle map."""
    end = np.cumsum(o.voxels["count"].astype(np.int64))
    return end - o.voxels["count"].astype(np.int64), end


def _tiles(s, e, tile=RED_TILE):
    """How many tiles the positions [s, e) touch."""
    return (e - 1) // tile - s // tile + 1


def assert_placement(o, cell, start=None, end=None, tiles=None, tile=RED_TILE):
    """State where a voxel sits in the sorted stream and assert that the oracle puts it there."""
    i = _voxel(o, *cell)
    s, e = (int(a[i]) for a in _stream(o))
    if start is not None:
        assert s == start, f"voxel {cell} starts at {s}, not {start}"
    if end is not None:
        assert e == end, f"voxel {cell} ends at {e}, not {end}"
    if tiles is not None:
        assert _tiles(s, e, tile) == tiles, f"voxel {cell} [{s}, {e}) touches {_tiles(s, e, tile)} tiles of {tile}, not {tiles}"
    return s, e


def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked test on a box without CUDA (no fallback exists)")
    return torch


def _parity(cloud, p, demand="slope", check_reach=True):
    from tests import parity
    rep = parity.run_case(cloud, p, demand, check_reach=check_reach)
    assert rep["ok"], json.dumps({k: v for k, v in rep.items() if k != "stage_ms"}, default=str)
    return rep


def _map(gl=GL, zl=ZL, si=SI, **params):
    from grid_ndt_b200 import TwoDmap
    m = TwoDmap(gl, zl)
    m.setInterval(si)
    for k, v in params.items():
        setattr(m.params, k, v)
    return m


def _tables(m):
    return m.voxels.tobytes(), m.slopes.tobytes(), m.columns.tobytes(), m.counts()


# ---- 1. reduce tiles and the carry chain ---------------------------------------------------

LEAD = 100  # points of voxel A, the first voxel of the stream, so that V starts mid-tile
MID = 564   # where V ends inside its last tile in endings (b) and (c)
SPANS = (1, 2, 31, 32, 33, 34, 64, 65, 66)
ENDINGS = ("a", "b", "c")


def chain_cloud(span, ending, seed=0, origin_point=True):
    """A (LEAD points, cell (-1, 0, 0)) opens the stream; V (cell (0, 0, 0)) follows and touches
    `span` reduce tiles; W (cell (0, 0, 1)) and X (cell (0, 0, 2)) follow V in the same column.
      a: V ends exactly at a tile end; W starts at offset 0 of the next tile and spills over.
      b: V ends mid-tile (offset MID) and W spills into the following tile: V's continuation
         chain ends in its last tile while the next tile carries W's lead.
      c: V ends mid-tile and W closes in the same tile; X spills into the following tile.
    Returns (cloud, placement) with placement = {cell: (start, end)} of the sorted stream."""
    rng = np.random.default_rng(1000 * span + ord(ending) + seed)
    end_v = span * RED_TILE if ending == "a" else (span - 1) * RED_TILE + MID
    n_w = 500 if ending == "c" else 3000
    n_x = 3000 if ending == "c" else 0
    a = _cell_points(rng, LEAD, -1, 0, 0, z_frac=(0.2, 0.8))
    v = _cell_points(rng, end_v - LEAD, 0, 0, 0)
    w = _cell_points(rng, n_w, 0, 0, 1)
    x = _cell_points(rng, n_x, 0, 0, 2)
    parts = [a, v, w, x]
    pts = _cloud(parts, rng) if origin_point else np.concatenate(parts)[rng.permutation(sum(map(len, parts)))]
    place = {(-1, 0, 0): (0, LEAD), (0, 0, 0): (LEAD, end_v), (0, 0, 1): (end_v, end_v + n_w)}
    if n_x:
        place[(0, 0, 2)] = (end_v + n_w, end_v + n_w + n_x)
    return pts, place


def check_chain_placement(o, span, ending, place):
    for cell, (s, e) in place.items():
        assert_placement(o, cell, start=s, end=e)
    s, e = place[(0, 0, 0)]
    assert _tiles(s, e) == span and s % RED_TILE != 0
    last = (e - 1) // RED_TILE  # V's last tile
    ws, we = place[(0, 0, 1)]
    if ending == "a":
        assert e % RED_TILE == 0 and ws % RED_TILE == 0 and (we - 1) // RED_TILE > last  # W: run at offset 0, spills
    elif ending == "b":
        assert e % RED_TILE == MID and ws // RED_TILE == last and (we - 1) // RED_TILE == last + 1
    else:
        assert e % RED_TILE == MID and (we - 1) // RED_TILE == last
        xs, xe = place[(0, 0, 2)]
        assert xs // RED_TILE == last and (xe - 1) // RED_TILE == last + 1


@pytest.mark.parametrize("ending", ENDINGS)
@pytest.mark.parametrize("span", SPANS)
def test_chain_construction(span, ending):
    cloud, place = chain_cloud(span, ending)
    o = _oracle(cloud, default_params(GL, ZL, SI))
    check_chain_placement(o, span, ending, place)


@pytest.mark.gpu
@pytest.mark.parametrize("ending", ENDINGS)
@pytest.mark.parametrize("span", SPANS)
def test_chain_parity(span, ending):
    _gpu()
    cloud, place = chain_cloud(span, ending)
    rep = _parity(cloud, default_params(GL, ZL, SI))
    assert rep["counts"]["n_binned"] == place[max(place)][1]


def run_length_cloud(seed=0):
    """One column of voxels whose runs are 62..67 points long (both sides of kLongRun), several
    of each length lying entirely inside one reduce tile."""
    rng = np.random.default_rng(77 + seed)
    lens = [62, 63, 64, 65, 66, 67] * 12
    parts = [_cell_points(rng, n, 0, 0, k) for k, n in enumerate(lens)]
    return _cloud(parts, rng), lens


def test_run_length_construction():
    cloud, lens = run_length_cloud()
    o = _oracle(cloud, default_params(GL, ZL, SI))
    s, e = _stream(o)
    assert list(o.voxels["count"]) == lens
    inside = _tiles(s, e) == 1
    for n in (LONG_RUN, LONG_RUN + 1):
        assert np.sum(inside & (o.voxels["count"] == n)) >= 3, n


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_run_length_parity(demand):
    _gpu()
    _parity(run_length_cloud()[0], default_params(GL, ZL, SI, demand), demand)


def single_point_tail_cloud(own_voxel):
    """n_valid = 2 * 2048 + 1: the last reduce tile holds one point, either a voxel of its own or
    the end of the heavy voxel that fills the two tiles before it."""
    rng = np.random.default_rng(5 if own_voxel else 6)
    if own_voxel:
        parts = [_cell_points(rng, 2 * RED_TILE, 0, 0, 0), _cell_points(rng, 1, 0, 0, 1)]
    else:
        parts = [_cell_points(rng, 2 * RED_TILE + 1, 0, 0, 0)]
    return _cloud(parts, rng)


@pytest.mark.parametrize("own_voxel", [True, False])
def test_single_point_tail_construction(own_voxel):
    o = _oracle(single_point_tail_cloud(own_voxel), default_params(GL, ZL, SI))
    assert o.counts["n_binned"] == 2 * RED_TILE + 1
    if own_voxel:
        assert_placement(o, (0, 0, 1), start=2 * RED_TILE, end=2 * RED_TILE + 1)
    else:
        assert_placement(o, (0, 0, 0), start=0, end=2 * RED_TILE + 1, tiles=3)


@pytest.mark.gpu
@pytest.mark.parametrize("own_voxel", [True, False])
def test_single_point_tail_parity(own_voxel):
    _gpu()
    _parity(single_point_tail_cloud(own_voxel), default_params(GL, ZL, SI))


def scan_chain_clouds():
    """A resident cloud A (origin first, scattered voxels, some in the cells of the chain) and a
    scan B that holds, on its own, the 33-tile chain of ending (b)."""
    rng = np.random.default_rng(33)
    a_parts = [_cell_points(rng, 7, cx, cy, cz) for cx in range(-3, 3) for cy in range(-2, 2) for cz in range(3)]
    a = _cloud(a_parts, rng)
    b, place = chain_cloud(33, "b", seed=1, origin_point=False)
    return a, b, place


def test_scan_chain_construction():
    a, b, place = scan_chain_clouds()
    # the scan is binned against the resident map's origin (point 0 of A, at 0,0,0): every point counts
    p = default_params(GL, ZL, SI, origin=(0, 0, 0), origin_is_first_point=0)
    o = _oracle(b, p)
    assert o.counts["n_binned"] == len(b)
    check_chain_placement(o, 33, "b", place)
    ob = _oracle(np.concatenate([a, b]), default_params(GL, ZL, SI))
    assert ob.counts["n_binned"] == len(a) + len(b) - 1


@pytest.mark.gpu
def test_scan_chain_update_and_remove():
    """build(A) + update(B) == build(A + B) and remove(B) gives build(A) back, with B's front end
    (the same sort + reduce + fixup as a build) running the 33-tile chain."""
    _gpu()
    from tests.test_gpu_update import _check_against_batch
    a, b, _ = scan_chain_clouds()
    p = default_params(GL, ZL, SI)
    m = _map()
    m.chatterCallback(a, "slope")
    ref = m.voxels.copy()
    m.change2DMap(b)
    _check_against_batch(m, np.concatenate([a, b]), p)
    m.del2DMap(b)
    for f in ("sx", "sy", "sz", "count", "first_index", "column", "slope"):
        assert np.array_equal(m.voxels[f], ref[f]), f
    _check_against_batch(m, a, p)
    m.close()


# ---- 2. key layout and index range ----------------------------------------------------------

def _edge(length, axis):
    """(inside, outside): the largest float offset from the origin whose index on `axis` is
    +GNDT_MAX_INDEX according to the ABI's gndt_trans_morton_xyz, and the next float outward,
    which that function (and so the build) rejects."""
    from grid_ndt_b200 import lib
    L = lib()
    o = (C.c_float * 3)(0, 0, 0)
    s = (C.c_int32(), C.c_int32(), C.c_int32())

    def index(x):
        pos = [0.05 * GL, 0.05 * GL, 0.05 * ZL]
        pos[axis] = x
        rc = L.gndt_trans_morton_xyz(o, np.float32(GL), np.float32(ZL), (C.c_float * 3)(*pos), *[C.byref(v) for v in s])
        return s[axis].value if rc == 0 else None

    lo, hi = int(np.float32(length).view(np.uint32)), 0x7F7FFFFF  # index(length) = 1, index(FLT_MAX) rejected
    while lo + 1 < hi:
        mid = (lo + hi) // 2
        if index(float(np.uint32(mid).view(np.float32))) is not None:
            lo = mid
        else:
            hi = mid
    inside = np.uint32(lo).view(np.float32)
    outside = np.nextafter(inside, np.float32(np.inf))
    assert index(float(inside)) == _abi.GNDT_MAX_INDEX and index(float(-inside)) == -_abi.GNDT_MAX_INDEX
    assert index(float(outside)) is None and index(float(-outside)) is None
    return inside, outside


def box_cloud(nx, ny, nz, n_fill=3000, extremes=False, seed=0):
    """Points whose contiguous index box is nx x ny x nz (lowest cell -(n // 2) on each axis):
    the 8 corner cells plus n_fill random cells inside.  With extremes, the box must span the whole
    index range on an axis: there the extreme points sit on the last float that still bins
    (index +-32767), and the next float outward is added as well and must be dropped."""
    rng = np.random.default_rng(seed + nx + 7 * ny + 13 * nz)
    lo = np.array([-(nx // 2), -(ny // 2), -(nz // 2)])
    hi = lo + np.array([nx, ny, nz]) - 1
    lens = np.array([GL, GL, ZL])
    corners = np.array([[(lo if (k >> a) & 1 else hi)[a] for a in range(3)] for k in range(8)])
    cells = np.concatenate([corners, rng.integers(lo, hi + 1, (n_fill, 3))])
    xyz = (cells + rng.uniform(0.1, 0.9, cells.shape)) * lens
    pts = [np.concatenate([xyz, np.ones((len(xyz), 1))], 1).astype(np.float32)]
    n_out = 0
    if extremes:
        for a in range(3):
            if (nx, ny, nz)[a] != 65534:
                continue
            inside, outside = _edge(lens[a], a)
            for v in (inside, -inside, outside, -outside):
                p = np.array([[0.5 * GL, 0.5 * GL, 0.5 * ZL, 1]], np.float32)
                p[0, a] = v
                pts.append(p)
            n_out += 2
    return _cloud(pts, rng), n_out


# (nx, ny, nz) -> (live passes, z field bits, column id bits), from plan_kernel's rule with
# 9-bit digits and a first digit of at most 8 bits inside the z field
LAYOUTS = [
    ((4, 4, 1), 2, 1, 4),
    ((64, 64, 2), 3, 1, 12),
    ((2000, 2000, 256), 4, 8, 22),
    ((8000, 8000, 512), 4, 9, 26),
    ((65534, 65534, 1), 5, 1, 32),
    ((65534, 65534, 65534), 6, 16, 32),
]


def _box_of(o):
    c = lambda s: np.where(s > 0, s - 1, s)
    return tuple(int(c(o.voxels[f]).max() - c(o.voxels[f]).min() + 1) for f in ("sx", "sy", "sz"))


@pytest.mark.parametrize("box,passes,bz,bcol", LAYOUTS)
def test_key_layout_construction(box, passes, bz, bcol):
    cloud, n_out = box_cloud(*box, extremes=True)
    o = _oracle(cloud, default_params(GL, ZL, SI))
    assert _box_of(o) == box
    assert o.counts["n_dropped"] == n_out and o.counts["n_binned"] == len(cloud) - 1 - n_out
    if 65534 in box:
        assert n_out > 0 and np.abs(o.voxels["sx"]).max() == _abi.GNDT_MAX_INDEX
    # the planner's rule, restated: the fewest passes P >= 2 whose first digit fits min(bz, 8) bits
    # and whose other digits fit 9 bits, the bits spread evenly
    nx, ny, nz = box
    assert bz == max(1, int(nz - 1).bit_length()) and bcol == max(1, int(nx * ny - 1).bit_length())
    B = bz + bcol
    P = max(2, -(-B // 9))
    while (B - min(bz, 8, -(-B // P)) + P - 2) // (P - 1) > 9:
        P += 1
    assert P == passes


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
@pytest.mark.parametrize("box,passes,bz,bcol", LAYOUTS)
def test_key_layout_parity(box, passes, bz, bcol, demand):
    _gpu()
    cloud, n_out = box_cloud(*box, extremes=True)
    p = default_params(GL, ZL, SI, demand)
    rep = _parity(cloud, p, demand)
    assert rep["counts"]["n_dropped"] == n_out
    m = _map()
    m.chatterCallback(cloud, demand)
    assert m.key_layout() == {"passes": passes, "bits_col": bcol, "ny": box[1], "bits_z": bz}
    m.close()


def _sized_cloud(n_valid, seed=0):
    """n_valid binned points (plus the origin) in a 4 m x 4 m x 1 m box."""
    rng = np.random.default_rng(n_valid + seed)
    pts = np.stack([rng.uniform(-2, 2, n_valid), rng.uniform(-2, 2, n_valid), rng.uniform(-0.5, 0.5, n_valid),
                    np.ones(n_valid)], 1).astype(np.float32)
    return _cloud([pts], rng, shuffle=False)


SIZES = [1, SORT_TILE - 1, SORT_TILE, SORT_TILE + 1, 16 * SORT_TILE, 16 * SORT_TILE + 1]


def _all_dropped():
    rng = np.random.default_rng(0)
    far = np.full((500, 4), 1.0, np.float32)
    far[:, 0] = rng.uniform(1e6, 2e6, 500)  # far beyond index 32767 on x
    return _cloud([far], rng)


@pytest.mark.parametrize("n_valid", SIZES)
def test_sized_cloud_construction(n_valid):
    o = _oracle(_sized_cloud(n_valid), default_params(GL, ZL, SI))
    assert o.counts["n_binned"] == n_valid and o.counts["n_dropped"] == 0


def test_all_dropped_construction():
    o = _oracle(_all_dropped(), default_params(GL, ZL, SI))
    assert o.counts["n_binned"] == 0 and o.counts["n_dropped"] == 500 and o.counts["n_voxels"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("n_valid", SIZES)
def test_sized_cloud_parity(n_valid):
    _gpu()
    rep = _parity(_sized_cloud(n_valid), default_params(GL, ZL, SI))
    assert rep["counts"]["n_binned"] == n_valid


@pytest.mark.gpu
def test_every_point_dropped():
    """n_valid = 0: plan_kernel's empty branch (one live pass), and an empty map."""
    _gpu()
    rep = _parity(_all_dropped(), default_params(GL, ZL, SI))
    assert rep["counts"]["n_dropped"] == 500 and rep["counts"]["n_voxels"] == 0
    m = _map()
    m.chatterCallback(_all_dropped(), "slope")
    assert m.key_layout()["passes"] == 1
    assert len(m.voxels) == len(m.columns) == len(m.slopes) == 0
    m.close()


# ---- 3. finalize blocks -------------------------------------------------------------------

def voxel_count_cloud(n_vox, seed=0):
    """Exactly n_vox voxels: 4 layers per column, columns along y then x, 1..6 points each (some
    below min_points), so that labels, heads and fitted counts differ from block to block."""
    rng = np.random.default_rng(n_vox + seed)
    cells = [(cx, cy, cz) for cx in range(-40, 40) for cy in range(-16, 16) for cz in range(4)][:n_vox]
    assert len(cells) == n_vox
    parts = [_cell_points(rng, int(rng.integers(1, 7)), *c) for c in cells]
    return _cloud(parts, rng)


VOXEL_COUNTS = [FIN_BLOCK - 1, FIN_BLOCK, FIN_BLOCK + 1, 32 * FIN_BLOCK, 32 * FIN_BLOCK + 1]


@pytest.mark.parametrize("n_vox", VOXEL_COUNTS)
def test_voxel_count_construction(n_vox):
    o = _oracle(voxel_count_cloud(n_vox), default_params(GL, ZL, SI))
    assert o.counts["n_voxels"] == n_vox
    assert 0 < o.counts["n_fitted"] < n_vox


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
@pytest.mark.parametrize("n_vox", VOXEL_COUNTS)
def test_voxel_count_parity(n_vox, demand):
    _gpu()
    rep = _parity(voxel_count_cloud(n_vox), default_params(GL, ZL, SI, demand), demand)
    assert rep["counts"]["n_voxels"] == n_vox


def tall_column_cloud(upper_first):
    """One column of 300 layers (records 0..299), 3 points each: record 255 (the last of finalize
    block 0) sits near the top of its layer and record 256 (the first of block 1) near the bottom
    of its own, 0.02 m apart.  Whether each sees the other as fitted BEFORE itself (first-seen
    order) decides up(255) and down(256), and each is the other's halo record:
      upper_first: 256 comes first in the cloud, so up(255) sees it (|dz| = 0.02 -> no UP) and
                   down(256) sees the constructor's 0 for 255 (|dz| = 25.6 -> DOWN);
      otherwise:   up(255) sees 0 (UP) and down(256) sees 255 (no DOWN).
    A halo read as absent clears the label that should be set; one read with the other
    first-seen order flips both."""
    rng = np.random.default_rng(255 + upper_first)
    layers = {}
    for k in range(300):
        frac = (0.88, 0.92) if k == 255 else ((0.08, 0.12) if k == 256 else (0.4, 0.6))
        layers[k] = _cell_points(rng, 3, 0, 0, k, z_frac=frac)
    first = [256, 255] if upper_first else [255, 256]
    rest = [layers[k] for k in range(300) if k not in first]
    body = np.concatenate(rest)[rng.permutation(3 * 298)]
    return _cloud([layers[first[0]], layers[first[1]], body], rng, shuffle=False)


@pytest.mark.parametrize("upper_first", [True, False])
def test_tall_column_construction(upper_first):
    o = _oracle(tall_column_cloud(upper_first), default_params(GL, ZL, SI))
    v = o.voxels
    assert len(o.columns) == 1 and len(v) == 300
    assert _voxel(o, 0, 0, 255) == FIN_BLOCK - 1 and _voxel(o, 0, 0, 256) == FIN_BLOCK
    up255 = bool(v["flags"][FIN_BLOCK - 1] & _abi.F_UP)
    down256 = bool(v["flags"][FIN_BLOCK] & _abi.F_DOWN)
    assert (up255, down256) == ((False, True) if upper_first else (True, False))
    assert (v["first_index"][FIN_BLOCK] < v["first_index"][FIN_BLOCK - 1]) == upper_first
    assert abs(float(v["mean"][FIN_BLOCK][2]) - float(v["mean"][FIN_BLOCK - 1][2])) < SI / 2


@pytest.mark.gpu
@pytest.mark.parametrize("upper_first", [True, False])
def test_tall_column_parity(upper_first):
    _gpu()
    rep = _parity(tall_column_cloud(upper_first), default_params(GL, ZL, SI))
    assert rep["label_mismatch"] == 0


def head_at_block_edge_cloud():
    """Column 0 holds 256 voxels, so column 1's head is record 256, the first of block 1."""
    rng = np.random.default_rng(256)
    parts = [_cell_points(rng, 4, 0, 0, k) for k in range(FIN_BLOCK)] + [_cell_points(rng, 4, 0, 1, k) for k in range(40)]
    return _cloud(parts, rng)


def test_head_at_block_edge_construction():
    o = _oracle(head_at_block_edge_cloud(), default_params(GL, ZL, SI))
    assert len(o.columns) == 2 and int(o.columns["voxel_begin"][1]) == FIN_BLOCK


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_head_at_block_edge_parity(demand):
    _gpu()
    cloud = head_at_block_edge_cloud()
    _parity(cloud, default_params(GL, ZL, SI, demand), demand)
    m = _map()
    m.chatterCallback(cloud, demand)
    heads = np.nonzero(m.voxels["flags"] & _abi.F_COLUMN_HEAD)[0]
    assert list(heads) == [0, FIN_BLOCK]
    m.close()


# ---- 4. parameters the defaults never set -------------------------------------------------

def _param_cloud():
    return synthetic.cfg2(300_000, scale=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_normalize_cov(demand):
    _gpu()
    _parity(_param_cloud(), default_params(GL, ZL, SI, demand, normalize_cov=1), demand)


def _without_pairs(cloud):
    """The cloud less one point of every two-point voxel (see test_min_points_two): with
    min_points = 1 single points are fitted (an all-zero scatter, whose normal the axis-order
    rule fixes), and no voxel is left whose normal is undefined."""
    lens = np.array([GL, GL, ZL], np.float32)
    d = cloud[1:, :3] - cloud[0, :3]
    n = np.maximum(np.ceil(np.abs(d) / lens), 1).astype(np.int64)  # binary32 throughout, as the index map
    c = np.where(cloud[1:, :3] > cloud[0, :3], n - 1, -n) + 32768
    key = (c[:, 0] << 32) | (c[:, 1] << 16) | c[:, 2]
    _, first, inv, cnt = np.unique(key, return_index=True, return_inverse=True, return_counts=True)
    keep = np.ones(len(cloud), bool)
    keep[1 + first[cnt == 2]] = False
    return cloud[keep]


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
@pytest.mark.parametrize("min_points", [1, 4, 10])
def test_min_points(min_points, demand):
    _gpu()
    cloud = _without_pairs(_param_cloud()) if min_points == 1 else _param_cloud()
    rep = _parity(cloud, default_params(GL, ZL, SI, demand, min_points=min_points), demand)
    assert rep["counts"]["n_fitted"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_min_points_two(demand):
    """A two-point voxel's scatter has rank 1: the eigenspace of its smallest eigenvalue is a plane,
    so neither the GPU nor the oracle has a defined normal there, and reach bits depend on that
    normal.  Reach bits are left out; everything else is held to the full bar."""
    _gpu()
    _parity(_param_cloud(), default_params(GL, ZL, SI, demand, min_points=2), demand, check_reach=False)


def test_min_points_construction():
    o3 = _oracle(_param_cloud(), default_params(GL, ZL, SI))
    counts = o3.voxels["count"]
    for k in (1, 2, 4, 10):
        o = _oracle(_param_cloud(), default_params(GL, ZL, SI, min_points=k))
        assert o.counts["n_fitted"] == int((counts >= k).sum()) and 0 < o.counts["n_fitted"] <= len(counts)
    assert ((counts == 2).sum() > 0) and ((counts >= 10).sum() > 0) and ((counts < 10).sum() > 0)
    single = _oracle(_without_pairs(_param_cloud()), default_params(GL, ZL, SI, min_points=1)).voxels["count"]
    assert (single == 2).sum() == 0 and (single == 1).sum() > 0 and len(single) == len(counts)


REACH_PARAMS = [{"rough_max": 5e-5}, {"angle_max_deg": 10.0}, {"reach_height": np.float32(0.05)},
                {"rough_max": 5e-5, "angle_max_deg": 10.0, "reach_height": np.float32(0.05)}]


@pytest.mark.parametrize("kw", REACH_PARAMS)
def test_reach_params_construction(kw):
    cloud = _param_cloud()
    base = _oracle(cloud, default_params(GL, ZL, SI))
    o = _oracle(cloud, default_params(GL, ZL, SI, **kw))
    changed = (o.voxels["flags"] & _abi.F_REACH_ALL) != (base.voxels["flags"] & _abi.F_REACH_ALL)
    assert changed.sum() > 100, kw
    assert np.array_equal(o.voxels["flags"] & 0x0F, base.voxels["flags"] & 0x0F)  # labels do not move


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
@pytest.mark.parametrize("kw", REACH_PARAMS)
def test_reach_params(kw, demand):
    _gpu()
    from oracle import oracle as O
    from tests import parity
    from tests import graph_reference as G
    cloud = _param_cloud()
    p = default_params(GL, ZL, SI, demand, **kw)
    _parity(cloud, p, demand)
    m = _map(**kw)
    m.chatterCallback(cloud, demand)
    off, tgt = m.edges()
    o = O.oracle_build(cloud, p)
    ooff, otgt = O.oracle_edges(o, p)
    assert np.array_equal(m.voxels["flags"] & parity.LABEL_BITS, o.voxels["flags"] & parity.LABEL_BITS)
    got, want = G.rows(off, tgt), G.rows(ooff, otgt)
    assert len(got) == len(want)
    bad = [i for i in range(len(got)) if got[i] != want[i]]
    if bad:  # a differing list must come from an edge within 1e-5 of a threshold
        assert parity._reach_adjacent(m.slopes["voxel"][bad], o.voxels, o.columns, p) == len(bad)
    G.assert_graph(off, tgt, m.slopes, m.columns, p, f"{kw} {demand}: ")  # exact on the GPU's own tables
    m.close()


# ---- 5. capacity at the exact edge, and one handle across builds --------------------------

@pytest.mark.gpu
def test_capacity_exact_edge_build():
    _gpu()
    from grid_ndt_b200 import GndtError
    cloud = synthetic.cfg1(60_000)
    m = _map()
    m.chatterCallback(cloud, "slope")
    V, want = m.counts()["n_voxels"], _tables(m)
    m.close()
    m = _map(max_voxels=V)
    m.chatterCallback(cloud, "slope")
    assert _tables(m) == want
    m.close()
    m = _map(max_voxels=V - 1)
    m.chatterCallback(cloud, "slope")
    with pytest.raises(GndtError) as e:
        m.counts()
    assert e.value.status == _abi.GNDT_ERR_CAPACITY
    m.close()


@pytest.mark.gpu
def test_capacity_exact_edge_update():
    _gpu()
    from grid_ndt_b200 import GndtError
    cloud = synthetic.cfg2(400_000, scale=0.2)
    a, b = cloud[:250_000], cloud[250_000:]
    m = _map()
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    V, want = m.counts()["n_voxels"], _tables(m)
    m.close()
    m = _map(max_voxels=V)
    m.chatterCallback(a, "slope")
    m.change2DMap(b)
    assert _tables(m) == want
    m.close()
    m = _map(max_voxels=V - 1)
    m.chatterCallback(a, "slope")
    before = _tables(m)
    m.change2DMap(b)
    with pytest.raises(GndtError) as e:
        m.counts()
    assert e.value.status == _abi.GNDT_ERR_CAPACITY
    assert _tables(m) == before
    m.close()


def reuse_sequence():
    """(cell lengths, cloud, live passes) of the builds one handle runs in turn."""
    seq = []
    for box, passes, _, _ in (LAYOUTS[5], LAYOUTS[0], LAYOUTS[2], LAYOUTS[4]):
        seq.append(((GL, ZL), box_cloud(*box, extremes=True, seed=1)[0], passes))
    seq.insert(2, ((GL, ZL), chain_cloud(33, "b", seed=2)[0], None))
    seq.insert(1, ((0.5, 0.05), synthetic.cfg1(80_000), None))
    seq.insert(4, ((GL, ZL), chain_cloud(65, "c", seed=3)[0], None))
    return seq


@pytest.mark.gpu
def test_one_handle_across_builds():
    """Look-back words, carries and the zeroed regions are reused from build to build: every build
    of the sequence (6 -> 2 -> 4 -> 5 live passes, cell lengths changed in between, reduce chains of
    33 and 65 tiles) must give the bytes a fresh handle gives."""
    _gpu()
    m = _map()
    for (gl, zl), cloud, passes in reuse_sequence():
        m.setLen(gl)
        m.setZLen(zl)
        m.chatterCallback(cloud, "slope")
        got = _tables(m)
        if passes is not None:
            assert m.key_layout()["passes"] == passes
        fresh = _map(gl, zl)
        fresh.chatterCallback(cloud, "slope")
        assert got == _tables(fresh), (gl, zl, len(cloud))
        fresh.close()
    m.close()
