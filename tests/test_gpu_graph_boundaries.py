"""The traversability graph (gndt_build_edges, csrc/gndt_graph.cuh) and the reach bits (edges_kernel,
csrc/gndt_label.cuh) held to the exact rule of tests/graph_reference.py at the places where the
neighbour search and the reach predicate go wrong.

`neighbour_columns` finds the forward / back cell by a gallop from a seed (the Slope's own offset in
its x row, clamped to the neighbour row) and a bisection of the bracket.  Hand-made table pairs,
uploaded and passed to gndt_build_edges as caller tables, put every search shape exactly where it is
wanted: targets at each distance after and before the seed, at the ends of the row, absent, a clamped
seed, empty rows, the ends of the index range.  They also place reach-predicate inputs on their
thresholds, to the ulp.  Built clouds, updates and removes then run the same rule on the GPU's own
tables, through the x-row directory of column_finish_kernel.

Tests without the gpu marker check, in numpy, that each construction puts its edge where it claims
(seed against target, the gallop's path, the reference's verdict).  The gpu tests hold the kernels to
the rule: same lists in the same order and the same reach bits, except for edges the reference
marks undecided (acosf's 2-ulp freedom), which are counted and printed."""
import ctypes as C

import numpy as np
import pytest

from grid_ndt_b200 import _abi
from grid_ndt_b200._abi import COLUMN_DTYPE, SLOPE_DTYPE, default_params
from tests import graph_reference as G
from tests.test_gpu_boundaries import REACH_PARAMS, _cell_points

GL, ZL, SI = 0.2, 0.1, 0.08
MAXI = _abi.GNDT_MAX_INDEX
DISTANCES = (1, 2, 3, 4, 7, 8, 9, 15, 16, 17, 255, 256, 257, 4095, 4096, 4097)
SLOPE_FLAGS = _abi.F_FITTED | _abi.F_SLOPE
SMOOTH = np.float32(1e-6)  # rough of a Slope that passes every rough_max used here


def _params(**kw):
    return default_params(GL, ZL, SI, origin=(0.0, 0.0, 0.0), origin_is_first_point=0, **kw)


# ---- (a) the reference against the oracle --------------------------------------------------

PIN_CLOUDS = {"cfg1": ("cfg1", 60_000, {}), "cfg2": ("cfg2", 100_000, {"scale": 0.15})}


@pytest.mark.parametrize("kw", [{}] + REACH_PARAMS)
@pytest.mark.parametrize("demand", ["slope", "true"])
@pytest.mark.parametrize("cloud", sorted(PIN_CLOUDS))
def test_reference_equals_oracle(cloud, demand, kw):
    """graph_reference on an oracle build's tables gives oracle_edges (gndt_oracle_edges, which
    tests/test_adapter.py pins to the reference's own AccessibleNeighbors)."""
    from grid_ndt_b200 import synthetic
    from oracle import oracle as O
    name, n, ckw = PIN_CLOUDS[cloud]
    p = default_params(GL, ZL, SI, demand, **kw)
    o = O.oracle_build(synthetic.make(name, n, **ckw), p)
    off, tgt = O.oracle_edges(o, p)
    assert len(tgt) > 1000
    G.assert_graph(off, tgt, *G.oracle_tables(o), p, f"{cloud} {demand} {kw}: ")
    G.assert_reach_bits(G.oracle_tables(o)[0], p, label=f"{cloud} {demand} {kw}: ")


# ---- table construction ------------------------------------------------------------------

def tables(cells, layers=1):
    """(slopes, columns) of contiguous cells [(cx, cy), ...] (any order; sorted here), `layers`
    Slopes per cell (an int, or a list per cell; 0 makes a Cell without a Slope).  Every Slope is flat
    (normal +z), smooth and at z = 0.01 * layer, so all of them reach each other unless changed."""
    cells = np.asarray(cells, np.int64).reshape(-1, 2)
    order = np.lexsort((cells[:, 1], cells[:, 0]))
    cells = cells[order]
    lay = np.full(len(cells), layers, np.int64) if np.isscalar(layers) else np.asarray(layers, np.int64)[order]
    cols = np.zeros(len(cells), COLUMN_DTYPE)
    cols["sx"], cols["sy"] = G.signed(cells[:, 0]), G.signed(cells[:, 1])
    cols["slope_count"] = lay
    cols["slope_begin"] = np.r_[0, np.cumsum(lay)[:-1]] if len(lay) else []
    cols["voxel_count"] = lay
    cols["voxel_begin"] = cols["slope_begin"]
    S = int(lay.sum())
    sl = np.zeros(S, SLOPE_DTYPE)
    ci = np.repeat(np.arange(len(cells)), lay)
    k = np.arange(S) - np.repeat(cols["slope_begin"].astype(np.int64), lay)
    sl["sx"], sl["sy"], sl["sz"] = cols["sx"][ci], cols["sy"][ci], G.signed(k)
    sl["normal"] = np.array([0, 0, 1], np.float32)
    sl["mean"][:, 2] = (0.01 * k).astype(np.float32)
    sl["rough"] = SMOOTH
    sl["flags"] = SLOPE_FLAGS
    sl["voxel"] = np.arange(S)
    return sl, cols


def column_of(cols, cx, cy):
    i = np.nonzero((G.contig(cols["sx"]) == cx) & (G.contig(cols["sy"]) == cy))[0]
    assert len(i) == 1
    return int(i[0])


def row_of(cols, cx):
    c = G.contig(cols["sx"])
    return int(np.searchsorted(c, cx)), int(np.searchsorted(c, cx, "right"))


def gallop(cols, ci, dx):
    """numpy restatement of neighbour_columns' search for column ci in row cx + dx: the seed, the
    lower bound of cy in that row (offsets in the row), the probes of the gallop and its ending."""
    cx, cy = int(G.contig(cols["sx"])[ci]), int(G.contig(cols["sy"])[ci])
    own_lo, _ = row_of(cols, cx)
    r_lo, r_hi = row_of(cols, cx + dx)
    ys = G.contig(cols["sy"])
    out = {"empty": r_lo == r_hi, "len": r_hi - r_lo}
    if r_lo == r_hi:
        return out
    g = r_lo + min(ci - own_lo, r_hi - r_lo - 1)
    probes, overshoot, reached_lo = [], False, False
    if ys[g] < cy:
        lo, step = g + 1, 1
        while True:
            probe = lo + step - 1
            if probe >= r_hi:
                overshoot = True
                break
            probes.append((probe, step))
            if ys[probe] >= cy:
                break
            lo, step = probe + 1, step * 2
    else:
        hi, step = g, 1
        while True:
            if hi < r_lo + step:
                reached_lo = True
                break
            probe = hi - step
            probes.append((probe, step))
            if ys[probe] < cy:
                break
            hi, step = probe, step * 2
    t = r_lo + int(np.searchsorted(ys[r_lo:r_hi], cy))
    out.update(seed=g - r_lo, target=t - r_lo, found=t < r_hi and ys[t] == cy, probes=[(p - r_lo, s) for p, s in probes],
               overshoot=overshoot, reached_lo=reached_lo,
               probe_hit=any(p == t and s >= 2 for p, s in probes))
    return out


def gallop_tables(o, n, t, present=True, after=2):
    """Own row cx = 0 with the own column at offset o; rows cx = -1 and +1 with n columns at
    cy = 2k.  The own cy is 2t (present: column t of the neighbour rows) or 2t - 1 (absent: between
    columns t - 1 and t, below the first for t = 0, above the last for t = n).  So the search
    target is offset t, and the seed is min(o, n - 1)."""
    y = 2 * t if present else 2 * t - 1
    own = [(0, y - o + k) for k in range(o)] + [(0, y)] + [(0, y + 1 + k) for k in range(after)]
    nbr = [(dx, 2 * k) for dx in (-1, 1) for k in range(n)]
    sl, cols = tables(own + nbr)
    return sl, cols, column_of(cols, 0, y)


def _gallop_cases():
    """name -> (own offset o, neighbour row length n, target offset t, present, target - seed)."""
    c = {"at_seed": (5, 12, 5, True, 0)}
    for d in DISTANCES:
        c[f"after_{d}_last"] = (3, 3 + d + 1, 3 + d, True, d)        # the row's last column: the gallop overshoots r_hi
        c[f"after_{d}_inner"] = (3, 3 + d + 4, 3 + d, True, d)
        c[f"before_{d}_first"] = (d, d + 3, 0, True, -d)              # the row's first column: the gallop reaches r_lo
        c[f"before_{d}_inner"] = (d + 3, d + 6, 3, True, -d)
        c[f"absent_after_{d}"] = (3, 3 + d + 3, 3 + d, False, d)      # between two columns
        c[f"absent_before_{d}"] = (d + 3, d + 6, 3, False, -d)
        c[f"absent_below_{d}"] = (d, d + 3, 0, False, -d)             # below the first column
        c[f"absent_above_{d}"] = (3, 3 + d, 3 + d, False, d)          # above the last column
    for n in (1, 2):                                                  # own offset >= row length: clamped seed
        for o in (n, n + 1, n + 9, 300):
            for t in range(n + 1):
                if t < n:
                    c[f"clamp_n{n}_o{o}_t{t}"] = (o, n, t, True, t - (n - 1))
                c[f"clamp_n{n}_o{o}_t{t}_absent"] = (o, n, t, False, t - (n - 1))
    return c


GALLOP = _gallop_cases()


def _other_layouts():
    c = {}
    # an empty neighbour x row: rows -2, 0 and 2 are populated, -1 and 1 are not
    c["empty_row"] = tables([(x, y) for x in (-2, 0, 2) for y in range(6)])
    # the own row is the first (cx_lo) / last (cx_hi) row of the table
    c["first_row"] = tables([(x, y) for x in (4, 5, 6) for y in range(5)] + [(4, 9)])
    c["last_row"] = tables([(x, y) for x in (-6, -5, -4) for y in range(5)] + [(-4, 9)])
    # the -1 / +1 crossing in x and in y
    c["sign_crossing"] = tables([(x, y) for x in range(-3, 3) for y in range(-3, 3)])
    # rows at signed x = -32767 and +32767: 65534 directory rows; y at the index ends too
    ends = [-MAXI, -MAXI + 1, MAXI - 2, MAXI - 1]
    c["index_ends"] = tables([(x, y) for x in ends for y in (-MAXI, -MAXI + 1, 0, MAXI - 2, MAXI - 1)])
    # adjacency traps: row 0 ends at cy = 5 and row 1 starts at cy = 6 (not a right neighbour);
    # row 3 starts at cy = 4 and row 2 ends at cy = 3 (not a left neighbour)
    c["adjacency_traps"] = tables([(0, y) for y in range(3, 6)] + [(1, y) for y in range(6, 9)]
                                  + [(2, y) for y in range(0, 4)] + [(3, y) for y in range(4, 7)])
    # Cells without a Slope between Slope cells (and as the neighbour cell itself)
    cells = [(x, y) for x in range(3) for y in range(8)]
    c["zero_slope_columns"] = tables(cells, [0 if (x + y) % 3 == 1 else 1 + (x + y) % 2 for x, y in cells])
    # a few thousand rows whose lengths range over 1 .. 5000 (log-uniform): neighbour rows differ
    # by orders of magnitude
    rng = np.random.default_rng(2024)
    lens = np.exp(rng.uniform(0, np.log(5000), 1500)).astype(np.int64).clip(1, 5000)
    cells = []
    for x, n in enumerate(lens):
        ys = np.sort(rng.choice(12000, int(n), replace=False)) - 6000
        cells += [(x - 750, int(y)) for y in ys]
    c["random_rows"] = tables(cells)
    return c


LAYOUTS = _other_layouts()


def test_gallop_constructions():
    """Each gallop case puts the target where its name says, relative to the seed; over the set,
    the gallop hits the target with a probe of step >= 2, overshoots r_hi and reaches r_lo."""
    events = {"probe_hit": 0, "overshoot": 0, "reached_lo": 0}
    for name, (o, n, t, present, dist) in GALLOP.items():
        sl, cols, ci = gallop_tables(o, n, t, present)
        for dx in (-1, 1):
            g = gallop(cols, ci, dx)
            assert g["len"] == n and g["target"] == t and g["found"] == present, name
            assert g["seed"] == min(o, n - 1) and g["target"] - g["seed"] == dist, name
            for k in events:
                events[k] += g[k]
            if name.endswith("_last"):
                assert g["target"] == n - 1 and (g["overshoot"] or g["probe_hit"] or dist == 1), name
            if name.endswith("_first"):
                assert g["target"] == 0 and (g["reached_lo"] or any(p == 0 for p, _ in g["probes"])), name
    assert all(events.values()), events


def test_layout_constructions():
    L = LAYOUTS
    cx = lambda k: G.contig(L[k][1]["sx"])
    assert set(cx("empty_row").tolist()) == {-2, 0, 2}
    assert cx("first_row").min() == 4 and cx("last_row").max() == -4
    assert set(L["sign_crossing"][1]["sx"].tolist()) >= {-1, 1} and set(L["sign_crossing"][1]["sy"].tolist()) >= {-1, 1}
    sx = L["index_ends"][1]["sx"]
    assert sx.min() == -MAXI and sx.max() == MAXI and int(cx("index_ends").max() - cx("index_ends").min() + 1) == 65534
    cols = L["adjacency_traps"][1]
    a, b = row_of(cols, 0)[1] - 1, row_of(cols, 1)[0]
    assert b == a + 1 and G.contig(cols["sy"][b]) == G.contig(cols["sy"][a]) + 1       # right trap
    a, b = row_of(cols, 2)[1] - 1, row_of(cols, 3)[0]
    assert b == a + 1 and G.contig(cols["sy"][b]) == G.contig(cols["sy"][a]) + 1       # left trap, seen from b
    ref = G.graph_reference(*L["adjacency_traps"], _params())
    for a in (row_of(cols, 0)[1] - 1, row_of(cols, 2)[1] - 1):   # the reference does not take the trap
        assert ref.nb[a, 1] == -1 and ref.nb[a + 1, 0] == -1
    assert (L["zero_slope_columns"][1]["slope_count"] == 0).sum() >= 5
    rl = np.diff(np.r_[0, np.nonzero(np.diff(cx("random_rows")))[0] + 1, len(cx("random_rows"))])
    assert len(rl) >= 1000 and rl.min() == 1 and rl.max() >= 4000
    assert np.max(np.abs(np.diff(np.log10(rl)))) >= 3                                   # neighbours differ 1000x
    for name, (sl, cols) in L.items():
        ref = G.graph_reference(sl, cols, _params())
        assert ref.n_undecided == 0 and (ref.verdict == G.TRUE).any(), name


# ---- predicate thresholds -----------------------------------------------------------------

def _unit(theta_deg):
    t = np.radians(theta_deg)
    return np.array([np.sin(t), 0.0, np.cos(t)])


def _angle_normals(theta_deg, p, span=3000):
    """Target normals near theta_deg from +z, one float32 step of x at a time, with their verdicts."""
    base = _unit(theta_deg).astype(np.float32)
    xs = base[0] + np.arange(-span, span + 1) * np.spacing(base[0])
    n = np.zeros((len(xs), 3), np.float32)
    n[:, 0] = xs
    n[:, 2] = base[2]
    v = G.angle_verdict(G.angle_res(n, np.array([0, 0, 1], np.float32)), p.angle_max_deg)
    return n, v


def _pick(n, v, k=6):
    """Up to k normals of each verdict, those closest to the verdict boundary first."""
    out = []
    for want in (G.TRUE, G.FALSE, G.UNDECIDED):
        idx = np.nonzero(v == want)[0]
        edge = np.nonzero(np.diff(v) != 0)[0]
        if len(idx) and len(edge):
            idx = idx[np.argsort(np.min(np.abs(idx[:, None] - edge[None, :]), axis=1), kind="stable")]
        out.append(n[idx[:k]])
    return out


def _nan_pairs(rng, count=8):
    """(source, target) normals, nearly parallel and not unit length, whose res rounds above 1 (so
    acosf gives NaN and the target is unreachable): found by search."""
    found = []
    while len(found) < count:
        s = rng.normal(size=(4096, 3)).astype(np.float32)
        t = (s * rng.uniform(0.5, 2.0, (4096, 1))).astype(np.float32)
        found += [(s[i], t[i]) for i in np.nonzero(G.angle_res(t, s) > 1)[0]]
    return found[:count]


def threshold_tables(p):
    """Source column (0, 0): one flat Slope (normal +z, z = 0) and one with F_UP (its own UP does not
    matter).  Column (0, 1): target Slopes whose normal, |dz|, rough or F_UP sit on the thresholds."""
    rng = np.random.default_rng(7)
    targets = []  # (normal, z, rough, flags)
    flat = np.array([0, 0, 1], np.float32)
    for theta in (p.angle_max_deg, 180.0 - p.angle_max_deg):  # the threshold and the fold at 90
        for grp in _pick(*_angle_normals(theta, p)):
            targets += [(nn, 0.0, SMOOTH, SLOPE_FLAGS) for nn in grp]
    targets.append((-flat, 0.0, SMOOTH, SLOPE_FLAGS))                                  # antiparallel: 180 -> 0
    targets.append((np.zeros(3, np.float32), 0.0, SMOOTH, SLOPE_FLAGS))                # zero normal: NaN
    h, r = np.float32(p.reach_height), np.float32(p.rough_max)
    for z in (np.nextafter(h, np.float32(0)), h, np.nextafter(h, np.float32(1e9))):
        targets += [(flat, z, SMOOTH, SLOPE_FLAGS), (flat, -z, SMOOTH, SLOPE_FLAGS)]
    for rough in (np.nextafter(r, np.float32(0)), r, np.nextafter(r, np.float32(1e9))):
        targets.append((flat, 0.0, rough, SLOPE_FLAGS))
    targets.append((flat, 0.0, SMOOTH, SLOPE_FLAGS | _abi.F_UP))                        # an UP target
    nan = _nan_pairs(rng)  # each pair in cells (2, 2k) and (2, 2k + 1)
    sl, cols = tables([(0, 0), (0, 1)] + [(2, k) for k in range(2 * len(nan))], [2, len(targets)] + [1] * (2 * len(nan)))
    sl["flags"][1] |= _abi.F_UP
    for k, (nn, z, rough, flags) in enumerate(targets):
        sl["normal"][2 + k], sl["rough"][2 + k], sl["flags"][2 + k], sl["mean"][2 + k, 2] = nn, rough, flags, z
    for k, (a, b) in enumerate(nan):
        sl["normal"][2 + len(targets) + 2 * k], sl["normal"][3 + len(targets) + 2 * k] = a, b
    sl["mean"][2 + len(targets):, 2] = 0.0
    sl["mean"][:2, 2] = 0.0
    return sl, cols


THRESHOLD_PARAMS = [{}] + REACH_PARAMS


def _set(p, kw):
    for k, v in kw.items():
        setattr(p, k, v)
    return p


@pytest.mark.parametrize("kw", THRESHOLD_PARAMS)
def test_threshold_constructions(kw):
    p = _set(_params(), kw)
    sl, cols = threshold_tables(p)
    ref = G.graph_reference(sl, cols, p)
    v = ref.verdict[ref.cand_src == 0]  # the flat source's candidates, in target order
    tg = sl[ref.cand_tgt[ref.cand_src == 0]]
    assert (v == G.TRUE).any() and (v == G.FALSE).any() and (v == G.UNDECIDED).any()
    res = G.angle_res(sl["normal"][ref.cand_tgt], sl["normal"][ref.cand_src])
    assert (res > 1).sum() >= 8 and np.all(ref.verdict[res > 1] == G.FALSE)
    assert np.all(v[np.all(tg["normal"] == 0, axis=1)] == G.FALSE)
    assert np.all(v[np.all(tg["normal"] == [0, 0, -1], axis=1)] == G.TRUE)
    dz = np.abs(tg["mean"][:, 2])
    h = np.float32(p.reach_height)
    flat = np.all(tg["normal"] == [0, 0, 1], axis=1) & (tg["rough"] == SMOOTH) & ((tg["flags"] & _abi.F_UP) == 0)
    assert np.all(v[flat & (dz == h)] == G.TRUE) and np.all(v[flat & (dz > h)] == G.FALSE) and (flat & (dz == h)).sum() == 2
    r = np.float32(p.rough_max)
    rough = np.all(tg["normal"] == [0, 0, 1], axis=1) & (dz == 0) & ((tg["flags"] & _abi.F_UP) == 0)
    assert np.all(v[rough & (tg["rough"] == r)] == G.TRUE) and np.all(v[rough & (tg["rough"] > r)] == G.FALSE)
    assert np.all(v[(tg["flags"] & _abi.F_UP) != 0] == G.FALSE)
    # the UP source has the same candidates and verdicts as the flat one
    assert np.array_equal(ref.verdict[ref.cand_src == 1], v)


# ---- CSR sizes ------------------------------------------------------------------------------

CSR_SIZES = (1, 1023, 1024, 1025, 2047, 2048, 2049, 64 * 1024 + 1)


def sized_tables(S):
    """S Slopes, one per cell, in a band of rows 32 cells wide: most Slopes have 2-4 edges."""
    return tables([(k // 32, k % 32) for k in range(S)])


def last_only_tables():
    """Isolated cells (every second cy) except the last two, (0, 200) and (0, 201): the last Slope
    reaches (0, 200), whose own candidate, the last Slope, is too rough."""
    sl, cols = tables([(0, 2 * k) for k in range(101)] + [(0, 201)])
    sl["rough"][-1] = np.float32(1e3)
    return sl, cols


def max_degree_tables():
    """A cell and its four neighbours with 64 Slopes each, all reachable: 256 edges per Slope of the centre."""
    sl, cols = tables([(0, 0), (0, -1), (0, 1), (1, 0), (-1, 0)], 64)
    sl["mean"][:, 2] = 0.0
    return sl, cols


def test_csr_constructions():
    for S in CSR_SIZES:
        sl, cols = sized_tables(S)
        assert len(sl) == S
    off, tgt = G.graph_reference(*last_only_tables(), _params()).csr()
    deg = np.diff(off.astype(np.int64))
    assert deg[-1] > 0 and deg[:-1].sum() == 0
    sl, cols = max_degree_tables()
    off, _ = G.graph_reference(sl, cols, _params()).csr()
    c = column_of(cols, 0, 0)
    b = int(cols["slope_begin"][c])
    assert np.all(np.diff(off.astype(np.int64))[b:b + 64] == 256)


# ---- GPU helpers ------------------------------------------------------------------------------

def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked test on a box without CUDA (no fallback exists)")
    return torch


def _dev(arr):
    torch = _gpu()
    b = np.ascontiguousarray(arr).view(np.uint8).reshape(-1)
    return torch.from_numpy(b.copy() if len(b) else np.zeros(64, np.uint8)).cuda()


def _handle(**kw):
    from grid_ndt_b200 import TwoDmap
    m = TwoDmap(GL, ZL)
    m.setInterval(SI)
    _apply(m, kw)
    return m


def _apply(m, kw):
    from grid_ndt_b200 import lib
    for k, v in kw.items():
        setattr(m.params, k, v)
    assert lib().gndt_set_params(m._h, C.byref(m.params)) == 0


def _raw_build(m, sl, cols, n_slopes=None, n_columns=None):
    """gndt_build_edges on caller tables; returns the status."""
    from grid_ndt_b200 import lib
    ds, dc = _dev(sl), _dev(cols)
    _gpu().cuda.synchronize()
    rc = lib().gndt_build_edges(m._h, ds.data_ptr(), len(sl) if n_slopes is None else n_slopes,
                                dc.data_ptr(), len(cols) if n_columns is None else n_columns, None)
    return rc


def caller_edges(m, sl, cols):
    ds, dc = _dev(sl), _dev(cols)
    _gpu().cuda.synchronize()
    return m.edges(ds.data_ptr(), len(sl), dc.data_ptr(), len(cols))


def check_caller(m, sl, cols, p, label=""):
    off, tgt = caller_edges(m, sl, cols)
    return G.assert_graph(off, tgt, sl, cols, p, label)


@pytest.fixture(scope="module")
def handle():
    _gpu()
    m = _handle()
    yield m
    m.close()


# ---- (b) caller tables: search shapes, thresholds, sizes ---------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GALLOP))
def test_gallop(handle, name):
    o, n, t, present, _ = GALLOP[name]
    sl, cols, ci = gallop_tables(o, n, t, present)
    ref = check_caller(handle, sl, cols, _params(), f"{name}: ")
    own = np.nonzero(ref.cand_src == int(cols["slope_begin"][ci]))[0]
    assert np.sum(np.isin(ref.cand_dir[own], (2, 3))) == (2 if present else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(LAYOUTS))
def test_layout(handle, name):
    check_caller(handle, *LAYOUTS[name], _params(), f"{name}: ")


@pytest.mark.gpu
@pytest.mark.parametrize("kw", THRESHOLD_PARAMS)
def test_thresholds(kw):
    p = _set(_params(), kw)
    m = _handle(**kw)
    sl, cols = threshold_tables(p)
    ref = check_caller(m, sl, cols, p, f"thresholds {kw}: ")
    m.close()
    assert ref.n_undecided > 0  # the deliberate ones


@pytest.mark.gpu
@pytest.mark.parametrize("S", CSR_SIZES)
def test_csr_size(handle, S):
    sl, cols = sized_tables(S)
    check_caller(handle, sl, cols, _params(), f"S = {S}: ")


@pytest.mark.gpu
def test_csr_shapes(handle):
    p = _params()
    # zero targets: every cell isolated
    sl, cols = tables([(0, 2 * k) for k in range(50)])
    off, tgt = caller_edges(handle, sl, cols)
    assert len(off) == 51 and not off.any() and len(tgt) == 0
    G.assert_graph(off, tgt, sl, cols, p)
    check_caller(handle, *last_only_tables(), p, "last only: ")
    ref = check_caller(handle, *max_degree_tables(), p, "max degree: ")
    assert ref.csr()[0][-1] > 0
    # C > 0, S = 0: Cells without Slopes
    sl, cols = tables([(0, 0), (0, 1), (1, 0)], 0)
    off, tgt = caller_edges(handle, sl, cols)
    assert list(off) == [0] and len(tgt) == 0
    # C = S = 0 (non-NULL pointers)
    off, tgt = caller_edges(handle, np.zeros(0, SLOPE_DTYPE), np.zeros(0, COLUMN_DTYPE))
    assert list(off) == [0] and len(tgt) == 0


# ---- (c) the build path: real clouds, the GPU's own tables ---------------------------------------

def patches(seed, cells, n=8):
    """n points in each contiguous cell (cx, cy, cz) given, flat inside its cell (z = cz * ZL + 0.05
    with a millimetre of noise): fitted Slopes; neighbours are reachable when their cz differ by at most 1."""
    rng = np.random.default_rng(seed)
    parts = [_cell_points(rng, n, cx, cy, cz, z_frac=(0.49, 0.51)) for cx, cy, cz in cells]
    pts = np.concatenate(parts)
    return pts[rng.permutation(len(pts))]


def _heights(rng, cells):
    return [(x, y, int(rng.choice([0, 0, 0, 1, 3]))) for x, y in cells]


def _clouds():
    rng = np.random.default_rng(11)
    c = {}
    # a long x row next to short ones, with the short rows' columns at the long row's two ends
    c["long_short"] = _heights(rng, [(0, y) for y in range(300)] + [(1, 0), (1, 150), (1, 299)] + [(-1, 299), (2, 1), (2, 298)])
    # an x gap: rows 0..3 and 6..8
    c["x_gap"] = _heights(rng, [(x, y) for x in list(range(0, 4)) + list(range(6, 9)) for y in range(12)])
    # the sign crossing in x and y
    c["sign_crossing"] = _heights(rng, [(x, y) for x in range(-4, 4) for y in range(-4, 4)])
    # first and last rows of very different length: row -5 holds one cell, row 5 forty
    c["first_last"] = _heights(rng, [(-5, 0)] + [(x, y) for x in range(-4, 5) for y in range(0, 10)] + [(5, y) for y in range(-15, 25)])
    return c


CLOUDS = _clouds()


@pytest.mark.parametrize("name", sorted(CLOUDS))
def test_cloud_constructions(name):
    from oracle import oracle as O
    p = _params()
    o = O.oracle_build(patches(1, CLOUDS[name]), p)
    sl, cols = G.oracle_tables(o)
    assert len(cols) == len(CLOUDS[name]) and len(sl) == len(cols)  # one Slope per cell
    cx = G.contig(cols["sx"])
    rows = {int(x): int((cx == x).sum()) for x in np.unique(cx)}
    ref = G.graph_reference(sl, cols, p)
    assert (ref.verdict == G.TRUE).any() and (ref.verdict == G.FALSE).any() and ref.n_undecided == 0
    if name == "long_short":
        assert rows[0] == 300 and rows[1] == 3 and rows[-1] == 1
        # the row-1 column at cy = 299 is found by a gallop from a seed clamped to row 0's end
        g = gallop(cols, column_of(cols, 1, 299), -1)
        assert g["seed"] == 2 and g["target"] == 299 and g["found"]
        g = gallop(cols, column_of(cols, 0, 299), 1)
        assert g["seed"] == 2 and g["target"] == 2 and g["found"]
    elif name == "x_gap":
        assert 4 not in rows and 5 not in rows and rows[3] == rows[6] == 12
    elif name == "sign_crossing":
        assert {-1, 1} <= set(cols["sx"].tolist()) and {-1, 1} <= set(cols["sy"].tolist())
    elif name == "first_last":
        assert min(rows) == -5 and rows[-5] == 1 and max(rows) == 5 and rows[5] == 40


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
@pytest.mark.parametrize("name", sorted(CLOUDS))
def test_cloud(name, demand):
    _gpu()
    from grid_ndt_b200 import TwoDmap
    p = _params(demand=demand)
    m = TwoDmap(GL, ZL)
    m.setInterval(SI)
    m.setCloudFirst((0.0, 0.0, 0.0))
    m.uniformDivision(patches(1, CLOUDS[name]))
    m.create2DMap(demand)
    sl, cols = m.slopes, m.columns
    G.assert_reach_bits(sl, p, cols, f"{name} {demand}: ")
    off, tgt = m.edges()
    G.assert_graph(off, tgt, sl, cols, p, f"{name} {demand}: ")
    m.close()


# ---- (d) streaming ----------------------------------------------------------------------------

def stream_clouds():
    """A: rows 0..2 and 5..7 (a gap at 3, 4), row 1 shorter than rows 0 and 2.  B: fills the gap and
    extends row 1 past the end of row 0."""
    rng = np.random.default_rng(5)
    a = _heights(rng, [(x, y) for x in (0, 2, 5, 6, 7) for y in range(10)] + [(1, y) for y in range(4)])
    b = _heights(rng, [(x, y) for x in (3, 4) for y in range(10)] + [(1, y) for y in range(4, 16)])
    return patches(2, a), patches(3, b)


def test_stream_construction():
    from oracle import oracle as O
    a, b = stream_clouds()
    p = _params()
    oa, ob = O.oracle_build(a, p), O.oracle_build(np.concatenate([a, b]), p)
    rows = lambda o: {int(x): int((G.contig(o.columns["sx"]) == x).sum()) for x in np.unique(G.contig(o.columns["sx"]))}
    ra, rb = rows(oa), rows(ob)
    assert 3 not in ra and 4 not in ra and rb[3] == rb[4] == 10
    assert ra[1] < ra[0] and rb[1] > rb[0] and rb[1] > rb[2]


@pytest.mark.gpu
@pytest.mark.parametrize("demand", ["slope", "true"])
def test_update_and_remove(demand):
    _gpu()
    from grid_ndt_b200 import TwoDmap
    p = _params(demand=demand)
    a, b = stream_clouds()
    m = TwoDmap(GL, ZL)
    m.setInterval(SI)
    m.setCloudFirst((0.0, 0.0, 0.0))
    m.uniformDivision(a)
    m.create2DMap(demand)
    for step, fn in (("update", m.change2DMap), ("remove", m.del2DMap)):
        fn(b)
        sl, cols = m.slopes, m.columns
        G.assert_reach_bits(sl, p, cols, f"{step} {demand}: ")
        off, tgt = m.edges()
        G.assert_graph(off, tgt, sl, cols, p, f"{step} {demand}: ")
    m.close()


# ---- (e) ABI ----------------------------------------------------------------------------------

@pytest.mark.gpu
def test_copy_edges_abi():
    torch = _gpu()
    from grid_ndt_b200 import lib
    L = lib()
    m = _handle()
    ns, nt = C.c_size_t(), C.c_size_t()
    assert L.gndt_copy_edges(m._h, None, 0, None, 0, _abi.GNDT_MEM_HOST, C.byref(ns), C.byref(nt)) == _abi.GNDT_ERR_STATE
    sl, cols = max_degree_tables()
    off, tgt = caller_edges(m, sl, cols)  # a fresh handle that never built a map
    G.assert_graph(off, tgt, sl, cols, _params())
    assert L.gndt_copy_edges(m._h, None, 0, None, 0, _abi.GNDT_MEM_HOST, C.byref(ns), C.byref(nt)) == 0
    assert ns.value == len(sl) and nt.value == len(tgt) > 0
    o2, t2 = np.zeros(len(off), np.uint32), np.zeros(len(tgt), np.uint32)
    host = _abi.GNDT_MEM_HOST
    assert L.gndt_copy_edges(m._h, o2.ctypes.data, len(off) - 1, t2.ctypes.data, len(tgt), host, None, None) == _abi.GNDT_ERR_CAPACITY
    assert L.gndt_copy_edges(m._h, o2.ctypes.data, len(off), t2.ctypes.data, len(tgt) - 1, host, None, None) == _abi.GNDT_ERR_CAPACITY
    assert L.gndt_copy_edges(m._h, o2.ctypes.data, len(off), t2.ctypes.data, len(tgt), host, None, None) == 0
    assert np.array_equal(o2, off) and np.array_equal(t2, tgt)
    do, dt = torch.zeros(len(off), dtype=torch.int32, device="cuda"), torch.zeros(len(tgt), dtype=torch.int32, device="cuda")
    assert L.gndt_copy_edges(m._h, do.data_ptr(), len(off), dt.data_ptr(), len(tgt), _abi.GNDT_MEM_DEVICE, None, None) == 0
    assert np.array_equal(do.cpu().numpy().view(np.uint32), off) and np.array_equal(dt.cpu().numpy().view(np.uint32), tgt)
    ds, dc = _dev(sl), _dev(cols)
    assert L.gndt_build_edges(m._h, ds.data_ptr(), len(sl), None, len(cols), None) == _abi.GNDT_ERR_INVALID_ARG
    assert L.gndt_build_edges(m._h, None, len(sl), dc.data_ptr(), len(cols), None) == _abi.GNDT_ERR_INVALID_ARG
    m.close()


def malformed_cases():
    """name -> (slopes, columns, n_slopes, n_columns) that break one rule of the caller tables."""
    sl, cols = tables([(x, y) for x in range(3) for y in range(4)], 2)
    c = {}
    c["unsorted"] = (sl, cols[[0, 2, 1] + list(range(3, len(cols)))], None, None)
    dup = cols.copy()
    dup[5]["sy"] = dup[4]["sy"]
    c["duplicate_key"] = (sl, dup, None, None)
    past = cols.copy()
    past[-1]["slope_count"] += 1
    c["range_past_n_slopes"] = (sl, past, None, None)
    c["n_slopes_short"] = (sl[:-1], cols, None, None)
    moved = sl.copy()
    moved[3]["sy"] = moved[3]["sy"] + 1
    c["slope_in_another_cell"] = (moved, cols, None, None)
    gap = cols.copy()
    gap[3]["slope_begin"] += 1
    gap[3]["slope_count"] -= 1
    c["range_not_contiguous"] = (sl, gap, None, None)
    zero = cols.copy()
    zero[2]["sy"] = 0
    c["zero_index"] = (sl, zero, None, None)
    c["slopes_without_columns"] = (sl, cols, None, 0)
    return c


MALFORMED = malformed_cases()


@pytest.mark.parametrize("name", sorted(MALFORMED))
def test_malformed_constructions(name):
    sl, cols, ns, nc = MALFORMED[name]
    cols = cols[: nc] if nc is not None else cols
    keys = G.contig(cols["sx"]) * 65536 + G.contig(cols["sy"])
    end = cols["slope_begin"].astype(np.int64) + cols["slope_count"]
    ok = (len(cols) > 0 or len(sl) == 0) and bool(np.all(np.diff(keys) > 0)) and bool(np.all(cols["sx"] != 0) and np.all(cols["sy"] != 0))
    ok = ok and len(cols) > 0 and cols["slope_begin"][0] == 0 and np.array_equal(cols["slope_begin"][1:], end[:-1]) and end[-1] == len(sl)
    if ok:
        ci = np.repeat(np.arange(len(cols)), cols["slope_count"].astype(np.int64))
        ok = np.array_equal(sl["sx"], cols["sx"][ci]) and np.array_equal(sl["sy"], cols["sy"][ci])
    assert not ok, f"{name} breaks no rule"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MALFORMED))
def test_malformed_tables_rejected(handle, name):
    from grid_ndt_b200 import lib
    sl, cols, ns, nc = MALFORMED[name]
    assert _raw_build(handle, sl, cols, ns, nc) == _abi.GNDT_ERR_INVALID_ARG
    msg = lib().gndt_last_error(handle._h).decode()
    assert msg.startswith("gndt_build_edges"), msg
    assert lib().gndt_copy_edges(handle._h, None, 0, None, 0, _abi.GNDT_MEM_HOST, None, None) == _abi.GNDT_ERR_STATE
    sl, cols = tables([(x, y) for x in range(3) for y in range(4)], 2)
    check_caller(handle, sl, cols, _params(), "after a rejected call: ")


@pytest.mark.gpu
def test_stale_graph_after_build_update_remove():
    _gpu()
    from grid_ndt_b200 import TwoDmap, lib
    L = lib()
    p = _params()
    a, b = stream_clouds()
    m = TwoDmap(GL, ZL)
    m.setInterval(SI)
    m.setCloudFirst((0.0, 0.0, 0.0))
    stale = lambda: L.gndt_copy_edges(m._h, None, 0, None, 0, _abi.GNDT_MEM_HOST, None, None) == _abi.GNDT_ERR_STATE
    for step in ("build", "rebuild", "update", "remove"):
        if step in ("build", "rebuild"):
            m.uniformDivision(a if step == "build" else np.concatenate([b, a]))
            m.create2DMap("slope")
        else:
            (m.change2DMap if step == "update" else m.del2DMap)(b)
        if step != "build":
            assert stale(), f"gndt_copy_edges hands out the graph of the map before the {step}"
        off, tgt = m.edges()
        G.assert_graph(off, tgt, m.slopes, m.columns, p, f"{step}: ")
        assert not stale()
    m.close()
