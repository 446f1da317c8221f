"""The x-strip exchange on ONE GPU: N handles on the current device play N ranks.

gndt_xchg_connect treats a peer of the same process on the same device as a plain pointer, so the
whole protocol (publish, halo send / wait, boundary edges, push with the index rewrite, done / wait,
both transports) runs in the single-GPU suite.  Every rank builds and exchanges on its own
non-blocking stream; all builds are enqueued before the first exchange and all exchanges before the
first host read, because the exchange kernels of a rank spin until every other rank has joined.

Clouds are built on purpose around the cuts, in contiguous index space (cell c >= 0 is signed index
c + 1, c < 0 is c) about an explicit origin (0, 0, 0); every point is binned.  The tests without the
gpu marker check on the oracle alone (tile_lo / tile_hi) that each construction puts its edge where
it claims; the gpu tests hold the gathered map to the same bar as the untiled build:
  * every rank's gathered tables are byte-identical, and identical across the two transports;
  * they equal the untiled GPU build (multi_gpu_worker.same_table) and pass parity.compare_gathered;
  * where strips meet, the forward / back bits of the boundary rows are set and equal the untiled build's.
"""
import ctypes as C
import json

import numpy as np
import pytest

from grid_ndt_b200 import _abi, synthetic
from grid_ndt_b200._abi import COLUMN_DTYPE, SLOPE_DTYPE, VOXEL_DTYPE, default_params
from grid_ndt_b200.tiles import halo_peers

GL, ZL, SI = 0.2, 0.1, 0.08
REC = VOXEL_DTYPE.itemsize
LO, HI = -32768, 32768  # outer cuts: the whole index range
FB = _abi.F_REACH_F | _abi.F_REACH_B
ALL = _abi.X_VOXELS | _abi.X_SLOPES | _abi.X_COLUMNS
TRANSPORTS = ("sm", "ce")
MAXI = _abi.GNDT_MAX_INDEX  # signed 32767 = contiguous 32766


# ---- construction helpers ----------------------------------------------------------------

def _params(**kw):
    return default_params(GL, ZL, SI, origin=(0.0, 0.0, 0.0), origin_is_first_point=0, **kw)


def _contig(s):
    return np.where(s > 0, s - 1, s)


def ground(seed, xs, ys, n=8, z=0.05, cz=0):
    """n points in each cell (cx, cy) of xs x ys, on a flat surface at height cz * ZL + z with 1 mm of
    noise: every cell is one fitted Slope whose neighbours are reachable (angle ~0, |dz| ~0), far
    from every threshold."""
    rng = np.random.default_rng(seed)
    cells = np.array([(x, y) for x in xs for y in ys], np.float64).reshape(-1, 2)
    cells = np.repeat(cells, n, axis=0)
    px = (cells[:, 0] + rng.uniform(0.1, 0.9, len(cells))) * GL
    py = (cells[:, 1] + rng.uniform(0.1, 0.9, len(cells))) * GL
    pz = cz * ZL + z + rng.uniform(-0.001, 0.001, len(cells))
    return np.stack([px, py, pz, np.ones(len(cells))], 1).astype(np.float32)


def cat(*parts):
    return np.concatenate([p for p in parts if len(p)]).astype(np.float32)


def _oracle(cloud, mode="faithful32"):
    from oracle import oracle as O
    return O.oracle_build(cloud, _params(), mode)


def _strip_of(cx, cuts):
    return np.searchsorted(np.asarray(cuts[1:-1]), cx, side="right")


def strip_rows(o, cuts):
    """{strip: sorted x rows it holds} of an oracle map."""
    cx = _contig(o.voxels["sx"])
    r = _strip_of(cx, cuts)
    return {k: sorted(set(cx[r == k].tolist())) for k in range(len(cuts) - 1)}


def strip_voxels(o, cuts):
    return np.bincount(_strip_of(_contig(o.voxels["sx"]), cuts), minlength=len(cuts) - 1)


def row_sizes(o, cuts):
    """[(first row, last row) voxel counts] per strip (0, 0 when empty)."""
    cx = _contig(o.voxels["sx"])
    out = []
    for k, rows in strip_rows(o, cuts).items():
        out.append((int((cx == rows[0]).sum()), int((cx == rows[-1]).sum())) if rows else (0, 0))
    return out


def cross_pairs(o, cuts):
    """Slope pairs (a, b) in x-adjacent cells of different strips, with their angle (deg) and |dz|."""
    v = o.voxels
    sl = np.nonzero(v["flags"] & _abi.F_SLOPE)[0]
    cx, cy, st = _contig(v["sx"]), _contig(v["sy"]), _strip_of(_contig(v["sx"]), cuts)
    by = {}
    for i in sl:
        by.setdefault((int(cx[i]), int(cy[i])), []).append(i)
    out = []
    for (x, y), lst in by.items():
        for j in by.get((x + 1, y), []):
            for i in lst:
                if st[i] != st[j]:
                    n1, n2 = v["normal"][i].astype(np.float64), v["normal"][j].astype(np.float64)
                    d = abs(float(np.dot(n1, n2))) / (np.linalg.norm(n1) * np.linalg.norm(n2))
                    out.append((i, j, float(np.degrees(np.arccos(min(d, 1.0)))), abs(float(v["mean"][i][2]) - float(v["mean"][j][2]))))
    return out


def assert_cross(o, cuts, expect):
    """Cross-strip reachable pairs exist (expect=True) or not, and every pair is clear of the
    angle / height thresholds by far more than the 1e-5 band."""
    p = _params()
    pairs = cross_pairs(o, cuts)
    for i, j, ang, dz in pairs:
        assert abs(ang - p.angle_max_deg) > 1.0 and abs(dz - p.reach_height) > 0.01, (i, j, ang, dz)
    reach = [q for q in pairs if q[2] < p.angle_max_deg and q[3] <= p.reach_height]
    assert bool(reach) == expect, f"{len(reach)} reachable cross-strip pairs, expected {'some' if expect else 'none'}"
    return reach


# ---- the constructions: name -> (cloud, cuts, cross-strip pairs expected) ------------------

def _constructions():
    c = {}
    g = ground(1, range(-4, 4), range(0, 10))
    c["sign_change"] = (g, [LO, 0, HI], True)                 # contiguous 0 = signed +1 | -1 meet at the cut
    c["sign_change_3"] = (g, [LO, -1, 1, HI], True)           # strip 1 = rows -1, 0: the quadrant crossing inside it
    c["index_edges"] = (cat(ground(2, range(-MAXI, -MAXI + 5), range(0, 6)),
                            ground(3, range(MAXI - 6, MAXI), range(0, 6))),
                        [LO, -MAXI + 2, MAXI - 3, HI], True)  # rows -32767 and 32766 hold points; cuts beside them
    c["one_row"] = (g, [LO, 0, 1, HI], True)                  # strip 1 is row 0 alone: cx_min == cx_max
    c["empty_between"] = (g, [LO, 0, 0, HI], True)            # equal cuts: strips 0 and 2 meet across strip 1
    c["no_points_gap"] = (cat(ground(4, range(-4, 0), range(0, 8)), ground(5, range(2, 5), range(0, 8))),
                          [LO, 0, 2, HI], False)              # strip 1 = rows 0, 1: a range without points
    c["empty_ends"] = (g, [LO, LO, 0, HI, HI], True)          # empty first and last strip
    c["one_of_four"] = (g, [LO, -40, -40, 40, HI], False)     # strip 2 holds everything
    c["gap_at_cut"] = (cat(ground(6, range(-5, -1), range(0, 8)), ground(7, range(0, 4), range(0, 8))),
                       [LO, 0, HI], False)                    # last row of strip 0 is cut - 2, first of strip 1 is cut
    # the halo search: in row -1 (the halo of strip 1), column cy = 2 holds a low Slope under the
    # reachable one; strip 1's columns cy = -3 and cy = 14 lie below / above every halo record and
    # cy = 5 has no neighbour column in the halo
    c["halo_search"] = (cat(ground(8, range(-3, 0), [0, 1, 2, 3, 4, 6, 7, 8]), ground(9, [-1], [2], cz=-12),
                            ground(10, range(0, 3), [-3, 0, 1, 2, 3, 4, 5, 6, 14])),
                        [LO, 0, HI], True)
    c["halo_single"] = (cat(ground(11, range(-3, -1), range(0, 6)), ground(12, [-1], [3]), ground(13, range(0, 3), range(0, 6))),
                        [LO, 0, HI], True)                    # the halo row of strip 1 holds one record
    return c


CONSTRUCTIONS = _constructions()


# ---- B: the constructions on the oracle alone ----------------------------------------------

@pytest.mark.parametrize("name", sorted(CONSTRUCTIONS))
def test_construction_puts_its_edge_where_it_claims(name):
    cloud, cuts, cross = CONSTRUCTIONS[name]
    o = _oracle(cloud)
    rows = strip_rows(o, cuts)
    assert o.counts["n_dropped"] == 0
    assert_cross(o, cuts, cross)
    if name in ("sign_change", "sign_change_3"):
        assert 0 in sum(rows.values(), []) and -1 in sum(rows.values(), [])
        assert set(np.unique(o.voxels["sx"][np.isin(_contig(o.voxels["sx"]), [-1, 0])])) == {-1, 1}
        if name == "sign_change_3":
            assert rows[1] == [-1, 0]
    elif name == "index_edges":
        assert rows[0] == list(range(-MAXI, -MAXI + 2)) and rows[2] == list(range(MAXI - 3, MAXI))
        assert o.voxels["sx"].min() == -MAXI and o.voxels["sx"].max() == MAXI  # points on the last valid index
    elif name == "one_row":
        assert rows[1] == [0]
    elif name == "empty_between":
        assert rows[1] == [] and rows[0][-1] == -1 and rows[2][0] == 0
    elif name == "no_points_gap":
        assert rows[1] == [] and rows[0][-1] == -1 and rows[2][0] == 2
    elif name == "empty_ends":
        assert rows[0] == [] and rows[3] == [] and rows[1] and rows[2]
    elif name == "one_of_four":
        assert [bool(rows[k]) for k in range(4)] == [False, False, True, False]
    elif name == "gap_at_cut":
        assert rows[0][-1] == -2 and rows[1][0] == 0
    elif name == "halo_search":
        v = o.voxels
        col = (_contig(v["sx"]) == -1) & (_contig(v["sy"]) == 2)
        assert col.sum() == 2 and np.all(v["flags"][col] & _abi.F_SLOPE)       # a lower Slope under the reachable one
        halo_cy = set(_contig(v["sy"])[_contig(v["sx"]) == -1].tolist())
        assert min(halo_cy) > -3 and max(halo_cy) < 14 and 5 not in halo_cy  # below, above, absent
        first = (_contig(v["sx"]) == 0)
        assert {-3, 5, 14} <= set(_contig(v["sy"])[first].tolist())
        assert not np.any(v["flags"][first & np.isin(_contig(v["sy"]), [-3, 5, 14])] & _abi.F_REACH_B)
    elif name == "halo_single":
        assert row_sizes(o, cuts)[0][1] == 1


def halo_cap_cloud(k):
    """Strip 0's last row (cx = -1) holds exactly k voxels; every other boundary row fewer."""
    return cat(ground(20, range(-3, -1), range(0, 4)), ground(21, [-1], range(0, k)), ground(22, range(0, 3), range(0, 4))), [LO, 0, HI]


@pytest.mark.parametrize("k", [6, 7])
def test_halo_capacity_construction(k):
    cloud, cuts = halo_cap_cloud(k)
    sizes = row_sizes(_oracle(cloud), cuts)
    assert sizes[0][1] == k and max(sizes[0][0], sizes[1][0], sizes[1][1]) < k


def test_gathered_capacity_and_streaming_constructions():
    g = CONSTRUCTIONS["sign_change"][0]
    assert _oracle(g).counts["n_voxels"] == 80
    # streaming: strip-local scans
    for name, (base, scan, cuts, check) in STREAMS.items():
        oa, ob = _oracle(base), _oracle(cat(base, scan))
        check(oa, ob, cuts)


def _only_strip(r):
    def check(oa, ob, cuts):
        cx = _contig(ob.voxels["sx"])
        assert set(_strip_of(cx[~np.isin(ob.voxels["sx"] * 100000 + ob.voxels["sy"], oa.voxels["sx"] * 100000 + oa.voxels["sy"])], cuts)) <= {r}
    return check


def _opens_edges(oa, ob, cuts):
    ra, rb = strip_rows(oa, cuts), strip_rows(ob, cuts)
    assert ra[1] == [-1, 0, 1] and rb[1] == [-2, -1, 0, 1, 2]          # rows at both edges of strip 1 opened
    assert not cross_pairs(oa, cuts) and cross_pairs(ob, cuts)


def wall(seed, cx, cy, n=200):
    """n points on the vertical plane through the middle of cell (cx, cy), inside its z cell 0."""
    rng = np.random.default_rng(seed)
    px = (cx + 0.5 + rng.uniform(-0.005, 0.005, n)) * GL
    py = (cy + rng.uniform(0.1, 0.9, n)) * GL
    pz = rng.uniform(0.01, 0.09, n) * (ZL / 0.1)
    return np.stack([px, py, pz, np.ones(n)], 1).astype(np.float32)


def _kills_f_bit(oa, ob, cuts):
    """A wall fused into strip 1's boundary Slope at (0, 3) turns its normal horizontal: strip 0's
    (-1, 3) loses its F bit."""
    def f(o):
        v = o.voxels
        i = np.nonzero((_contig(v["sx"]) == -1) & (_contig(v["sy"]) == 3))[0]
        return int(v["flags"][i[0]]) & _abi.F_REACH_F
    assert f(oa) and not f(ob)


STREAMS = {
    "one_strip": (ground(30, range(-4, 4), range(0, 8)), cat(ground(31, range(1, 3), range(0, 10)), ground(32, [3], [12])), [LO, 0, HI], _only_strip(1)),
    "new_edge_rows": (cat(ground(33, range(-5, -2), range(0, 6)), ground(34, range(-1, 2), range(0, 6)), ground(35, range(3, 6), range(0, 6))),
                      cat(ground(36, [-2], range(0, 6)), ground(37, [2], range(0, 6))), [LO, -2, 3, HI], _opens_edges),
    "tilt_boundary": (ground(38, range(-3, 3), range(0, 6)), wall(39, 0, 3), [LO, 0, HI], _kills_f_bit),
}


# ---- the one-GPU world ---------------------------------------------------------------------

def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked test on a box without CUDA (no fallback exists)")
    return torch


def _tile(cuts, r):
    lo, hi = int(cuts[r]), int(cuts[r + 1])
    return (lo, hi) if lo < hi else _abi.TILE_EMPTY


class World:
    """N TwoDmap handles on the current device, one x strip and one non-blocking stream each, their
    exchange buffers connected (peers in the same process on the same device: plain pointers)."""

    def __init__(self, cuts, transport="sm", what=ALL, cap_records=1 << 20, cap_halo=16384, max_voxels=None):
        torch = _gpu()
        from grid_ndt_b200 import TwoDmap, lib
        from grid_ndt_b200.builder import _check
        self.L, self.check, self.torch = lib(), _check, torch
        self.n, self.transport, self.what = len(cuts) - 1, transport, what
        self.maps = []
        for r in range(self.n):
            m = TwoDmap(GL, ZL)
            m.setInterval(SI)
            m.setCloudFirst((0.0, 0.0, 0.0))
            if max_voxels and max_voxels.get(r):
                m.params.max_voxels = max_voxels[r]
            self.maps.append(m)
        self.set_cuts(cuts)
        infos = (_abi.XchgInfo * self.n)()
        for r, m in enumerate(self.maps):
            _check(m._h, self.L.gndt_xchg_create(m._h, r, self.n, int(cap_records), int(cap_halo), what, C.byref(infos[r])))
        for m in self.maps:
            _check(m._h, self.L.gndt_xchg_connect(m._h, infos, self.n))
        self.streams = [torch.cuda.Stream() for _ in range(self.n)]

    def set_cuts(self, cuts):
        self.cuts = list(cuts)
        for r, m in enumerate(self.maps):
            m.setTile(*_tile(cuts, r))

    def build(self, cloud):
        """Every rank gets the whole cloud and keeps its strip (enqueued, nothing read back)."""
        dev = self.torch.from_numpy(np.ascontiguousarray(cloud)).cuda()
        self.torch.cuda.synchronize()
        self._keep = dev
        for m, s in zip(self.maps, self.streams):
            m.uniformDivision(dev)
            m.create2DMap("slope", stream=s.cuda_stream)

    def fuse(self, scan, remove=False):
        dev = self.torch.from_numpy(np.ascontiguousarray(scan)).cuda()
        self.torch.cuda.synchronize()
        self._keep_scan = dev
        fn = self.L.gndt_remove if remove else self.L.gndt_update
        for m, s in zip(self.maps, self.streams):
            self.check(m._h, fn(m._h, dev.data_ptr(), dev.shape[0], dev.shape[1] * 4, _abi.GNDT_MEM_DEVICE, s.cuda_stream))

    def exchange(self):
        """Enqueue the exchange of every rank; returns the status of each rank's send (ce) or run (sm)."""
        rcs = []
        if self.transport == "sm":
            for m, s in zip(self.maps, self.streams):
                rcs.append(self.L.gndt_xchg_run(m._h, s.cuda_stream))
        else:
            for m, s in zip(self.maps, self.streams):
                self.check(m._h, self.L.gndt_xchg_stage(m._h, s.cuda_stream))
            for m, s in zip(self.maps, self.streams):
                rcs.append(self.L.gndt_xchg_send(m._h, s.cuda_stream))
        return rcs

    def views(self):
        """[(status, message, XchgView)] of every rank."""
        out = []
        for m in self.maps:
            v = _abi.XchgView()
            rc = self.L.gndt_xchg_view_get(m._h, C.byref(v))
            out.append((rc, (self.L.gndt_last_error(m._h) or b"").decode() if rc else "", v))
        return out

    def tables(self, v):
        """Host copies of one rank's gathered tables (None where not gathered)."""
        from grid_ndt_b200.tiles import _as_tensor
        out = {}
        for name, ptr, n, dt in (("voxels", v.voxels, v.n_voxels, VOXEL_DTYPE), ("slopes", v.slopes, v.n_slopes, SLOPE_DTYPE),
                                 ("columns", v.columns, v.n_columns, COLUMN_DTYPE)):
            if not ptr:
                out[name] = None
            elif n == 0:
                out[name] = np.zeros(0, dt)
            else:
                out[name] = _as_tensor(ptr, int(n) * dt.itemsize, self.torch.device("cuda")).cpu().numpy().view(dt).copy()
        out["strip_voxels"] = list(v.strip_voxels[: self.n])
        return out

    def run(self):
        """Exchange and read every rank's gathered tables; asserts success and agreement between ranks."""
        rcs = self.exchange()
        views = self.views()
        assert all(rc == 0 for rc in rcs), rcs
        assert all(rc == 0 for rc, _, _ in views), [(rc, msg) for rc, msg, _ in views]
        t = [self.tables(v) for _, _, v in views]
        for r in range(1, self.n):
            for k in ("voxels", "slopes", "columns"):
                assert (t[r][k] is None) == (t[0][k] is None)
                if t[0][k] is not None:
                    assert t[r][k].tobytes() == t[0][k].tobytes(), f"rank {r} holds different {k} than rank 0"
        return t[0]

    def close(self):
        self.torch.cuda.synchronize()
        for m in self.maps:
            m.close()


def untiled(cloud):
    """The untiled GPU build of the same cloud: (voxels, slopes, columns)."""
    _gpu()
    from grid_ndt_b200 import TwoDmap
    m = TwoDmap(GL, ZL)
    m.setInterval(SI)
    m.setCloudFirst((0.0, 0.0, 0.0))
    m.uniformDivision(np.ascontiguousarray(cloud))
    m.create2DMap("slope")
    out = (m.voxels.copy(), m.slopes.copy(), m.columns.copy())
    m.close()
    return out


def hold_to_the_bar(tag, t, cloud, cuts, cross, ref=None, oracle=True):
    """Gathered tables vs the untiled GPU build and the oracle; boundary F/B bits where strips meet."""
    from tests import parity
    from tests.multi_gpu_worker import same_table
    ref_v, ref_s, ref_c = ref if ref is not None else untiled(cloud)
    for k, r in (("voxels", ref_v), ("slopes", ref_s), ("columns", ref_c)):
        if t[k] is not None:
            same_table(f"{tag}: gathered {k} vs untiled build", t[k], r)
    if t["voxels"] is not None:
        v = t["voxels"]
        rows = np.isin(_contig(v["sx"]), np.concatenate([np.asarray(cuts[1:-1]), np.asarray(cuts[1:-1]) - 1]))
        bits = v["flags"][rows] & FB
        assert np.array_equal(bits, ref_v["flags"][rows] & FB), f"{tag}: boundary F/B bits differ from the untiled build"
        if cross:
            assert np.any(bits), f"{tag}: no F/B bit on a strip boundary row"
        # strips concatenated in rank order, each holding exactly the records of its cut range
        sv = np.asarray(t["strip_voxels"], np.int64)
        assert np.array_equal(_strip_of(_contig(v["sx"]), cuts), np.repeat(np.arange(len(sv)), sv)), f"{tag}: strips out of place"
        assert all(sv[r] == 0 for r in range(len(sv)) if cuts[r] >= cuts[r + 1]), f"{tag}: an empty strip sent records"
    if oracle and t["voxels"] is not None and t["columns"] is not None and t["slopes"] is not None:
        o32, o64 = _oracle(cloud), _oracle(cloud, "truth64")
        rep = parity.compare_gathered(t["voxels"], t["columns"], t["slopes"], o32, o64, _params())
        assert rep["ok"], f"{tag}: " + json.dumps(rep, default=str)


def caller_abi(cloud, cuts, cap_halo=16384, fuse=None):
    """The same strips through gndt_halo_pack / gndt_halo_edges / gndt_apply_strip_offsets (legacy
    stream, no peer exchange): returns the gathered tables {voxels, slopes, columns}, or (status,
    message) of the first failing strip.  The voxels come from gndt_apply_strip_offsets, the slopes
    and columns from the host statement of the index rewrite (parity.assemble_strips, and
    slope.voxel += voxels before), which the voxels must match byte for byte."""
    torch = _gpu()
    from grid_ndt_b200 import GndtError, TwoDmap, lib
    from grid_ndt_b200.builder import _check
    from tests import parity
    L, n = lib(), len(cuts) - 1
    maps = []
    for r in range(n):
        m = TwoDmap(GL, ZL)
        m.setInterval(SI)
        m.setCloudFirst((0.0, 0.0, 0.0))
        m.setTile(*_tile(cuts, r))
        m.uniformDivision(np.ascontiguousarray(cloud))
        m.create2DMap("slope")
        if fuse is not None:
            m.change2DMap(np.ascontiguousarray(fuse))
        maps.append(m)
    halo = torch.zeros(n, 2, (cap_halo + 1) * REC, dtype=torch.uint8, device="cuda")
    for r, m in enumerate(maps):
        _check(m._h, L.gndt_halo_pack(m._h, halo[r, 0].data_ptr(), halo[r, 1].data_ptr(), cap_halo, 0))
    for r, m in enumerate(maps):
        prev, nxt = halo_peers(np.asarray(cuts), r, n)
        _check(m._h, L.gndt_halo_edges(m._h, halo[prev, 1].data_ptr() if prev is not None else None,
                                       halo[nxt, 0].data_ptr() if nxt is not None else None, 0))
    try:
        strips = [(m.voxels.copy(), m.columns.copy()) for m in maps]
        slopes = [m.slopes.copy() for m in maps]
    except GndtError as e:
        for m in maps:
            m.close()
        return e.status, str(e)
    sizes = [len(v) for v, _ in strips]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    col_off = np.concatenate([[0], np.cumsum([len(c) for _, c in strips])])[:-1].astype(np.uint32)
    slope_off = np.concatenate([[0], np.cumsum([int((v["slope"] != 0xFFFFFFFF).sum()) for v, _ in strips])])[:-1].astype(np.uint32)
    table = torch.empty(max(int(offsets[-1]), 1) * REC, dtype=torch.uint8, device="cuda")
    for r, m in enumerate(maps):
        if sizes[r]:
            _check(m._h, L.gndt_copy_voxels(m._h, table.data_ptr() + int(offsets[r]) * REC, sizes[r], _abi.GNDT_MEM_DEVICE, None))
    _check(maps[0]._h, L.gndt_apply_strip_offsets(maps[0]._h, table.data_ptr(), (C.c_uint64 * (n + 1))(*[int(x) for x in offsets]),
                                                  (C.c_uint32 * n)(*[int(x) for x in col_off]), (C.c_uint32 * n)(*[int(x) for x in slope_off]), n, 0))
    torch.cuda.synchronize()
    got = table.cpu().numpy().view(VOXEL_DTYPE)[: int(offsets[-1])].copy()
    # the host statement of the index rewrite, with the slope table's voxel index made global too
    want_v, want_c = parity.assemble_strips(strips)
    assert got.tobytes() == want_v.tobytes(), "gndt_apply_strip_offsets differs from parity.assemble_strips"
    for sl, off in zip(slopes, offsets[:-1]):
        sl["voxel"] += np.uint32(off)
    for m in maps:
        m.close()
    return {"voxels": got, "slopes": np.concatenate(slopes), "columns": want_c}


def _exchange_all(cloud, cuts, cross, tag, what=ALL, **kw):
    """Both transports, full bar, byte-identical across transports and to the caller-ABI path."""
    got = {}
    ref = untiled(cloud)
    for tr in TRANSPORTS:
        w = World(cuts, tr, what, **kw)
        w.build(cloud)
        got[tr] = w.run()
        w.close()
        hold_to_the_bar(f"{tag} {tr}", got[tr], cloud, cuts, cross, ref)
        for k, bit in (("voxels", _abi.X_VOXELS), ("slopes", _abi.X_SLOPES), ("columns", _abi.X_COLUMNS)):
            assert (got[tr][k] is None) == (not what & bit), f"{k}: view pointer must be NULL exactly when not gathered"
    for k in ("voxels", "slopes", "columns"):
        if got["sm"][k] is not None:
            assert got["sm"][k].tobytes() == got["ce"][k].tobytes(), f"{tag}: transports differ in {k}"
    return got["sm"], ref


# ---- C: GPU cases --------------------------------------------------------------------------

PLAN_CLOUD = None


def _plan_cloud():
    global PLAN_CLOUD
    if PLAN_CLOUD is None:
        c = synthetic.cfg2(250_000, scale=0.2)
        PLAN_CLOUD = c[1:]  # the explicit origin (0, 0, 0) is used; point 0 is an ordinary point here
    return PLAN_CLOUD


def _plan_cuts(cloud, world):
    from grid_ndt_b200 import TwoDmap
    m = TwoDmap(GL, ZL)
    m.setCloudFirst((0.0, 0.0, 0.0))
    cuts = m.plan_tiles(cloud, world)
    m.close()
    return cuts


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 4])
def test_planned_worlds_all_transports_and_selections(world):
    _gpu()
    cloud = _plan_cloud()
    cuts = _plan_cuts(cloud, world)
    assert cuts[0] == LO and cuts[-1] == HI and np.all(np.diff(cuts) > 0)
    full, _ = _exchange_all(cloud, cuts, True, f"plan{world}")
    for what in (_abi.X_SLOPES | _abi.X_COLUMNS, _abi.X_VOXELS):
        sub, _ = _exchange_all(cloud, cuts, True, f"plan{world} what={what}", what=what)
        for k in ("voxels", "slopes", "columns"):
            if sub[k] is not None:
                assert sub[k].tobytes() == full[k].tobytes(), k
    abi = caller_abi(cloud, cuts)
    for k in ("voxels", "slopes", "columns"):
        assert abi[k].tobytes() == full[k].tobytes(), f"caller-ABI strips differ from the peer exchange in {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CONSTRUCTIONS))
def test_constructed_boundaries(name):
    cloud, cuts, cross = CONSTRUCTIONS[name]
    full, _ = _exchange_all(cloud, cuts, cross, name)
    abi = caller_abi(cloud, cuts)
    for k in ("voxels", "slopes", "columns"):
        assert abi[k].tobytes() == full[k].tobytes(), f"caller-ABI strips differ from the peer exchange in {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("over", [False, True])
def test_halo_capacity_edge(over):
    cloud, cuts = halo_cap_cloud(7 if over else 6)
    cap = 6
    res = caller_abi(cloud, cuts, cap_halo=cap)
    if not over:
        _exchange_all(cloud, cuts, True, "halo exactly cap_halo", cap_halo=cap)
        assert isinstance(res, dict), res
        return
    assert res[0] == _abi.GNDT_ERR_CAPACITY and "cap_halo" in res[1], res
    for tr in TRANSPORTS:
        w = World(cuts, tr, cap_halo=cap)
        w.build(cloud)
        assert w.exchange() == [0, 0]
        (rc0, msg0, _), (rc1, msg1, _) = w.views()
        assert rc0 == 0, (tr, msg0)  # strip 0 receives strip 1's first row, which fits
        assert rc1 == _abi.GNDT_ERR_CAPACITY and "cap_halo" in msg1, (tr, rc1, msg1)
        w.close()


@pytest.mark.gpu
def test_gathered_capacity_edge_then_smaller_rebuild():
    cloud, cuts, _ = CONSTRUCTIONS["sign_change_3"]
    total = _oracle(cloud).counts["n_voxels"]
    small = ground(40, range(-2, 2), range(0, 5))
    for tr in TRANSPORTS:
        w = World(cuts, tr, cap_records=total)
        w.build(cloud)
        hold_to_the_bar(f"cap_records exact {tr}", w.run(), cloud, cuts, True)
        w.close()
        w = World(cuts, tr, cap_records=total - 1)
        w.build(cloud)
        rcs = w.exchange()
        views = w.views()
        assert all(rc == _abi.GNDT_ERR_CAPACITY for rc, _, _ in views), (tr, [(rc, m) for rc, m, _ in views])
        if tr == "ce":
            assert all(rc == _abi.GNDT_ERR_CAPACITY for rc in rcs), rcs
        w.build(small)
        hold_to_the_bar(f"smaller rebuild {tr}", w.run(), small, cuts, True)
        w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("transport", TRANSPORTS)
def test_epochs_on_the_same_handles(transport):
    g = CONSTRUCTIONS["sign_change"][0]
    steps = [
        (g, [LO, -2, 1, HI]),
        (ground(41, range(-6, 2), range(0, 4)), [LO, -2, 1, HI]),
        (g, [LO, 0, 0, HI]),                                # strip 1 goes empty
        (ground(42, range(-1, 6), range(-2, 9)), [LO, -1, 2, HI]),  # ... and comes back
        (g, [LO, -3, -2, HI]),
        (ground(43, range(-3, 3), range(0, 3)), [LO, -2, 1, HI]),
    ]
    w = World(steps[0][1], transport)
    for i, (cloud, cuts) in enumerate(steps):
        w.set_cuts(cuts)
        w.build(cloud)
        got = w.run()
        fresh = World(cuts, transport)
        fresh.build(cloud)
        want = fresh.run()
        fresh.close()
        for k in ("voxels", "slopes", "columns"):
            assert got[k].tobytes() == want[k].tobytes(), f"exchange {i}: {k} differ from a fresh world's"
        assert got["strip_voxels"] == want["strip_voxels"]
    w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(STREAMS) + ["remove_first_row"])
def test_streaming_on_strips(name):
    if name == "remove_first_row":
        base = cat(ground(44, range(-3, 0), range(0, 6)), ground(46, range(1, 4), range(0, 6)))
        row0 = ground(45, [0], range(0, 6), n=6)  # strip 1's whole first row, the last points of the build
        cloud, scan, cuts, final = cat(base, row0), row0, [LO, 0, HI], base
    else:
        cloud, scan, cuts, _ = STREAMS[name]
        final = cat(cloud, scan)
    for tr in TRANSPORTS:
        w = World(cuts, tr)
        w.build(cloud)
        w.run()
        w.fuse(scan, remove=name == "remove_first_row")
        got = w.run()
        w.close()
        hold_to_the_bar(f"{name} {tr}", got, final, cuts, name != "remove_first_row")


@pytest.mark.gpu
def test_update_then_halo_overflow_reports_the_exchange():
    """A successful update followed by a halo overflow: the update stands, the overflow is reported,
    and no query returns the old counts over the new records."""
    cuts = [LO, 0, HI]
    a = cat(ground(50, range(-3, 0), range(0, 5)), ground(51, range(0, 3), range(0, 5)))
    b = cat(ground(52, [-1], range(5, 9)), ground(53, [2], range(6, 9)))  # strip 0's last row: 5 -> 9 > cap; strip 1 grows
    cap = 6

    def check_queries(m):
        from grid_ndt_b200 import GndtError
        with pytest.raises(GndtError) as e:
            m.counts()
        assert e.value.status == _abi.GNDT_ERR_CAPACITY and "max_voxels" not in str(e.value) and "cap_halo" in str(e.value), str(e.value)
        try:
            c, v = m.counts(), m.voxels
        except GndtError as e2:
            assert e2.status == _abi.GNDT_ERR_CAPACITY, str(e2)
            return
        want = _oracle(cat(a, b)).voxels
        want = want[_strip_of(_contig(want["sx"]), cuts) == 1]
        assert c["n_voxels"] == len(v) == len(want), "counts and records of different maps"

    # caller ABI
    _gpu()
    from grid_ndt_b200 import TwoDmap, lib
    from grid_ndt_b200.builder import _check
    import torch
    L = lib()
    maps = []
    for r in range(2):
        m = TwoDmap(GL, ZL)
        m.setInterval(SI)
        m.setCloudFirst((0.0, 0.0, 0.0))
        m.setTile(*_tile(cuts, r))
        m.uniformDivision(a)
        m.create2DMap("slope")
        m.change2DMap(b)
        maps.append(m)
    halo = torch.zeros(2, 2, (cap + 1) * REC, dtype=torch.uint8, device="cuda")
    for r, m in enumerate(maps):
        _check(m._h, L.gndt_halo_pack(m._h, halo[r, 0].data_ptr(), halo[r, 1].data_ptr(), cap, 0))
    _check(maps[0]._h, L.gndt_halo_edges(maps[0]._h, None, halo[1, 0].data_ptr(), 0))
    _check(maps[1]._h, L.gndt_halo_edges(maps[1]._h, halo[0, 1].data_ptr(), None, 0))
    assert maps[0].counts()["n_voxels"] > 0
    check_queries(maps[1])
    for m in maps:
        m.close()
    # peer exchange
    for tr in TRANSPORTS:
        w = World(cuts, tr, cap_halo=cap)
        w.build(a)
        w.run()
        w.fuse(b)
        w.exchange()
        views = w.views()
        assert views[0][0] == 0, views[0][1]
        assert views[1][0] == _abi.GNDT_ERR_CAPACITY and "max_voxels" not in views[1][1] and "cap_halo" in views[1][1], (tr, views[1][:2])
        check_queries(w.maps[1])
        w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("transport", TRANSPORTS)
def test_update_failing_on_one_strip_is_named_by_the_others(transport):
    cuts = [LO, -2, 2, HI]
    a = ground(54, range(-5, 5), range(0, 5))
    n1 = int(strip_voxels(_oracle(a), cuts)[1])
    b = ground(55, [0], range(5, 10))  # 5 new voxels in strip 1 only
    w = World(cuts, transport, max_voxels={1: n1 + 2})
    w.build(a)
    before = w.run()
    w.fuse(b)
    w.exchange()
    views = w.views()
    assert views[1][0] == _abi.GNDT_ERR_CAPACITY and "max_voxels" in views[1][1], views[1][:2]
    for r in (0, 2):
        assert views[r][0] == _abi.GNDT_ERR_STATE and "strip 1" in views[r][1], (r, views[r][:2])
    after = w.run()  # a second exchange with no update: the map from before the update
    for k in ("voxels", "slopes", "columns"):
        assert after[k].tobytes() == before[k].tobytes(), k
    w.close()


@pytest.mark.gpu
def test_multi_front_door_on_one_gpu():
    torch = _gpu()
    from grid_ndt_b200.multi import MultiTwoDmap
    from oracle import oracle as O
    from tests import parity
    dev = torch.cuda.current_device()
    cloud = synthetic.cfg2(400_000, scale=0.25)
    p = default_params(GL, ZL, SI)
    mm = MultiTwoDmap(GL, ZL, SI, [dev] * 3, capacity=1_000_000)
    o32, o64 = O.oracle_build(cloud, p, "faithful32"), O.oracle_build(cloud, p, "truth64")
    for src in (cloud, torch.from_numpy(cloud).cuda(dev)):
        mm.chatterCallback(src)
        t0, t2 = mm.tables(0), mm.tables(2)
        for k in ("voxels", "slopes", "columns"):
            assert t0[k].tobytes() == t2[k].tobytes(), k
        rep = parity.compare_gathered(t0["voxels"], t0["columns"], t0["slopes"], o32, o64, p)
        assert rep["ok"], rep["fail"]
        assert min(t0["strip_voxels"]) > 0
    mm.chatterCallback(cloud[:250_000])
    mm.change2DMap(cloud[250_000:])
    t = mm.tables(1)
    rep = parity.compare_gathered(t["voxels"], t["columns"], t["slopes"], o32, o64, p)
    assert rep["ok"], rep["fail"]
    mm.close()


@pytest.mark.gpu
def test_graph_from_gathered_tables():
    from tests import graph_reference as G
    _gpu()
    from grid_ndt_b200 import TwoDmap
    cloud = _plan_cloud()
    cuts = _plan_cuts(cloud, 3)
    w = World(cuts, "sm")
    w.build(cloud)
    t = w.run()
    v = w.views()[1][2]
    off, tgt = w.maps[1].edges(v.slopes, v.n_slopes, v.columns, v.n_columns)
    w.close()
    m = TwoDmap(GL, ZL)
    m.setInterval(SI)
    m.setCloudFirst((0.0, 0.0, 0.0))
    m.uniformDivision(cloud)
    m.create2DMap("slope")
    uoff, utgt = m.edges()
    m.close()
    assert np.array_equal(off, uoff) and np.array_equal(tgt, utgt), "graph of the gathered tables differs from the untiled graph"
    G.assert_graph(off, tgt, t["slopes"], t["columns"], _params(), "gathered: ")
    sl = t["slopes"]
    cx = _contig(sl["sx"]).astype(np.int64)
    src = np.repeat(np.arange(len(sl)), np.diff(off.astype(np.int64)))
    across = _strip_of(cx[src], cuts) != _strip_of(cx[tgt], cuts)
    assert across.any(), "no edge crosses a strip boundary"
