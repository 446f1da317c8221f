"""gndt_register_d2d on the GPU against the numpy restatement in tests/ndt_d2d_oracle.py.  The oracle
is fed the map's gndt_copy_voxels and the records of a public gndt_build of the scan on another
handle with the parameters the header names, which also pins the scan Gaussians the library builds
internally.  Evaluation parity per level, scan Gaussians on cell edges, convergence against the
oracle, NO_MATCH, map state, no side effects, determinism and the argument checks."""
import ctypes as C
import functools

import numpy as np
import pytest

import grid_ndt_b200 as g
from grid_ndt_b200 import _abi
from tests import ndt_d2d_oracle as D
from tests import ndt_levels_cases as K
from tests import ndt_oracle as N
from tests.test_gpu_ndt import TOL, _state, cloud, make_map, scan_of, within_bounds
from tests.test_gpu_ndt_levels import raw as raw_levels
from tests.test_gpu_ndt_levels import raw_register
from tests.test_ndt_d2d import BASIN, BASIN_GUESSES, PYRAMID

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def scan_voxels(m, scan):
    """Records of the scan as the header says it is built: a public gndt_build on another handle with
    the map's parameters, origin = the map's origin, every point binned."""
    s = g.TwoDmap(m.getGridLen(), m.getZLen())
    s._p = D.scan_params(m.params, m.origin())
    s.uniformDivision(np.ascontiguousarray(scan[:, :3], np.float32))
    s.create2DMap("slope" if m.params.demand == _abi.GNDT_DEMAND_SLOPE else "true")
    v = s.voxels.copy()
    s.close()
    return v


def d2d_eval(m, scan, T, factors=(), stride=16, device=False, **ndt):
    """max_iterations = 0 on every level and the map level at pose T: counts exact and S / g / H within
    TOL of the oracle's bound on each; returns the GPU result."""
    sc = np.ascontiguousarray(np.pad(scan[:, :3], ((0, 0), (0, stride // 4 - 3))), dtype=np.float32)
    arg = torch.from_numpy(sc).cuda() if device else sc
    r = m.register(arg, T, levels=[dict(factor=k, max_iterations=0) for k in factors], method="d2d", max_iterations=0, **ndt)
    mv, sv = m.voxels, scan_voxels(m, scan)
    for k, got in list(zip(factors, r["levels"])) + [(1, r)]:
        e = D.Problem(mv, sv, m.origin(), m.getGridLen(), m.getZLen(), scan, k, int(m.params.normalize_cov), **ndt).evaluate(T, with_abs=True)
        assert (got["n_points"], got["n_matched"], got["n_pairs"]) == (e["n_points"], e["n_matched"], e["n_pairs"]), k
        aS, ag, aH = e["abs"]
        assert abs(got["score"] - e["score"]) <= TOL * aS + 1e-300, k
        assert np.all(np.abs(got["gradient"] - e["gradient"]) <= TOL * ag + 1e-300), k
        assert np.all(np.abs(got["hessian"] - e["hessian"]) <= TOL * aH + 1e-300), k
        assert np.array_equal(got["pose"], T) and got["termination"] in (_abi.NDT_MAX_ITER, _abi.NDT_NO_MATCH)
        np.testing.assert_allclose(got["center"], e["center"], rtol=0, atol=1e-9)
    return r


def raw(m, scan, T, levels, p=None):
    """(out bytes, [level bytes]) of one gndt_register_d2d call on the raw ABI."""
    sc = np.ascontiguousarray(scan[:, :3], np.float32)
    Tc = (C.c_double * 16)(*np.asarray(T, np.float64).ravel())
    p = p or _abi.default_ndt_params()
    lv = (_abi.NdtLevel * max(len(levels), 1))(*[_abi.default_ndt_level(k) for k in levels])
    per = (_abi.Registration * max(len(levels), 1))()
    out = _abi.Registration()
    rc = g.lib().gndt_register_d2d(m._h, sc.ctypes.data, len(sc), 12, 0, Tc, C.byref(p), lv, len(levels), C.byref(out), per, None)
    assert rc == 0, g.lib().gndt_last_error(m._h)
    return bytes(out), [bytes(per[i]) for i in range(len(levels))]


def dense_scan(radius=5.0, centre=N.PIER_CENTRE):
    return D.dense_disc(cloud()[1:, :3], centre, radius)


@pytest.mark.parametrize("res,demand,ncov", [(0.2, "slope", 0), (0.1, "true", 0), (0.2, "true", 1)])
def test_d2d_evaluation_parity(res, demand, ncov):
    m = make_map(cloud(), res, demand, ncov)
    scan = dense_scan()
    for T in (np.eye(4), N.pose((0.5, -0.3, 0.4), (0.05, -0.03, 0.02))):
        for stride, dev in ((12, False), (16, True), (32, False)):
            d2d_eval(m, scan, T, (8, 4, 2), stride, dev)
    bad = scan.copy()
    bad[::7, 0] = np.nan
    bad[1::7, 2] = np.inf
    bad[2::7, 1] = 1e4  # finite, index out of range: dropped by the scan build, counted in the centre
    d2d_eval(m, bad, np.eye(4), (4,))


# ---- scan Gaussians whose means land on cell edges and one ulp either side -------------------
# Each Gaussian is 4 points that share the edge coordinate and spread, without symmetry, over the
# other two axes inside one cell (a double eigenvalue costs eig3_sym half its digits); each sits in
# its own cell of those axes, so no two merge.
PAT = np.array([(1, 2), (-3, 1), (2, -2), (0, -1)], np.float64) / 16.0


def edge_gaussian_scan(k, axis, coarse):
    L = (K.GRID, K.GRID, K.ZLEN)
    cells = [X * k for X in (-3, -1, 0, 1, 2)] if coarse else [X * k + j for X in (-3, -1, 0, 1, 2) for j in range(1, k)]
    vals = [v for c in cells for v in K.edge_values(c * L[axis])]
    o1, o2 = [a for a in range(3) if a != axis]
    pts = []
    for j, v in enumerate(vals):
        c1, c2 = j % (2 * k) - k, j // (2 * k) - k
        assert c2 < k
        for d1, d2 in PAT:
            p = np.zeros(3, np.float32)
            p[axis] = v
            p[o1], p[o2] = (c1 + 0.5 + d1) * L[o1], (c2 + 0.5 + d2) * L[o2]
            pts.append(p)
    return np.array(pts, np.float32)


@pytest.mark.parametrize("k", [2, 4, 8])
def test_d2d_cell_edges(k):
    m = g.TwoDmap(K.GRID, K.ZLEN)
    m.chatterCallback(K.edge_map(k))
    for axis in range(3):
        for coarse in (True, False):
            scan = edge_gaussian_scan(k, axis, coarse)
            sv = scan_voxels(m, scan)
            assert np.all(sv["count"] == 4) and len(sv) == len(scan) // 4  # one Gaussian per cluster
            # means on the edge values (the build flushes the subnormal +-1 ulp around 0 to 0)
            v = scan[::4, axis]
            assert np.array_equal(np.sort(sv["mean"][:, axis]), np.sort(np.where(np.abs(v) < np.finfo(np.float32).tiny, 0, v)))
            r = d2d_eval(m, scan, np.eye(4), (k,), min_voxel_points=3)
            assert r["n_pairs"] > 0


# ---- convergence on the dense-disc instance -------------------------------------------------

@functools.lru_cache(maxsize=1)
def _instance():
    mp, scan = D.d2d_instance(cloud())
    m = make_map(mp)
    P = D.Pyramid(m.voxels, scan_voxels(m, scan), m.origin(), m.getGridLen(), m.getZLen(), scan, PYRAMID)
    return m, scan, P


def test_d2d_convergence_matches_oracle():
    """Map level from 1 cm / 0.1 deg: CONVERGED at the true pose, as the oracle's run.  Pyramid from
    0.3 m / 3 deg (tests/test_ndt_d2d.py): every level as the oracle's run; the map level ends as the
    oracle's does, off the true pose."""
    m, scan, P = _instance()
    centre = N.transform(N.T_TRUE, P.map.pbar[None])[0]

    def same(a, b):
        assert a["termination"] == b["termination"], (a["termination"], b["termination"])
        dt, deg = N.pose_error(a["pose"], b["pose"], P.map.pbar)
        assert dt <= 1e-5 and np.radians(deg) <= 1e-5, (dt, deg)

    for G in N.guesses(N.T_TRUE, centre, **N.GUESS_OFFSETS)[:3]:
        r = m.register(scan, G, method="d2d")
        ok, err = within_bounds(r["pose"], N.T_TRUE, P.map.pbar)
        assert ok and r["termination"] == _abi.NDT_CONVERGED, (err, r["termination"])
        same(r, P.map.register(G))
    gs = N.guesses(N.T_TRUE, centre, n=6, seed=11, **BASIN)
    for i in BASIN_GUESSES:
        r = m.register(scan, gs[i], levels=PYRAMID, method="d2d")
        o, olv = P.register(gs[i], PYRAMID)
        for a, b in zip(r["levels"], olv):
            same(a, b)
        assert r["termination"] == o["termination"] and not within_bounds(r["pose"], N.T_TRUE, P.map.pbar)[0]


def test_d2d_reproducible_at_out_pose_and_out_is_the_last_level_continued():
    m, scan, P = _instance()
    centre = N.transform(N.T_TRUE, P.map.pbar[None])[0]
    G = N.guesses(N.T_TRUE, centre, n=6, seed=11, **BASIN)[BASIN_GUESSES[0]]
    out, per = raw(m, scan, G, list(PYRAMID))
    r = m.register(scan, G, levels=PYRAMID, method="d2d")
    assert out == raw(m, scan, r["levels"][-1]["pose"], [])[0]
    e = m.register(scan, r["pose"], method="d2d", max_iterations=0)
    for k in ("score", "gradient", "hessian", "center", "n_points", "n_matched", "n_pairs"):
        assert np.array_equal(e[k], r[k]), k
    assert raw(m, scan, G, list(PYRAMID)) == (out, per)  # determinism


def test_d2d_no_match():
    m = make_map(cloud()[:300_000])
    T = N.pose((0.1, 0, 0), (0.01, 0, 0))
    # every scan cell below min_points: one point per map cell
    o = m.origin()
    ij = np.stack(np.meshgrid(np.arange(-20, 20), np.arange(-20, 20), indexing="ij"), -1).reshape(-1, 2)
    sparse = np.zeros((len(ij), 3), np.float32)
    sparse[:, :2] = (o[:2] + (ij + 0.5) * 0.2).astype(np.float32)
    sparse[:, 2] = np.float32(o[2] + 0.05)
    for levels in (None, [4]):
        r = m.register(sparse, T, levels=levels, method="d2d")
        assert r["termination"] == _abi.NDT_NO_MATCH and np.array_equal(r["pose"], T) and r["n_points"] == 0 and r["n_pairs"] == 0
        assert r["score"] == 0 and not r["gradient"].any() and not r["hessian"].any()
    far = N.pose((0, 0, 0), (1000.0, 0, 0))
    r = m.register(dense_scan(3.0), far, levels=[8], method="d2d")
    assert r["levels"][0]["termination"] == _abi.NDT_NO_MATCH and np.array_equal(r["levels"][0]["pose"], far)
    assert r["termination"] == _abi.NDT_NO_MATCH and np.array_equal(r["pose"], far) and r["n_points"] > 0


def test_d2d_map_state_and_p2d_unchanged():
    pts = cloud()[:600_000]
    s1, s2 = scan_of(cloud()[600_000:], 30_000, 5), scan_of(cloud()[600_000:], 30_000, 6)
    q = dense_scan(4.0, (16.0, 10.0))
    T = N.pose((0.4, -0.3, 0.8), (0.05, -0.04, 0.01))

    def updated():
        m = make_map(pts)
        m.change2DMap(s1)
        return m

    a, b = updated(), updated()
    p2d, p2d_lv = raw_register(a, q, T), raw_levels(a, q, T, [8, 4, 2])
    before = _state(a)
    first = raw(a, q, T, [8, 4, 2])
    assert _state(a) == before  # tables, counts, changed columns, key layout, launch count
    assert raw_register(a, q, T) == p2d and raw_levels(a, q, T, [8, 4, 2]) == p2d_lv  # P2D: the same bytes
    assert raw(a, q, T, [8, 4, 2]) == first == raw(b, q, T, [8, 4, 2])  # D2D, P2D, D2D
    d2d_eval(a, q, T, (8, 2))
    a.del2DMap(s1); b.del2DMap(s1)
    assert raw(a, q, T, [8, 3]) == raw(b, q, T, [8, 3])
    d2d_eval(a, q, T, (8, 3))
    c = make_map(pts, max_voxels=make_map(pts).counts()["n_voxels"])
    raw(c, q, T, [8, 4, 2])
    far = s2.copy()
    far[:, 0] += 500.0
    c.change2DMap(far)
    with pytest.raises(g.GndtError) as e:
        c.register(q, T, levels=[4], method="d2d")
    assert e.value.status == _abi.GNDT_ERR_CAPACITY
    assert raw(c, q, T, [8, 4, 2]) == raw(make_map(pts), q, T, [8, 4, 2])


def test_d2d_stage_times_unchanged():
    m = make_map(cloud()[:300_000])
    m.stage_timing(True)
    m.chatterCallback(cloud()[:300_000])
    ms = m.stage_ms()
    m.register(dense_scan(3.0), None, levels=[4], method="d2d")
    assert m.stage_ms() == ms


def test_d2d_invalid_arguments():
    m = make_map(cloud()[:300_000])
    scan = np.ascontiguousarray(dense_scan(3.0), np.float32)
    L = g.lib()
    T = (C.c_double * 16)(*np.eye(4).ravel())
    p, out = _abi.default_ndt_params(), _abi.Registration()

    def call(levels, n=None, h=m._h, T=T, p=p, out=out, stride=12):
        arr = (_abi.NdtLevel * max(len(levels), 1))(*levels) if levels is not None else None
        return L.gndt_register_d2d(h, scan.ctypes.data, len(scan) * 12 // stride, stride, 0, T, C.byref(p) if p else None, arr,
                                   len(levels or []) if n is None else n, C.byref(out) if out else None, None, None)

    lv = _abi.default_ndt_level
    assert call([lv(8), lv(2)]) == 0
    assert call(None, 0) == 0
    bad = [(None, 1), ([lv(8)] * 9, None), ([lv(4)], -1), ([lv(1)], None), ([lv(33)], None), ([lv(4), lv(4)], None),
           ([lv(2), lv(4)], None), ([lv(4, max_iterations=-1)], None), ([lv(4, translation_epsilon=-1.0)], None),
           ([lv(4, rotation_epsilon=float("inf"))], None), ([lv(4, translation_epsilon=float("nan"))], None)]
    for levels, n in bad:
        assert call(levels, n) == _abi.GNDT_ERR_INVALID_ARG, (levels and [(l.factor, l.max_iterations) for l in levels], n)
    assert call([], T=None) == _abi.GNDT_ERR_INVALID_ARG
    assert call([], p=None) == _abi.GNDT_ERR_INVALID_ARG
    assert call([], out=None) == _abi.GNDT_ERR_INVALID_ARG
    assert call([], stride=13) == _abi.GNDT_ERR_INVALID_ARG
    for kw in (dict(min_voxel_points=2), dict(outlier_ratio=1.0), dict(max_iterations=-1), dict(rotation_epsilon=float("nan")), dict(reserved=1)):
        with pytest.raises(g.GndtError) as e:
            m.register(scan, None, method="d2d", **kw)
        assert e.value.status == _abi.GNDT_ERR_INVALID_ARG, kw
    for Tb in (np.full((4, 4), np.nan), np.diag([1, 1, 1, 2.0]), np.diag([1.0, 1.0, 1.01, 1.0])):
        with pytest.raises(g.GndtError) as e:
            m.register(scan, Tb, method="d2d")
        assert e.value.status == _abi.GNDT_ERR_INVALID_ARG
    fresh = g.TwoDmap(0.2, 0.1)
    assert call([lv(4)], h=fresh._h) == _abi.GNDT_ERR_STATE
    with pytest.raises(g.GndtError):
        m.register(scan, None, method="icp")
