"""gndt_register on the GPU against the numpy restatement in tests/ndt_oracle.py: evaluation
parity, edge cases, convergence, consistency, determinism, no side effects on the map, a
degenerate scan and a register -> transform -> update loop."""
import ctypes as C
import functools

import numpy as np
import pytest

import grid_ndt_b200 as g
from grid_ndt_b200 import _abi, synthetic
from tests import ndt_oracle as N

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

TOL = 1e-9  # of the oracle's sum of |per-pair contribution|, per entry


@functools.lru_cache(maxsize=1)
def cloud():
    return synthetic.cfg2(900_000, scale=0.3)


def make_map(pts, res=0.2, demand="slope", normalize_cov=0, max_voxels=0):
    m = g.TwoDmap(res, 0.1)
    m.params.normalize_cov = normalize_cov
    m.params.max_voxels = max_voxels
    m.chatterCallback(pts, demand)
    return m


def problem(m, scan, **ndt):
    return N.Problem(m.voxels, m.origin(), m.getGridLen(), m.getZLen(), scan, int(m.params.normalize_cov), **ndt)


def check_eval(m, scan, T, stride=16, device=False, **ndt):
    """max_iterations = 0 at pose T: counts exact, S / g / H within TOL of the oracle's bound."""
    sc = np.ascontiguousarray(np.pad(scan[:, :3], ((0, 0), (0, stride // 4 - 3))), dtype=np.float32)
    arg = torch.from_numpy(sc).cuda() if device else sc
    r = m.register(arg, T, max_iterations=0, **ndt)
    e = problem(m, scan, **ndt).evaluate(T, with_abs=True)
    assert (r["n_points"], r["n_matched"], r["n_pairs"]) == (e["n_points"], e["n_matched"], e["n_pairs"])
    aS, ag, aH = e["abs"]
    assert abs(r["score"] - e["score"]) <= TOL * aS + 1e-300
    assert np.all(np.abs(r["gradient"] - e["gradient"]) <= TOL * ag + 1e-300), (r["gradient"], e["gradient"])
    assert np.all(np.abs(r["hessian"] - e["hessian"]) <= TOL * aH + 1e-300)
    np.testing.assert_allclose(r["center"], e["center"], rtol=0, atol=1e-9)
    return r


def scan_of(pts, n, seed=0):
    idx = np.random.default_rng(seed).choice(len(pts), n, replace=False)
    return pts[np.sort(idx)].copy()


def edge_scan(m, n=20_000, seed=3):
    """Scan points that land, under the pose EDGE_T (a translation by binary fractions, so R p + t
    is exact), on a cell edge of x or y or one float32 ulp to either side."""
    rng = np.random.default_rng(seed)
    base = scan_of(cloud()[1:800_000], n, seed)[:, :3].astype(np.float32)
    o = m.origin()
    L = np.float32(m.getGridLen())
    for ax in (0, 1):
        k = np.round((base[:, ax] - o[ax]) / L).astype(np.float32)
        e = (o[ax] + k * L).astype(np.float32)
        step = rng.integers(-1, 2, n)
        e = np.where(step < 0, np.nextafter(e, np.float32(-np.inf)), np.where(step > 0, np.nextafter(e, np.float32(np.inf)), e))
        base[:, ax] = e.astype(np.float32)
    return (base - EDGE_T[:3, 3].astype(np.float32)).astype(np.float32)


EDGE_T = np.eye(4)
EDGE_T[:3, 3] = (0.25, -0.5, 0.125)


@pytest.mark.parametrize("res,demand,ncov", [(0.2, "slope", 0), (0.1, "true", 0), (0.2, "true", 1)])
def test_evaluation_parity(res, demand, ncov):
    m = make_map(cloud(), res, demand, ncov)
    scan = scan_of(cloud(), 60_000, 1)
    poses = [np.eye(4), N.pose((0.5, -0.3, 0.4), (0.05, -0.03, 0.02))]
    for T in poses:
        for stride, dev in ((12, False), (16, True), (32, False), (32, True)):
            check_eval(m, scan, T, stride, dev)
    es = edge_scan(m)
    x = N.transform(EDGE_T, es)
    assert np.array_equal(x.astype(np.float32), x)  # the pose moves the points exactly
    check_eval(m, es, EDGE_T, 16, False)
    check_eval(m, es, EDGE_T, 12, True)


def test_edge_cases():
    m = make_map(cloud()[:600_000])
    scan = scan_of(cloud(), 20_000, 2)
    bad = scan.copy()
    bad[::7, 0] = np.nan
    bad[1::7, 2] = np.inf
    bad[2::7, 1] = 1e30  # finite, index out of range
    r = check_eval(m, bad, np.eye(4))
    assert r["n_points"] == len(bad) - len(bad[::7]) - len(bad[1::7])
    far = N.pose((0, 0, 0), (1000.0, 0, 0))
    r = m.register(scan, far)
    assert r["termination"] == _abi.NDT_NO_MATCH and np.array_equal(r["pose"], far)
    assert r["score"] == 0 and not r["gradient"].any() and not r["hessian"].any() and r["n_pairs"] == 0
    r = m.register(scan, None, min_voxel_points=10**9)
    assert r["termination"] == _abi.NDT_NO_MATCH and r["n_pairs"] == 0
    # INVALID_ARG
    for T in (np.full((4, 4), np.nan), np.diag([1, 1, 1, 2.0]), np.diag([1.0, 1.0, 1.01, 1.0])):
        with pytest.raises(g.GndtError) as e:
            m.register(scan, T)
        assert e.value.status == _abi.GNDT_ERR_INVALID_ARG
    for kw in (dict(min_voxel_points=2), dict(outlier_ratio=1.0), dict(outlier_ratio=0.0), dict(max_iterations=-1),
               dict(translation_epsilon=-1.0), dict(rotation_epsilon=float("nan")), dict(reserved=1)):
        with pytest.raises(g.GndtError) as e:
            m.register(scan, None, **kw)
        assert e.value.status == _abi.GNDT_ERR_INVALID_ARG, kw
    L = g.lib()
    T = (C.c_double * 16)(*np.eye(4).ravel())
    p, out = _abi.default_ndt_params(), _abi.Registration()
    assert L.gndt_register(m._h, scan.ctypes.data, len(scan), 16, 0, None, C.byref(p), C.byref(out), None) == _abi.GNDT_ERR_INVALID_ARG
    assert L.gndt_register(m._h, scan.ctypes.data, len(scan), 16, 0, T, None, C.byref(out), None) == _abi.GNDT_ERR_INVALID_ARG
    assert L.gndt_register(m._h, scan.ctypes.data, len(scan), 16, 0, T, C.byref(p), None, None) == _abi.GNDT_ERR_INVALID_ARG
    assert L.gndt_register(m._h, scan.ctypes.data, len(scan), 13, 0, T, C.byref(p), C.byref(out), None) == _abi.GNDT_ERR_INVALID_ARG
    fresh = g.TwoDmap(0.2, 0.1)
    with pytest.raises(g.GndtError) as e:
        fresh.register(scan)
    assert e.value.status == _abi.GNDT_ERR_STATE


def test_failed_update_then_register():
    pts = cloud()[:300_000]
    ref = make_map(pts)
    V = ref.counts()["n_voxels"]
    m = make_map(pts, max_voxels=V)
    scan = scan_of(cloud(), 20_000, 4)
    far = scan.copy()
    far[:, 0] += 500.0  # opens new voxels: capacity exceeded at the verdict
    m.change2DMap(far)
    with pytest.raises(g.GndtError) as e:
        m.register(scan)
    assert e.value.status == _abi.GNDT_ERR_CAPACITY
    a, b = m.register(scan), ref.register(scan)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _convergence():
    mp, scan = N.convergence_instance(cloud())
    m = make_map(mp)
    pr = problem(m, scan)
    centre = N.transform(N.T_TRUE, pr.pbar[None])[0]
    return m, scan, pr, N.guesses(N.T_TRUE, centre, **N.GUESS_OFFSETS)


def within_bounds(T, T_true, at):
    dt, deg = N.pose_error(T, T_true, at)
    return dt <= 5e-3 and deg <= 0.02, (dt, deg)


def test_convergence_matches_oracle():
    m, scan, pr, guesses = _convergence()
    for G in guesses:
        r = m.register(scan, G)
        ok, err = within_bounds(r["pose"], N.T_TRUE, pr.pbar)
        assert ok and r["termination"] == _abi.NDT_CONVERGED, (err, r["termination"], r["iterations"])
        o = pr.register(G)
        assert o["termination"] == r["termination"]
        dt, deg = N.pose_error(r["pose"], o["pose"], pr.pbar)
        assert dt <= 1e-5 and np.radians(deg) <= 1e-5, (dt, deg)


def test_monotone_and_consistent():
    m, scan, pr, guesses = _convergence()
    for G in guesses[:3]:
        r0 = m.register(scan, G, max_iterations=0)
        r = m.register(scan, G)
        assert r["score"] >= r0["score"]
        e = m.register(scan, r["pose"], max_iterations=0)
        for k in ("score", "gradient", "hessian", "center", "n_points", "n_matched", "n_pairs"):
            assert np.array_equal(e[k], r[k]), k


def test_determinism():
    m, scan, pr, guesses = _convergence()
    L = g.lib()
    T = (C.c_double * 16)(*guesses[0].ravel())
    p = _abi.default_ndt_params()
    outs = []
    for _ in range(2):
        out = _abi.Registration()
        assert L.gndt_register(m._h, scan.ctypes.data, len(scan), 16, 0, T, C.byref(p), C.byref(out), None) == 0
        outs.append(bytes(out))
    assert outs[0] == outs[1]


def _state(m):
    m._tables.clear()
    return (m.voxels.tobytes(), m.slopes.tobytes(), m.columns.tobytes(), m.counts(), m.key_layout(), m.launch_count(),
            m.changed_columns.tobytes())


def test_no_side_effects():
    pts = cloud()[:600_000]
    a, b = make_map(pts), make_map(pts)
    s1, s2 = scan_of(cloud()[600_000:], 30_000, 5), scan_of(cloud()[600_000:], 30_000, 6)
    a.change2DMap(s1)
    b.change2DMap(s1)
    before = _state(a)
    a.register(s2, N.pose((0.2, 0, 0.1), (0.02, 0, 0)))
    assert _state(a) == before
    a.change2DMap(s2)
    b.change2DMap(s2)
    a._tables.clear(); b._tables.clear()
    assert a.voxels.tobytes() == b.voxels.tobytes() and a.columns.tobytes() == b.columns.tobytes()
    # the Gaussians follow the map through update and remove
    q = scan_of(cloud(), 30_000, 7)
    check_eval(a, q, np.eye(4))
    a.del2DMap(s1)
    check_eval(a, q, np.eye(4))


def test_degenerate_parallel_planes():
    m = make_map(cloud())
    planes = next(synthetic.scans(cfg2_scale=0.3))[:40_000]
    scan = N.apply(np.linalg.inv(N.T_TRUE), planes)
    pbar = N.finite_points(scan).astype(np.float64).mean(0)
    centre = N.transform(N.T_TRUE, pbar[None])[0]
    for G in N.guesses(N.T_TRUE, centre, n=3, seed=13, **N.GUESS_OFFSETS):
        r = m.register(scan, G)
        assert all(np.all(np.isfinite(r[k])) for k in ("pose", "score", "gradient", "hessian"))
        dz = (r["pose"][:3, :3] @ pbar + r["pose"][:3, 3] - centre)[2]
        up = r["pose"][:3, :3] @ np.linalg.inv(N.T_TRUE)[:3, :3] @ np.array([0.0, 0.0, 1.0])
        tilt = np.degrees(np.arccos(np.clip(up[2], -1, 1)))
        assert abs(dz) <= 5e-3 and tilt <= 0.02, (dz, tilt, r["termination"])


def test_register_transform_update_loop():
    mp, scans = N.workflow_instance(cloud())
    m = make_map(mp)
    for scan, T, guess in scans:
        pbar = scan[:, :3].astype(np.float64).mean(0)
        r = m.register(scan, guess)
        ok, err = within_bounds(r["pose"], T, pbar)
        assert ok, (err, r["termination"], r["iterations"])
        m.change2DMap(N.apply(r["pose"], scan))
