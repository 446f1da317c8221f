"""gndt_register_levels on the GPU against the numpy restatement in tests/ndt_levels_oracle.py:
evaluation parity per level on real maps and on hand-made boundaries (tests/ndt_levels_cases.py),
the wide-basin convergence the CPU test proves, consistency with gndt_register, the level cache
across map states, no side effects, determinism and the argument checks."""
import ctypes as C
import functools

import numpy as np
import pytest

import grid_ndt_b200 as g
from grid_ndt_b200 import _abi
from tests import ndt_levels_cases as K
from tests import ndt_levels_oracle as NL
from tests import ndt_oracle as N
from tests.test_gpu_ndt import TOL, _state, cloud, make_map, scan_of, within_bounds
from tests.test_ndt_levels import BASIN, BASIN_GUESSES, PYRAMID

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def level_eval(m, scan, T, factors, stride=16, device=False, **ndt):
    """max_iterations = 0 on every level at pose T: each level's counts exact and S / g / H within
    TOL of the oracle's bound; returns the GPU result."""
    sc = np.ascontiguousarray(np.pad(scan[:, :3], ((0, 0), (0, stride // 4 - 3))), dtype=np.float32)
    arg = torch.from_numpy(sc).cuda() if device else sc
    r = m.register(arg, T, levels=[dict(factor=k, max_iterations=0) for k in factors], max_iterations=0, **ndt)
    vox = m.voxels
    for k, lv in zip(factors, r["levels"]):
        e = NL.Level(vox, m.origin(), m.getGridLen(), m.getZLen(), scan, k, int(m.params.normalize_cov), **ndt).evaluate(T, with_abs=True)
        assert (lv["n_points"], lv["n_matched"], lv["n_pairs"]) == (e["n_points"], e["n_matched"], e["n_pairs"]), k
        aS, ag, aH = e["abs"]
        assert abs(lv["score"] - e["score"]) <= TOL * aS + 1e-300, k
        assert np.all(np.abs(lv["gradient"] - e["gradient"]) <= TOL * ag + 1e-300), k
        assert np.all(np.abs(lv["hessian"] - e["hessian"]) <= TOL * aH + 1e-300), k
        assert np.array_equal(lv["pose"], T) and lv["termination"] in (_abi.NDT_MAX_ITER, _abi.NDT_NO_MATCH)
    return r


def raw(m, scan, T, levels, np_=None, with_levels=True):
    """(out bytes, [level bytes]) of one gndt_register_levels call on the raw ABI."""
    L = g.lib()
    sc = np.ascontiguousarray(scan[:, :3], np.float32)
    Tc = (C.c_double * 16)(*np.asarray(T, np.float64).ravel())
    p = np_ or _abi.default_ndt_params()
    lv = (_abi.NdtLevel * max(len(levels), 1))(*[_abi.default_ndt_level(k) for k in levels])
    per = (_abi.Registration * max(len(levels), 1))()
    out = _abi.Registration()
    rc = L.gndt_register_levels(m._h, sc.ctypes.data, len(sc), 12, 0, Tc, C.byref(p), lv, len(levels), C.byref(out),
                                per if with_levels else None, None)
    assert rc == 0, g.lib().gndt_last_error(m._h)
    return bytes(out), [bytes(per[i]) for i in range(len(levels))]


def raw_register(m, scan, T):
    L = g.lib()
    sc = np.ascontiguousarray(scan[:, :3], np.float32)
    Tc = (C.c_double * 16)(*np.asarray(T, np.float64).ravel())
    p, out = _abi.default_ndt_params(), _abi.Registration()
    assert L.gndt_register(m._h, sc.ctypes.data, len(sc), 12, 0, Tc, C.byref(p), C.byref(out), None) == 0
    return bytes(out)


def test_no_levels_is_gndt_register():
    m = make_map(cloud()[:600_000])
    scan = scan_of(cloud(), 20_000, 2)
    T = N.pose((0.3, -0.2, 0.5), (0.03, -0.02, 0.01))
    assert raw(m, scan, T, [])[0] == raw_register(m, scan, T)


@pytest.mark.parametrize("res,demand,ncov", [(0.2, "slope", 0), (0.1, "true", 0), (0.2, "true", 1)])
def test_level_evaluation_parity(res, demand, ncov):
    m = make_map(cloud(), res, demand, ncov)
    scan = scan_of(cloud(), 60_000, 1)
    for T in (np.eye(4), N.pose((0.5, -0.3, 0.4), (0.05, -0.03, 0.02))):
        for stride, dev in ((12, False), (16, True), (32, False)):
            level_eval(m, scan, T, (8, 4, 3, 2), stride, dev)


def built(cloud_):
    m = g.TwoDmap(K.GRID, K.ZLEN)
    m.chatterCallback(cloud_)
    return m


@pytest.mark.parametrize("k", [2, 3, 4, 8])
def test_cell_edges(k):
    m = built(K.edge_map(k))
    for axis in range(3):
        for coarse in (True, False):
            level_eval(m, K.edge_scan(k, axis, coarse), np.eye(4), (k,), min_voxel_points=3)


@pytest.mark.parametrize("k", [2, 3, 8])
def test_hand_made_slabs(k):
    for name, (c, scan) in K.slab_maps(k).items():
        m = built(c)
        r = level_eval(m, scan, np.eye(4), (k,), min_voxel_points=3)
        assert r["levels"][0]["n_pairs"] > 0, name


@pytest.mark.parametrize("k", [2, 3, 8])
def test_mixed_fitted_and_unfitted(k):
    c = K.mixed_map(k)
    level_eval(built(c), c[1:], np.eye(4), (k,), min_voxel_points=3)


def test_extreme_indices():
    c = K.extreme_map()
    m = built(c)
    for k in (2, 3, 32):
        level_eval(m, c[1:], np.eye(4), (k,), min_voxel_points=3)


@pytest.mark.parametrize("k", [2, 5])
def test_merged_count_at_min_voxel_points(k):
    c = K.count_map(k)
    m = built(c)
    r = level_eval(m, c[1:], np.eye(4), (k,), min_voxel_points=8)
    assert r["levels"][0]["n_pairs"] == 8
    r = level_eval(m, c[1:], np.eye(4), (k,), min_voxel_points=9)
    assert r["levels"][0]["n_pairs"] == 0


def test_no_usable_gaussian_hands_the_pose_on():
    c = K.count_map(4)
    m = built(c)
    T = N.pose((0.1, 0, 0), (0.01, 0, 0))
    r = m.register(c[1:], T, levels=[4], min_voxel_points=9)
    assert r["levels"][0]["termination"] == _abi.NDT_NO_MATCH and np.array_equal(r["levels"][0]["pose"], T)
    assert r["termination"] == _abi.NDT_NO_MATCH and np.array_equal(r["pose"], T)


@functools.lru_cache(maxsize=1)
def _convergence():
    mp, scan = N.convergence_instance(cloud())
    m = make_map(mp)
    P = NL.Pyramid(m.voxels, m.origin(), m.getGridLen(), m.getZLen(), scan, PYRAMID)
    centre = N.transform(N.T_TRUE, P.map.pbar[None])[0]
    gs = N.guesses(N.T_TRUE, centre, n=6, seed=11, **BASIN)
    return m, scan, P, [gs[i] for i in BASIN_GUESSES]


def test_pyramid_converges_and_matches_oracle():
    m, scan, P, guesses = _convergence()
    for G in guesses:
        r = m.register(scan, G, levels=PYRAMID)
        ok, err = within_bounds(r["pose"], N.T_TRUE, P.map.pbar)
        assert ok and r["termination"] == _abi.NDT_CONVERGED, (err, r["termination"], [l["iterations"] for l in r["levels"]])
        o, olv = P.register(G, PYRAMID)
        for a, b in zip(r["levels"] + [r], olv + [o]):
            assert a["termination"] == b["termination"], (a["termination"], b["termination"])
            dt, deg = N.pose_error(a["pose"], b["pose"], P.map.pbar)
            assert dt <= 1e-5 and np.radians(deg) <= 1e-5, (dt, deg)


def test_out_is_register_from_the_last_level_and_levels_rise():
    m, scan, P, guesses = _convergence()
    for G in guesses[:2]:
        out, per = raw(m, scan, G, list(PYRAMID))
        r = m.register(scan, G, levels=PYRAMID)
        assert out == raw_register(m, scan, r["levels"][-1]["pose"])
        T = G
        for k, lv in zip(PYRAMID, r["levels"]):
            r0 = m.register(scan, T, levels=[dict(factor=k, max_iterations=0)], max_iterations=0)["levels"][0]
            assert lv["score"] >= r0["score"]
            T = lv["pose"]


def test_map_state_and_cache():
    pts = cloud()[:600_000]
    s1, s2 = scan_of(cloud()[600_000:], 30_000, 5), scan_of(cloud()[600_000:], 30_000, 6)
    q = scan_of(cloud(), 20_000, 7)
    T = N.pose((0.4, -0.3, 0.8), (0.05, -0.04, 0.01))

    def updated():
        m = make_map(pts)
        m.change2DMap(s1)
        return m

    a, b = updated(), updated()
    plain = raw_register(a, q, T)
    before = _state(a)
    first = raw(a, q, T, [8, 4, 2])
    assert _state(a) == before and raw_register(a, q, T) == plain
    # factors 8, then 2, then 8 against fresh handles with the same history
    for ks in ([8], [2], [8]):
        assert raw(a, q, T, ks) == raw(updated(), q, T, ks)
    assert raw(a, q, T, [8, 4, 2]) == first == raw(b, q, T, [8, 4, 2])
    level_eval(a, q, T, (8, 4, 2))
    # a remove, then a failed update: equal to a second handle with the same history
    a.del2DMap(s1); b.del2DMap(s1)
    assert raw(a, q, T, [8, 3]) == raw(b, q, T, [8, 3])
    level_eval(a, q, T, (8, 3))
    c = make_map(pts, max_voxels=make_map(pts).counts()["n_voxels"])
    raw(c, q, T, [8, 4, 2])
    far = s2.copy()
    far[:, 0] += 500.0
    c.change2DMap(far)
    with pytest.raises(g.GndtError) as e:
        c.register(q, T, levels=[4])
    assert e.value.status == _abi.GNDT_ERR_CAPACITY
    assert raw(c, q, T, [8, 4, 2]) == raw(make_map(pts), q, T, [8, 4, 2])
    level_eval(c, q, T, (8, 4, 2))


def test_determinism_and_null_level_out():
    m, scan, P, guesses = _convergence()
    a = raw(m, scan, guesses[0], list(PYRAMID))
    assert raw(m, scan, guesses[0], list(PYRAMID)) == a
    assert raw(m, scan, guesses[0], list(PYRAMID), with_levels=False)[0] == a[0]


def test_invalid_arguments():
    m = make_map(cloud()[:300_000])
    scan = np.ascontiguousarray(scan_of(cloud(), 5_000, 2)[:, :3], np.float32)
    L = g.lib()
    T = (C.c_double * 16)(*np.eye(4).ravel())
    p, out = _abi.default_ndt_params(), _abi.Registration()

    def call(levels, n=None, h=m._h):
        arr = (_abi.NdtLevel * max(len(levels), 1))(*levels) if levels is not None else None
        return L.gndt_register_levels(h, scan.ctypes.data, len(scan), 12, 0, T, C.byref(p), arr, len(levels or []) if n is None else n,
                                      C.byref(out), None, None)

    lv = _abi.default_ndt_level
    assert call([lv(8), lv(2)]) == 0
    assert call(None, 0) == 0
    bad = [(None, 1), ([lv(8)] * 9, None), ([lv(4)], -1), ([lv(1)], None), ([lv(33)], None), ([lv(4), lv(4)], None),
           ([lv(2), lv(4)], None), ([lv(4, max_iterations=-1)], None), ([lv(4, translation_epsilon=-1.0)], None),
           ([lv(4, rotation_epsilon=float("inf"))], None), ([lv(4, translation_epsilon=float("nan"))], None)]
    for levels, n in bad:
        assert call(levels, n) == _abi.GNDT_ERR_INVALID_ARG, (levels and [(l.factor, l.max_iterations) for l in levels], n)
    fresh = g.TwoDmap(0.2, 0.1)
    assert call([lv(4)], h=fresh._h) == _abi.GNDT_ERR_STATE
    with pytest.raises(g.GndtError) as e:
        m.register(scan, None, levels=[4, 8])
    assert e.value.status == _abi.GNDT_ERR_INVALID_ARG
