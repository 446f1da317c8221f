"""The D2D oracle (tests/ndt_d2d_oracle.py) on its own, without a GPU: its gradient and Hessian
against central differences of its own score with the pairs frozen, its reduction to the P2D pair
when the scan's covariance is zero, the basins D2D converges from on the dense-disc instance, and
the ctypes signature against include/gndt.h."""
import ctypes as C
import functools
import os
import subprocess
import tempfile

import numpy as np

import grid_ndt_b200 as g
from grid_ndt_b200 import _abi, _lib, synthetic
from oracle import oracle as O
from tests import ndt_d2d_oracle as D
from tests import ndt_oracle as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the pyramid and the guesses of the basin claims (shared with tests/test_gpu_ndt_d2d.py):
# N.guesses(n=6, seed=11, **BASIN)[i] for i in BASIN_GUESSES, as in tests/test_ndt_levels.py
PYRAMID = (8, 4, 2)
BASIN = dict(max_t=0.3, max_deg=3.0)
BASIN_GUESSES = (1, 2)
# usable scan Gaussians of the dense-disc instance (144 473 points) per factor
USABLE = {1: 11574, 2: 3903, 4: 1034, 8: 261}
MAP_LEVEL_ERROR = (5e-3, 0.02)  # m, deg: the bounds of tests/test_gpu_ndt.py's within_bounds


@functools.lru_cache(maxsize=2)
def instance(radius=10.0):
    """(map voxels, scan voxels, origin, scan) of D.d2d_instance, both built by the C oracle; the
    scan at the map's origin with every point binned."""
    cloud = synthetic.cfg2(900_000, scale=0.3)
    mp, scan = D.d2d_instance(cloud, radius)
    p = _abi.default_params(0.2, 0.1)
    mv = O.oracle_build(mp, p).voxels
    origin = cloud[0, :3]
    sv = O.oracle_build(scan, D.scan_params(p, origin)).voxels
    return mv, sv, origin, scan


def _fd(pr, T):
    e = pr.evaluate(T)
    h = 1e-6
    f = lambda xi: pr.frozen_score(T, e["pi"], e["vi"], xi)
    gd = np.array([(f(h * np.eye(6)[j]) - f(-h * np.eye(6)[j])) / (2 * h) for j in range(6)])
    h2 = 2e-5
    H = np.zeros((6, 6))
    for a in range(6):
        for b in range(6):
            ea, eb = h2 * np.eye(6)[a], h2 * np.eye(6)[b]
            H[a, b] = (f(ea + eb) - f(ea - eb) - f(-ea + eb) + f(-ea - eb)) / (4 * h2 * h2)
    return e, gd, H


def test_d2d_derivatives_match_finite_differences():
    mv, sv, origin, scan = instance(4.0)
    for k in (1, 4):
        pr = D.Problem(mv, sv, origin, 0.2, 0.1, scan, k)
        centre = N.transform(N.T_TRUE, pr.pbar[None])[0]
        for T in [N.T_TRUE] + N.guesses(N.T_TRUE, centre, n=2, seed=4, max_t=0.2, max_deg=2.0):
            e, gd, H = _fd(pr, T)
            assert e["n_pairs"] > 200, (k, e["n_pairs"])
            np.testing.assert_allclose(e["gradient"], gd, rtol=1e-5, atol=1e-6 * np.abs(e["gradient"]).max())
            np.testing.assert_allclose(e["hessian"], H, rtol=2e-3, atol=2e-3 * np.abs(e["hessian"]).max())


def test_zero_scan_covariance_is_the_p2d_pair():
    mv, sv, origin, scan = instance(4.0)
    pr = D.Problem(mv, sv, origin, 0.2, 0.1, scan)
    G = N.Gaussians(mv)
    assert np.array_equal(G.key, pr.G.key) and np.array_equal(G.count, pr.G.count)
    T = N.guesses(N.T_TRUE, N.transform(N.T_TRUE, pr.pbar[None])[0], n=2, seed=3, max_t=0.05, max_deg=0.5)[1]
    e = pr.evaluate(T, sig_s=np.zeros_like(pr.S.sig))
    assert e["n_pairs"] > 1000
    sel = np.random.default_rng(0).choice(e["n_pairs"], 300, replace=False)
    c = e["center"]
    for j in sel:
        pi, vi = e["pi"][j:j + 1], e["vi"][j:j + 1]
        d = D.derivatives(pr.G, np.zeros((len(e["x"]), 3, 3)), e["x"], c, T[:3, :3], pi, vi, pr.d1, pr.d2)
        p = N.derivatives(G, e["x"], c, pi, vi, pr.d1, pr.d2)  # a point at mu_i
        for a, b in zip(d, p):
            np.testing.assert_allclose(a, b, rtol=0, atol=1e-12 * np.abs(b).max())


def test_usable_scan_gaussians_per_level():
    """What the dense disc gives: thousands of scan Gaussians at the map level, fewer per level."""
    mv, sv, origin, scan = instance()
    P = D.Pyramid(mv, sv, origin, 0.2, 0.1, scan, PYRAMID)
    n = {k: len(pr.scan_gaussians()) for k, pr in [(1, P.map)] + list(P.levels.items())}
    assert n == USABLE, n


def test_d2d_basin_at_the_map_level():
    mv, sv, origin, scan = instance()
    pr = D.Problem(mv, sv, origin, 0.2, 0.1, scan)
    centre = N.transform(N.T_TRUE, pr.pbar[None])[0]
    for G in N.guesses(N.T_TRUE, centre, **N.GUESS_OFFSETS):
        r = pr.register(G)
        dt, deg = N.pose_error(r["pose"], N.T_TRUE, pr.pbar)
        assert r["termination"] == N.CONVERGED and dt <= MAP_LEVEL_ERROR[0] and deg <= MAP_LEVEL_ERROR[1], (dt, deg, r["iterations"])


def test_d2d_pyramid_does_not_widen_the_basin():
    """What the oracle shows from 0.3 m / 3 deg: every level converges, but the optimum of level 8
    (261 scan Gaussians of 1.6 m cells, binned in the scan's frame) lies 0.31 m from the true pose,
    levels 4 and 2 keep it, and the map level ends MAX_ITER about 0.36 m off.  Unlike P2D's pyramid
    (tests/test_ndt_levels.py), D2D 8 -> 4 -> 2 does not reach the true pose."""
    mv, sv, origin, scan = instance()
    P = D.Pyramid(mv, sv, origin, 0.2, 0.1, scan, PYRAMID)
    r8 = P.levels[8].register(N.T_TRUE)
    assert r8["termination"] == N.CONVERGED and N.pose_error(r8["pose"], N.T_TRUE, P.map.pbar)[0] > 0.25
    centre = N.transform(N.T_TRUE, P.map.pbar[None])[0]
    gs = N.guesses(N.T_TRUE, centre, n=6, seed=11, **BASIN)
    for i in BASIN_GUESSES:
        r, lv = P.register(gs[i], PYRAMID)
        assert all(l["termination"] == N.CONVERGED for l in lv), (i, [l["termination"] for l in lv])
        dt, deg = N.pose_error(r["pose"], N.T_TRUE, P.map.pbar)
        assert r["termination"] == N.MAX_ITER and dt > 0.25, (i, dt, deg, r["termination"])


def test_ctypes_signature_matches_header():
    src = ("#include \"gndt.h\"\n"
           "int (*f)(gndt_handle *, const void *, size_t, size_t, int, const double *, const gndt_ndt_params *,"
           " const gndt_ndt_level *, int, gndt_registration *, gndt_registration *, void *) = gndt_register_d2d;\n"
           "int (*l)(gndt_handle *, const void *, size_t, size_t, int, const double *, const gndt_ndt_params *,"
           " const gndt_ndt_level *, int, gndt_registration *, gndt_registration *, void *) = gndt_register_levels;\n")
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-c", "-I" + os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t.o")])
    assert _lib.SYMBOLS["gndt_register_d2d"] == _lib.SYMBOLS["gndt_register_levels"]
    out = _abi.Registration()
    assert g.lib().gndt_register_d2d(None, None, 0, 16, 0, None, None, None, 0, C.byref(out), None, None) == _abi.GNDT_ERR_INVALID_ARG
