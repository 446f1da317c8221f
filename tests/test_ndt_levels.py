"""The NDT level oracle (tests/ndt_levels_oracle.py) on its own, without a GPU: merged Gaussians
against the raw points, the floor division, coarse derivatives against finite differences, the
wider basin of the pyramid on the convergence instance, each hand-made boundary of
tests/ndt_levels_cases.py, and the ctypes mirrors against include/gndt.h and the library."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import grid_ndt_b200 as g
from grid_ndt_b200 import _abi, synthetic
from oracle import oracle as O
from tests import ndt_levels_cases as K
from tests import ndt_levels_oracle as NL
from tests import ndt_oracle as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# The pyramid and the guesses of the basin claim (shared with tests/test_gpu_ndt_levels.py):
# N.guesses(n=6, seed=11, **BASIN)[i] for i in BASIN_GUESSES.  From guess 2 single-level
# registration stalls 0.19 m / 2.5 deg from the true pose; guess 5 ends MAX_ITER 0.28 m / 4.3 deg off.
PYRAMID = (8, 4, 2)
BASIN = dict(max_t=0.3, max_deg=3.0)
BASIN_GUESSES = (1, 2, 5)


def _cloud():
    return synthetic.cfg2(900_000, scale=0.3)


def oracle_map(pts, grid=K.GRID, zlen=K.ZLEN, **kw):
    return O.oracle_build(pts, _abi.default_params(grid, zlen, **kw)).voxels


def test_merged_gaussians_equal_raw_moments():
    rng = np.random.default_rng(3)
    cells = K.block((-9, 9), (-7, 8), (-5, 5))
    cells = cells[rng.random(len(cells)) < 0.6]
    npts = rng.choice([1, 2, 4], len(cells), p=[0.15, 0.15, 0.7])
    pts = K.cloud_of(cells, npts)
    vox = oracle_map(pts)
    fitted = (vox["flags"] & 1) != 0
    fit_keys = set(zip(*(N.contiguous(vox[f][fitted]) for f in ("sx", "sy", "sz"))))
    cx, cy, cz, ok = N.keys(pts[1:, :3], np.zeros(3, np.float32), K.GRID, K.ZLEN)
    assert ok.all()
    for k in (2, 3, 4, 7):
        key, n, mu, S = NL.merged_moments(vox, k)
        keep = np.array([c in fit_keys for c in zip(cx, cy, cz)])
        p = pts[1:, :3].astype(np.float64)[keep]
        pk = N._pack(NL.floor_div(cx[keep], k), NL.floor_div(cy[keep], k), NL.floor_div(cz[keep], k))
        assert set(pk) == set(key[n > 0])
        for j, kk in enumerate(key):
            q = p[pk == kk]
            assert n[j] == len(q)
            if not len(q):
                continue
            m = q.mean(0)
            d = q - m
            s = np.array([(d[:, a] * d[:, b]).sum() for a, b in zip([0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2])])
            assert np.all(np.abs(mu[j] - m) <= 1e-12 * np.abs(m).max() + 1e-300)
            assert np.all(np.abs(S[j] - s) <= 1e-12 * np.abs(s).max() + 1e-300)


def _brute_floor(c, k):
    X = 0
    while X * k > c:
        X -= 1
    while (X + 1) * k <= c:
        X += 1
    return X


def test_floor_division_against_brute_force():
    c = list(range(-40, 41)) + [32767, 32766, 32765, -32767, -32766, -32765]
    for k in range(1, 33):
        assert list(NL.floor_div(c, k)) == [_brute_floor(ci, k) for ci in c], k
        if k > 1:  # contiguous -1 and 0 never share a coarse cell
            assert NL.floor_div(-1, k) == -1 and NL.floor_div(0, k) == 0
    # k that does not divide the extent [-32767, 32766]
    c = np.arange(-32767, 32767)
    for k in (3, 7, 32):
        q = NL.floor_div(c, k)
        assert np.all(q * k <= c) and np.all(c < (q + 1) * k)
        assert (q[0], q[-1]) == (_brute_floor(-32767, k), _brute_floor(32766, k))


def _instance(n_scan=30_000):
    cloud = _cloud()
    mp, scan = N.convergence_instance(cloud, n_scan)
    om = O.oracle_build(mp, _abi.default_params(0.2, 0.1))
    return om.voxels, cloud[0, :3], scan


def test_coarse_derivatives_match_finite_differences():
    vox, origin, scan = _instance(4000)
    for k in (2, 8):
        pr = NL.Level(vox, origin, 0.2, 0.1, scan, k)
        centre = N.transform(N.T_TRUE, pr.pbar[None])[0]
        for T in [N.T_TRUE] + N.guesses(N.T_TRUE, centre, n=2, seed=4, max_t=0.2, max_deg=2.0):
            e = pr.evaluate(T)
            assert e["n_pairs"] > 1000
            h = 1e-6
            gd = np.array([(pr.frozen_score(T, e["pi"], e["vi"], h * np.eye(6)[j]) - pr.frozen_score(T, e["pi"], e["vi"], -h * np.eye(6)[j]))
                           / (2 * h) for j in range(6)])
            np.testing.assert_allclose(e["gradient"], gd, rtol=1e-5, atol=1e-6 * np.abs(e["gradient"]).max())
            h2 = 2e-5
            f = lambda xi: pr.frozen_score(T, e["pi"], e["vi"], xi)
            H = np.zeros((6, 6))
            for a in range(6):
                for b in range(6):
                    ea, eb = h2 * np.eye(6)[a], h2 * np.eye(6)[b]
                    H[a, b] = (f(ea + eb) - f(ea - eb) - f(-ea + eb) + f(-ea - eb)) / (4 * h2 * h2)
            np.testing.assert_allclose(e["hessian"], H, rtol=2e-3, atol=2e-3 * np.abs(e["hessian"]).max())


def test_pyramid_widens_the_basin():
    vox, origin, scan = _instance()
    P = NL.Pyramid(vox, origin, 0.2, 0.1, scan, PYRAMID)
    centre = N.transform(N.T_TRUE, P.map.pbar[None])[0]
    gs = N.guesses(N.T_TRUE, centre, n=6, seed=11, **BASIN)
    for i in BASIN_GUESSES:
        r, lv = P.register(gs[i], PYRAMID)
        dt, deg = N.pose_error(r["pose"], N.T_TRUE, P.map.pbar)
        assert r["termination"] == N.CONVERGED and dt <= 5e-3 and deg <= 0.02, (i, dt, deg, [l["iterations"] for l in lv])
    r = P.map.register(gs[2])  # single level from the same guess
    dt, deg = N.pose_error(r["pose"], N.T_TRUE, P.map.pbar)
    assert not (dt <= 5e-3 and deg <= 0.02), (dt, deg)


# ---- the hand-made boundaries of the GPU tests, checked on the oracle ----------------------

def _map_cells(x):
    cx, cy, cz, ok = N.keys(x[:, :3].astype(np.float32), np.zeros(3, np.float32), K.GRID, K.ZLEN)
    assert ok.all()
    return cx, cy, cz


@pytest.mark.parametrize("k", [2, 3, 4, 8])
def test_edge_scans_put_points_where_they_claim(k):
    for axis in range(3):
        for coarse in (True, False):
            s = K.edge_scan(k, axis, coarse)
            c = _map_cells(s)[axis].reshape(-1, 3)  # (below, on, above) per edge
            edges = np.array([X * k for X in (-3, -1, 0, 1, 2)] if coarse else [X * k + j for X in (-3, -1, 0, 1, 2) for j in range(1, k)])
            # a point on edge e * len lies in cell e - 1 when e > 0, in cell e when e <= 0 (binning's ceil)
            on = np.where(edges > 0, edges - 1, np.where(edges == 0, -1, edges))
            assert np.array_equal(c[:, 0], edges - 1) and np.array_equal(c[:, 1], on) and np.array_equal(c[:, 2], edges)
            X = NL.floor_div(c, k)
            if coarse:  # one ulp either side of a coarse edge: different coarse cells
                assert np.all(X[:, 0] != X[:, 2])
            else:       # map-cell edges inside a coarse cell: the same one
                assert np.all(X[:, 0] == X[:, 2])
    # the -1/0 crossing: coordinate 0 and one ulp above it on every axis
    s = K.edge_scan(k, 2, True, around=(0,))
    assert list(_map_cells(s)[2]) == [-1, -1, 0]


@pytest.mark.parametrize("k", [2, 3, 8])
def test_slab_maps_are_what_they_claim(k):
    for name, (c, _) in K.slab_maps(k).items():
        vox = oracle_map(c)
        cx = N.contiguous(vox["sx"])
        rows = set(cx % k)
        cols = {(x, y) for x, y in zip(cx, N.contiguous(vox["sy"]))}
        X = {(int(a), int(b)) for a, b in zip(NL.floor_div(cx, k), NL.floor_div(N.contiguous(vox["sy"]), k))}
        per_coarse = {}
        for x, y in cols:
            per_coarse.setdefault((x // k, y // k), set()).add(x % k)
        want = {"first_row": rows == {0}, "last_row": rows == {k - 1},
                "all_columns": len(cols) == 6 * k * k and all(len(r) == k for r in per_coarse.values()),
                "missing_rows": rows == {0, k - 1},
                "single_column": len(cols) == 1 and len(X) == 1}[name]
        assert want, name


def test_mixed_and_count_maps_are_what_they_claim():
    for k in (2, 3, 8):
        vox = oracle_map(K.mixed_map(k))
        f = (vox["flags"] & 1) != 0
        key = N._pack(*NL.coarse_keys(vox, k))
        assert any(f[key == u].any() and (~f[key == u]).any() for u in np.unique(key))
        G = NL.CoarseGaussians(vox, k)
        key_f, n, _, _ = NL.merged_moments(vox, k)
        assert np.array_equal(n, [vox["count"][(key == u) & f].sum() for u in key_f])
    for k in (2, 5):
        vox = oracle_map(K.count_map(k))
        G = NL.CoarseGaussians(vox, k)
        assert len(vox) == 2 and list(G.count) == [8]


def test_extreme_map_reaches_the_index_limit():
    vox = oracle_map(K.extreme_map())
    for f in ("sx", "sy", "sz"):
        assert vox[f].max() == 32767 and vox[f].min() == -32767
    for k in (2, 3, 32):
        X = NL.coarse_keys(vox, k)[0]
        assert X.max() == 32766 // k and X.min() == -((32767 + k - 1) // k)


def test_ctypes_level_struct_matches_header_and_defaults_match_library():
    src = ("#include <stdio.h>\n#include <stddef.h>\n#include \"gndt.h\"\nint main(){printf(\"%zu %zu %zu %zu %d\\n\","
           " sizeof(gndt_ndt_level), offsetof(gndt_ndt_level, max_iterations), offsetof(gndt_ndt_level, translation_epsilon),"
           " offsetof(gndt_ndt_level, rotation_epsilon), GNDT_NDT_MAX_LEVELS); return 0;}\n")
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I" + os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")])
        got = [int(x) for x in subprocess.check_output([os.path.join(d, "t")]).split()]
    L = _abi.NdtLevel
    assert got == [C.sizeof(L), L.max_iterations.offset, L.translation_epsilon.offset, L.rotation_epsilon.offset, _abi.NDT_MAX_LEVELS]
    for k in (2, 8, 32):
        a = _abi.NdtLevel()
        g.lib().gndt_default_ndt_level(C.byref(a), k)
        assert bytes(a) == bytes(_abi.default_ndt_level(k))
        assert (a.factor, a.max_iterations, a.translation_epsilon, a.rotation_epsilon) == (k, 50, 1e-3, 1e-3)
    assert NL.LEVEL_DEFAULTS == dict(max_iterations=50, translation_epsilon=1e-3, rotation_epsilon=1e-3)
    out = _abi.Registration()
    assert g.lib().gndt_register_levels(None, None, 0, 16, 0, None, None, None, 0, C.byref(out), None, None) == _abi.GNDT_ERR_INVALID_ARG
