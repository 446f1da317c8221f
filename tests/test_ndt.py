"""The NDT registration oracle (tests/ndt_oracle.py) on its own, without a GPU: derivatives
against finite differences, the vectorised cell key against the C oracle at cell edges, the
convergence instances of the GPU tests, and the ctypes mirrors against include/gndt.h."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import grid_ndt_b200 as g
from grid_ndt_b200 import _abi, synthetic
from oracle import oracle as O
from tests import ndt_oracle as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cloud():
    return synthetic.cfg2(900_000, scale=0.3)


def _instance(n_scan=30_000):
    cloud = _cloud()
    mp, scan = N.convergence_instance(cloud, n_scan)
    om = O.oracle_build(mp, _abi.default_params(0.2, 0.1))
    return N.Problem(om.voxels, cloud[0, :3], 0.2, 0.1, scan)


def test_derivatives_match_finite_differences():
    pr = _instance(4000)
    centre = N.transform(N.T_TRUE, pr.pbar[None])[0]
    poses = [N.T_TRUE] + N.guesses(N.T_TRUE, centre, n=3, seed=2, max_t=0.05, max_deg=0.5)
    for T in poses:
        e = pr.evaluate(T)
        assert e["n_pairs"] > 1000
        h = 1e-6
        gd = np.array([(pr.frozen_score(T, e["pi"], e["vi"], h * np.eye(6)[k]) - pr.frozen_score(T, e["pi"], e["vi"], -h * np.eye(6)[k])) / (2 * h)
                       for k in range(6)])
        np.testing.assert_allclose(e["gradient"], gd, rtol=1e-5, atol=1e-6 * np.abs(e["gradient"]).max())
        # Hessian: central differences of the analytic gradient, pairs frozen
        x = N.transform(T, pr.p)
        c = pr.center(T)

        def grad(xi):
            xn = (x - c) @ N.so3_exp(xi[3:]).T + c + xi[:3]
            # the gradient about the moved centre equals d/dxi of S composed with the increment
            return N.derivatives(pr.G, xn, c + xi[:3], e["pi"], e["vi"], pr.d1, pr.d2)[1]

        hd = np.array([(grad(h * np.eye(6)[k]) - grad(-h * np.eye(6)[k])) / (2 * h) for k in range(3)])
        np.testing.assert_allclose(e["hessian"][:3], hd, rtol=1e-4, atol=1e-5 * np.abs(e["hessian"]).max())
        # all 6 x 6 by second differences of S
        h2 = 2e-5
        f = lambda xi: pr.frozen_score(T, e["pi"], e["vi"], xi)
        H = np.zeros((6, 6))
        for k in range(6):
            for l in range(6):
                ek, el = h2 * np.eye(6)[k], h2 * np.eye(6)[l]
                H[k, l] = (f(ek + el) - f(ek - el) - f(-ek + el) + f(-ek - el)) / (4 * h2 * h2)
        np.testing.assert_allclose(e["hessian"], H, rtol=2e-3, atol=2e-3 * np.abs(e["hessian"]).max())


def test_vectorised_key_matches_c_oracle_at_cell_edges():
    rng = np.random.default_rng(1)
    for origin, gl, zl in (((0.013, -4.7, 1.0), 0.2, 0.1), ((-3.3, 7.25, -0.5), 0.1, 0.05)):
        o = np.array(origin, np.float32)
        pts = []
        for k in list(rng.integers(-300, 300, 40)) + [1, -1, 0, 32767, -32767, 32766, -32766]:
            for ax, L in ((0, gl), (1, gl), (2, zl)):
                e = np.float32(o[ax] + np.float32(k) * np.float32(L))
                for v in (np.nextafter(e, np.float32(-np.inf)), e, np.nextafter(e, np.float32(np.inf))):
                    for sign in (1, -1):
                        p = o.copy() + np.float32(sign) * np.float32(0.37) * np.float32(L)
                        p[ax] = v if sign > 0 else np.float32(2 * o[ax] - v)
                        pts.append(p.astype(np.float32))
        pts = np.array(pts, np.float32)
        cx, cy, cz, ok = N.keys(pts, o, gl, zl)
        for i, p in enumerate(pts):
            rc, sx, sy, sz = O.oracle_trans(o, gl, zl, p)
            assert (rc == 0) == bool(ok[i]), p
            if rc == 0:
                assert (N.contiguous(sx), N.contiguous(sy), N.contiguous(sz)) == (cx[i], cy[i], cz[i]), p


def test_oracle_converges_on_the_gpu_instances():
    pr = _instance()
    centre = N.transform(N.T_TRUE, pr.pbar[None])[0]
    for G in N.guesses(N.T_TRUE, centre, **N.GUESS_OFFSETS):
        r = pr.register(G)
        dt, deg = N.pose_error(r["pose"], N.T_TRUE, pr.pbar)
        assert r["termination"] == N.CONVERGED and dt <= 5e-3 and deg <= 0.02, (dt, deg, r["termination"])


def test_oracle_registers_the_workflow_scans():
    """The scans of the register -> transform -> update GPU test, each against the initial map."""
    cloud = _cloud()
    mp, scans = N.workflow_instance(cloud)
    om = O.oracle_build(mp, _abi.default_params(0.2, 0.1))
    for scan, T, guess in scans:
        pr = N.Problem(om.voxels, cloud[0, :3], 0.2, 0.1, scan)
        r = pr.register(guess)
        dt, deg = N.pose_error(r["pose"], T, pr.pbar)
        assert dt <= 5e-3 and deg <= 0.02, (dt, deg, r["termination"])


def test_ctypes_structs_match_header():
    src = ("#include <stdio.h>\n#include <stddef.h>\n#include \"gndt.h\"\nint main(){printf(\"%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n\","
           " sizeof(gndt_ndt_params), offsetof(gndt_ndt_params, translation_epsilon), offsetof(gndt_ndt_params, rotation_epsilon),"
           " sizeof(gndt_registration), offsetof(gndt_registration, center), offsetof(gndt_registration, score),"
           " offsetof(gndt_registration, hessian), offsetof(gndt_registration, n_points), offsetof(gndt_registration, iterations),"
           " offsetof(gndt_registration, termination)); return 0;}\n")
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I" + os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")])
        got = [int(x) for x in subprocess.check_output([os.path.join(d, "t")]).split()]
    P, R = _abi.NdtParams, _abi.Registration
    assert got == [C.sizeof(P), P.translation_epsilon.offset, P.rotation_epsilon.offset, C.sizeof(R), R.center.offset,
                   R.score.offset, R.hessian.offset, R.n_points.offset, R.iterations.offset, R.termination.offset]


def test_default_ndt_params_match_library():
    p = _abi.NdtParams()
    g.lib().gndt_default_ndt_params(C.byref(p))
    q = _abi.default_ndt_params()
    assert bytes(p) == bytes(q)
    assert [getattr(p, k) for k in ("min_voxel_points", "max_iterations", "reserved")] == [6, 100, 0]
    assert abs(p.outlier_ratio - 0.55) < 1e-7 and N.DEFAULTS["max_iterations"] == 100


def test_register_rejects_null_handle():
    out = _abi.Registration()
    assert g.lib().gndt_register(None, None, 0, 16, 0, None, None, C.byref(out), None) == _abi.GNDT_ERR_INVALID_ARG
