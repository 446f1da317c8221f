"""Time distribution-to-distribution registration (gndt_register_d2d) against point-to-distribution
(gndt_register / gndt_register_levels) on the map of tools/ndt_levels_bench.py: the cfg2 cloud of
bench.py (10 M points, 0.2 m / 0.1 m cells).  The scans are dense discs of about 100 k and 1 M
points (EVERY point within a radius of the cloud's median x-y, so that cells hold enough points for
a scan Gaussian), moved by a known pose, from guesses 0.05 m / 0.5 deg and 0.3 m / 3 deg per axis
off.  Modes: P2D single, P2D 8 -> 4 -> 2, D2D single, D2D 8 -> 4 -> 2, on the same scans.  Writes
one JSON document (stdout, and --out if given):

  ms_per_call        host clock around the blocking call, median of --reps
  levels             per level (the map level last): passes, device ms per pass of the pass kernel
                     (torch.profiler kernel records, in a separate call), usable scan Gaussians
                     (D2D) or finite points (P2D)
  scan_build_ms      D2D: device ms per call of the scan's build, its Sigma' prepare and level tables
  first_call_ms      D2D: host ms of the first call on a handle minus a warm call (creates the scan
                     builder, the map's Sigma' tables and scratch)
  pose_error_m_deg   against the true pose, at the scan's centroid

--ab LIB: also compare the raw P2D results (gndt_register, gndt_register_levels) of this build with
another build of libgndt.so (GNDT_LIB) on the same map and scans, in fresh processes.

usage: python tools/ndt_d2d_bench.py [--reps 5] [--out f.json] [--ab /path/to/libgndt.so]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import grid_ndt_b200 as g  # noqa: E402
from grid_ndt_b200 import _abi, synthetic  # noqa: E402
from tests import ndt_oracle as N  # noqa: E402
from tools.ndt_bench import card  # noqa: E402
from tools.ndt_levels_bench import OFFSETS, PYRAMID, T_TRUE, cuda_events, dev_ms  # noqa: E402

SIZES = (100_000, 1_000_000)
PASS = {"p2d": "ndt_pass_kernel", "d2d": "ndt_d2d_pass_kernel"}
# kernels of a warm call that are not the scan's build: mean, passes, finish
SOLVER = ("ndt_mean_kernel", "ndt_pass_kernel", "ndt_d2d_pass_kernel", "ndt_finish_kernel")


def setup():
    spec = synthetic.CONFIGS["cfg2"]
    cloud = synthetic.cfg2(spec.n)
    m = g.TwoDmap(spec.grid_len, spec.z_len)
    m.chatterCallback(torch.from_numpy(cloud).cuda())
    m.counts()
    return spec, cloud, m


def dense_scan(cloud, n):
    """Every point of the cloud within the radius of its median x-y that holds n of them."""
    xy = cloud[1:, :2].astype(np.float64)
    d = np.hypot(*(xy - np.median(xy, 0)).T)
    radius = np.partition(d, n - 1)[n - 1]
    pts = cloud[1:][d <= radius]
    scan = torch.from_numpy(N.apply(np.linalg.inv(T_TRUE), pts)).cuda()
    return scan, scan[:, :3].double().mean(0).cpu().numpy(), float(radius)


def p2d_dump():
    """sha256 of the raw gndt_register / gndt_register_levels structs on every scan and guess."""
    if os.environ.get("GNDT_LIB"):  # another build: only the P2D entry points are used
        from grid_ndt_b200 import _lib
        _lib.SYMBOLS.pop("gndt_register_d2d", None)
    spec, cloud, m = setup()
    L, h = g.lib(), hashlib.sha256()
    for n in SIZES:
        scan, pbar, _ = dense_scan(cloud, n)
        sc = scan.contiguous()
        centre = N.transform(T_TRUE, pbar[None])[0]
        for off in OFFSETS.values():
            T = N.guesses(T_TRUE, centre, n=1, seed=1, **off)[0]
            Tc = (C.c_double * 16)(*T.ravel())
            p, out = _abi.default_ndt_params(), _abi.Registration()
            assert L.gndt_register(m._h, sc.data_ptr(), len(sc), 16, 1, Tc, C.byref(p), C.byref(out), None) == 0
            h.update(bytes(out))
            lv = (_abi.NdtLevel * 3)(*[_abi.default_ndt_level(k) for k in PYRAMID])
            per = (_abi.Registration * 3)()
            assert L.gndt_register_levels(m._h, sc.data_ptr(), len(sc), 16, 1, Tc, C.byref(p), lv, 3, C.byref(out), per, None) == 0
            h.update(bytes(out) + bytes(per))
    print(json.dumps({"sha256": h.hexdigest()}))


def call(m, scan, guess, method, levels):
    return m.register(scan, guess, levels=levels, method=method)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    ap.add_argument("--ab", default="")
    ap.add_argument("--p2d-dump", action="store_true")
    a = ap.parse_args()
    if a.p2d_dump:
        return p2d_dump()
    from torch.profiler import ProfilerActivity, profile
    spec, cloud, m = setup()
    res = {"card": card(), "map_points": spec.n, "grid_len": spec.grid_len, "z_len": spec.z_len, "pyramid": PYRAMID, "runs": []}
    for n in SIZES:
        scan, pbar, radius = dense_scan(cloud, n)
        centre = N.transform(T_TRUE, pbar[None])[0]
        # first-call cost on a fresh handle: scan builder, Sigma' tables of the map, scratch
        f = g.TwoDmap(spec.grid_len, spec.z_len)
        f.chatterCallback(torch.from_numpy(cloud).cuda())
        f.counts()
        guess0 = N.guesses(T_TRUE, centre, n=1, seed=1, **OFFSETS["5cm_0.5deg"])[0]
        first = []
        for _ in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f.register(scan, guess0, method="d2d", max_iterations=0)
            first.append((time.perf_counter() - t0) * 1e3)
        f.close()
        res.setdefault("first_call_ms", {})[n] = {"first": first[0], "warm": first[1], "difference": first[0] - first[1]}
        for oname, off in OFFSETS.items():
            guess = N.guesses(T_TRUE, centre, n=1, seed=1, **off)[0]
            for method in ("p2d", "d2d"):
                for mode, levels in (("single", None), ("pyramid", PYRAMID)):
                    call(m, scan, guess, method, levels)  # warm-up: module load, Gaussians, levels, scratch
                    times, r = [], None
                    for _ in range(a.reps):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        r = call(m, scan, guess, method, levels)
                        times.append((time.perf_counter() - t0) * 1e3)
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        rp = call(m, scan, guess, method, levels)
                    ev = cuda_events(prof)
                    passes = [e for e in ev if e.name.split("(")[0].endswith(PASS[method])]
                    per, i = [], 0
                    for k, lv in list(zip(levels or (), r["levels"] if levels else ())) + [(1, r)]:
                        c = lv["iterations"] + 1
                        per.append({"factor": k, "passes": c, "pass_ms": sum(map(dev_ms, passes[i:i + c])) / c, "n_points": lv["n_points"],
                                    "iterations": lv["iterations"], "termination": lv["termination"]})
                        i += c
                    run = {"points": int(len(scan)), "radius_m": radius, "offset": oname, "method": method, "mode": mode,
                           "ms_per_call": float(np.median(times)), "ms_min": float(min(times)), "levels": per,
                           "passes_profiled": len(passes), "termination": r["termination"],
                           "pose_error_m_deg": N.pose_error(r["pose"], T_TRUE, pbar), "same_as_profiled": bool(np.array_equal(rp["pose"], r["pose"]))}
                    if method == "d2d":
                        run["scan_build_ms"] = sum(dev_ms(e) for e in ev if not any(s in e.name for s in SOLVER))
                    res["runs"].append(run)
                    print(json.dumps(run), file=sys.stderr, flush=True)
    if a.ab:
        ab = {}
        for name, lib in (("new", ""), ("base", a.ab)):
            env = dict(os.environ)
            env.pop("GNDT_LIB", None)
            if lib:
                env["GNDT_LIB"] = lib
            q = subprocess.run([sys.executable, os.path.abspath(__file__), "--p2d-dump"], env=env, capture_output=True, text=True, check=True)
            ab[name] = json.loads(q.stdout.strip().splitlines()[-1])["sha256"]
        res["p2d_raw_sha256_ab"] = dict(ab, identical=ab["new"] == ab["base"])
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(txt)


if __name__ == "__main__":
    main()
