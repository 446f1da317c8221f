"""Time coarse-to-fine registration (gndt_register_levels) against single-level gndt_register on
the map of tools/ndt_bench.py: the cfg2 cloud of bench.py (10 M points, 0.2 m / 0.1 m cells) and
scans of 100 k and 1 M of its points moved by a known pose, from guesses 0.05 m / 0.5 deg and
0.3 m / 3 deg per axis off.  Writes one JSON document (stdout, and --out if given):

  ms_per_call        host clock around the blocking call, median of --reps
  levels             per level (the map level last): passes and device ms per pass of
                     ndt_pass_kernel (torch.profiler kernel records, in a separate call)
  level_build_ms     device time of the level-build kernels per factor, after a map change
  pose_error_m_deg   against the true pose, at the scan's centroid

--ab LIB: also compare the device time per map-level pass with another build of libgndt.so
(GNDT_LIB), alternating the two builds in fresh processes.

usage: python tools/ndt_levels_bench.py [--reps 5] [--out f.json] [--ab /path/to/libgndt.so]
"""
import argparse
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
from grid_ndt_b200 import synthetic  # noqa: E402
from tests import ndt_oracle as N  # noqa: E402
from tools.ndt_bench import card  # noqa: E402

PYRAMID = (8, 4, 2)
OFFSETS = {"5cm_0.5deg": dict(max_t=0.05, max_deg=0.5), "30cm_3deg": dict(max_t=0.3, max_deg=3.0)}
T_TRUE = N.pose((0.5, -0.4, 1.5), (0.4, -0.3, 0.05))


def cuda_events(prof):
    return [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def dev_ms(e):
    return (e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total) / 1000.0


def setup():
    spec = synthetic.CONFIGS["cfg2"]
    cloud = synthetic.cfg2(spec.n)
    m = g.TwoDmap(spec.grid_len, spec.z_len)
    m.chatterCallback(torch.from_numpy(cloud).cuda())
    m.counts()
    return spec, cloud, m


def scan_of(spec, cloud, n):
    pts = cloud[1 + np.sort(np.random.default_rng(n).choice(int(spec.n * 0.97), n, replace=False))]
    scan = torch.from_numpy(N.apply(np.linalg.inv(T_TRUE), pts)).cuda()
    pbar = scan[:, :3].double().mean(0).cpu().numpy()
    return scan, pbar


def invalidate(m, scan):
    """A map change that leaves the map as it was: the next call rebuilds Gaussians and levels."""
    m.change2DMap(scan[:1000])
    m.del2DMap(scan[:1000])
    m.counts()


def pass_only(reps):
    """Device ms per map-level ndt_pass_kernel, single level, 1 M scan, 5 cm guess."""
    if os.environ.get("GNDT_LIB"):  # another build, which may predate the level or D2D entry points
        from grid_ndt_b200 import _lib
        for s in ("gndt_default_ndt_level", "gndt_register_levels", "gndt_register_d2d"):
            _lib.SYMBOLS.pop(s, None)
    spec, cloud, m = setup()
    scan, pbar = scan_of(spec, cloud, 1_000_000)
    guess = N.guesses(T_TRUE, N.transform(T_TRUE, pbar[None])[0], n=1, seed=1, **OFFSETS["5cm_0.5deg"])[0]
    m.register(scan, guess)
    from torch.profiler import ProfilerActivity, profile
    out = []
    for _ in range(reps):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.register(scan, guess)
        ev = [e for e in cuda_events(prof) if "ndt_pass_kernel" in e.name]
        out.append(sum(map(dev_ms, ev)) / len(ev))
    print(json.dumps({"pass_ms": out}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    ap.add_argument("--ab", default="")
    ap.add_argument("--pass-only", action="store_true")
    a = ap.parse_args()
    if a.pass_only:
        return pass_only(a.reps)
    from torch.profiler import ProfilerActivity, profile
    spec, cloud, m = setup()
    res = {"card": card(), "map_points": spec.n, "grid_len": spec.grid_len, "z_len": spec.z_len, "pyramid": PYRAMID, "runs": []}
    for n in (100_000, 1_000_000):
        scan, pbar = scan_of(spec, cloud, n)
        centre = N.transform(T_TRUE, pbar[None])[0]
        for oname, off in OFFSETS.items():
            guess = N.guesses(T_TRUE, centre, n=1, seed=1, **off)[0]
            for mode, levels in (("single", None), ("pyramid", PYRAMID)):
                m.register(scan, guess, levels=levels)  # warm-up: module load, Gaussians, levels, scratch
                times, r = [], None
                for _ in range(a.reps):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    r = m.register(scan, guess, levels=levels)
                    times.append((time.perf_counter() - t0) * 1e3)
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    rp = m.register(scan, guess, levels=levels)
                passes = [e for e in cuda_events(prof) if "ndt_pass_kernel" in e.name]
                per, i = [], 0
                for k, lv in zip(levels or (), r["levels"] if levels else ()):
                    c = lv["iterations"] + 1
                    per.append({"factor": k, "passes": c, "pass_ms": sum(map(dev_ms, passes[i:i + c])) / c,
                                "iterations": lv["iterations"], "termination": lv["termination"]})
                    i += c
                c = len(passes) - i
                per.append({"factor": 1, "passes": c, "pass_ms": sum(map(dev_ms, passes[i:])) / max(c, 1),
                            "iterations": r["iterations"], "termination": r["termination"]})
                res["runs"].append({
                    "points": n, "offset": oname, "mode": mode, "ms_per_call": float(np.median(times)), "ms_min": float(min(times)),
                    "levels": per, "termination": r["termination"], "pose_error_m_deg": N.pose_error(r["pose"], T_TRUE, pbar),
                    "same_as_profiled": bool(np.array_equal(rp["pose"], r["pose"]))})
                print(json.dumps(res["runs"][-1]), file=sys.stderr, flush=True)
        if n == 100_000:  # level build: the kernels of one pyramid call right after a map change
            invalidate(m, scan)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                m.register(scan, guess, levels=PYRAMID, max_iterations=0)
            build = [e for e in cuda_events(prof) if "ndt_level_" in e.name or "exclusive_scan" in e.name]
            build.sort(key=lambda e: e.time_range.start)
            res["level_build_ms"] = {k: sum(map(dev_ms, build[6 * j:6 * j + 6])) for j, k in enumerate(PYRAMID)}
            res["level_build_kernels"] = len(build)
    if a.ab:
        ab = {"new": [], "base": []}
        for _ in range(3):
            for name, lib in (("new", ""), ("base", a.ab)):
                env = dict(os.environ)
                env.pop("GNDT_LIB", None)
                if lib:
                    env["GNDT_LIB"] = lib
                q = subprocess.run([sys.executable, os.path.abspath(__file__), "--pass-only", "--reps", "3"], env=env, capture_output=True,
                                   text=True, check=True)
                ab[name] += json.loads(q.stdout.strip().splitlines()[-1])["pass_ms"]
        res["map_pass_ms_ab"] = {k: {"median": float(np.median(v)), "all": v} for k, v in ab.items()}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(txt)


if __name__ == "__main__":
    main()
