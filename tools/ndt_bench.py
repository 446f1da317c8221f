"""Time gndt_register on the benchmark map: the cfg2 cloud of bench.py (10 M points, 0.2 m / 0.1 m
cells) and scans of 100 k and 1 M of its points moved by a known pose, registered from a guess
0.05 m / 0.5 deg off.  Writes one JSON document (stdout, and --out if given):

  ms_per_register      host clock around the blocking call (it ends in a stream synchronise)
  iterations           derivative passes after the first
  pass_ms, prepare_ms  device time per derivative pass / per Gaussian prepare (torch.profiler
                       kernel records, in a separate profiled call)
  round_trip_share     1 - device time of one call / its host time: launches, read-backs, host LM
  pairs_per_pass, bytes_per_pass   from the counts: scan bytes + 80 B per (point, voxel) pair
                       (the column searches are not counted)

usage: python tools/ndt_bench.py [--reps 5] [--out ndt_bench.json]
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def kernel_ms(prof, name):
    tot, cnt = 0.0, 0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and name in e.name:
            tot += e.device_time_total / 1000.0 if hasattr(e, "device_time_total") else e.cuda_time_total / 1000.0
            cnt += 1
    return tot, cnt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    spec = synthetic.CONFIGS["cfg2"]
    cloud = synthetic.cfg2(spec.n)
    m = g.TwoDmap(spec.grid_len, spec.z_len)
    m.chatterCallback(torch.from_numpy(cloud).cuda())
    m.counts()
    T = N.pose((0.5, -0.4, 1.5), (0.4, -0.3, 0.05))
    res = {"card": card(), "map_points": spec.n, "grid_len": spec.grid_len, "z_len": spec.z_len, "scans": []}
    for n in (100_000, 1_000_000):
        pts = cloud[1 + np.sort(np.random.default_rng(n).choice(int(spec.n * 0.97), n, replace=False))]
        scan = torch.from_numpy(N.apply(np.linalg.inv(T), pts)).cuda()
        pbar = scan[:, :3].double().mean(0).cpu().numpy()
        guess = N.guesses(T, N.transform(T, pbar[None])[0], n=1, seed=1, max_t=0.05, max_deg=0.5)[0]
        m.register(scan, guess)  # warm-up (module load, prepare, scratch)
        times, r = [], None
        for _ in range(a.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = m.register(scan, guess)
            times.append((time.perf_counter() - t0) * 1e3)
        # device time per kernel, in a profiled call of its own; the prepare runs after a map change,
        # so the profiled call follows an update by an empty-effect scan (remove it again after)
        m.change2DMap(scan[:1000])
        m.del2DMap(scan[:1000])
        m.counts()
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rp = m.register(scan, guess)
            prof_ms = (time.perf_counter() - t0) * 1e3
        pass_ms, n_pass = kernel_ms(prof, "ndt_pass_kernel")
        prep_ms, n_prep = kernel_ms(prof, "ndt_prepare_kernel")
        dev_ms = sum(kernel_ms(prof, k)[0] for k in ("ndt_pass_kernel", "ndt_prepare_kernel", "ndt_mean_kernel", "ndt_finish_kernel"))
        med = float(np.median(times))
        steady_dev = dev_ms - prep_ms
        res["scans"].append({
            "points": n, "ms_per_register": med, "ms_min": float(min(times)), "iterations": r["iterations"],
            "termination": r["termination"], "passes": n_pass, "pass_ms": pass_ms / max(n_pass, 1),
            "prepare_ms": prep_ms / max(n_prep, 1), "device_ms_per_register": steady_dev,
            "round_trip_share": 1.0 - steady_dev / med, "profiled_call_ms": prof_ms,
            "pairs_per_pass": r["n_pairs"], "bytes_per_pass": 16 * n + 80 * r["n_pairs"],
            "pose_error_m_deg": N.pose_error(r["pose"], T, pbar), "same_as_profiled": bool(np.array_equal(rp["pose"], r["pose"])),
        })
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(txt)


if __name__ == "__main__":
    main()
