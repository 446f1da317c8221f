"""A/B stage timings of libgndt variants (GNDT_LIB) on the same clouds, one process per variant.
usage: ab_variants.py [--cfgs cfg2:10000000,cfg3:20000000] [--builds 8] lib1.so lib2.so ...   ('default' = in-tree lib)"""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

WORKER = r'''
import json, os, sys
sys.path.insert(0, %r)
import numpy as np, torch
from grid_ndt_b200 import TwoDmap
path, gl, zl, builds = sys.argv[1], float(sys.argv[2]), float(sys.argv[3]), int(sys.argv[4])
cloud = torch.from_numpy(np.load(path)).cuda()
m = TwoDmap(gl, zl); m.setInterval(0.08); m.stage_timing(os.environ.get("GNDT_STAGES", "1") == "1")
best, tot = None, []
for _ in range(builds):
    m.chatterCallback(cloud, "slope"); torch.cuda.synchronize()
    s = m.stage_ms(); tot.append(s["total"])
    best = s if best is None else {k: min(best[k], s[k]) for k in s}
c = m.counts()
print(json.dumps({"lib": os.path.basename(os.environ.get("GNDT_LIB", "default")), "stage_ms": {k: round(v, 4) for k, v in best.items() if k != "h2d"},
                  "median_total": round(sorted(tot)[len(tot) // 2], 4), "layout": m.key_layout(), "voxels": c["n_voxels"], "launches": m.launch_count()}))
''' % ROOT

ap = argparse.ArgumentParser()
ap.add_argument("--cfgs", default="cfg2:10000000")
ap.add_argument("--builds", type=int, default=8)
ap.add_argument("libs", nargs="*", default=["default"])
a = ap.parse_args()
from grid_ndt_b200 import synthetic
for item in a.cfgs.split(","):
    parts = item.split(":")
    name, n = parts[0], int(parts[1])
    spec = synthetic.CONFIGS[name]
    gl = float(parts[2]) if len(parts) > 2 else spec.grid_len
    kw = {}
    if name == "cfg2" and n != spec.n: kw["scale"] = (n / spec.n) ** 0.5
    if name in ("cfg3", "cfg5") and n != spec.n: kw["extent"] = (224.0 if name == "cfg3" else 500.0) * (n / spec.n) ** 0.5
    path = f"/tmp/ab_{name}_{n}.npy"
    if not os.path.exists(path):
        np.save(path, synthetic.make(name, n, **kw))
    print(f"## {name} n={n} grid={gl}", flush=True)
    for lib in a.libs:
        env = dict(os.environ)
        lib, *extra = lib.split("@")   # lib.so@VAR=VALUE@VAR2=VALUE2
        for kv in extra:
            k, _, v = kv.partition("=")
            env[k] = v
        if lib != "default":
            env["GNDT_LIB"] = os.path.join(ROOT, lib) if not os.path.isabs(lib) else lib
        r = subprocess.run([sys.executable, "-c", WORKER, path, str(gl), str(spec.z_len), str(a.builds)], env=env, capture_output=True, text=True, timeout=600)
        print(r.stdout.strip() if r.returncode == 0 else f"{lib}: FAILED rc={r.returncode} {r.stderr[-1500:]}", flush=True)
